"""FunctionAdaCoF / batch_edt on the GPU vs the oracle (pinned to the reference's kernels on the CPU).  The kernels were
written after r01's last GPU minute; first GPU run r02 (profiles/r02_a_gpu_tests.log): green."""
import pytest
import torch

from oracle import ops_ref
from ops_cases import first_mismatch

pytestmark = [pytest.mark.gpu]


def test_adacof_gpu(pkg):
    from cfi_b200 import ops
    g = torch.Generator().manual_seed(5)
    n, c, ho, wo, f, dil = 2, 19, 33, 47, 5, 2
    x = torch.randn(n, c, ho + (f - 1) * dil, wo + (f - 1) * dil, generator=g)
    w = torch.randn(n, f * f, ho, wo, generator=g)
    oi = torch.randn(n, f * f, ho, wo, generator=g) * 3
    oj = torch.randn(n, f * f, ho, wo, generator=g) * 3
    out = ops.FunctionAdaCoF.apply(x.cuda(), w.cuda(), oi.cuda(), oj.cuda(), dil).cpu()
    ref = ops_ref.adacof(x, w, oi, oj, dil)
    assert (out - ref).abs().max().item() <= 2e-5 * max(1.0, float(ref.abs().max()))


def test_batch_edt_gpu(pkg):
    from cfi_b200 import ops
    g = torch.Generator().manual_seed(6)
    img = (torch.rand(3, 1, 40, 56, generator=g) > 0.95).float()
    img[2] = 0
    out = ops.batch_edt(img.cuda()).cpu()
    assert out.shape == img.shape
    assert (out - ops_ref.batch_edt(img)).abs().max().item() <= 1e-4


@pytest.mark.parametrize("mode", ["avg", "linear", "soft", "soft-zeroeps", "linear-clipeps"])
def test_softsplat_fused_gpu(pkg, mode):
    """ops.softsplat's weighted modes (vfi_softsplat_weighted: the implementation since r02) vs the oracle at a GMFSS-like shape."""
    from cfi_b200 import ops
    g = torch.Generator().manual_seed(11)
    x = torch.randn(2, 32, 96, 128, generator=g)
    flow = (torch.rand(2, 2, 96, 128, generator=g) - 0.5) * 20
    metric = torch.rand(2, 1, 96, 128, generator=g) * 2 - (0.5 if mode.startswith("soft") else -0.2)
    m = None if mode == "avg" else metric
    out = ops.softsplat(x.cuda(), flow.cuda(), None if m is None else m.cuda(), mode).cpu()
    ref = ops_ref.softsplat(x, flow, m, mode)
    err = first_mismatch(out, ref, 2e-6 * max(1.0, float(ref.abs().max())))
    assert err is None, err

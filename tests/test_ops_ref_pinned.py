"""Pin oracle/ops_ref.py (the CPU restatements the sm_100a op kernels are checked against on the GPU) to the REFERENCE'S OWN
kernels: the cupy kernel strings of vfi_models/ops/cupy_ops, specialised by the reference's own pre-processor and executed
on the CPU through tests/host_emu (oracle/ref_ops.py).  Their inputs and outputs are stored in
tests/golden/ops_ref_kernels.npz (tools/make_golden_ops.py), so these tests need no copy of the reference."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import ops_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from make_golden_ops import ADACOF, CORRELATION, COSTVOL, NPZ, SEPCONV, SOFTSPLAT, case  # noqa: E402

_GOLD = np.load(NPZ)


def golden(name):
    prefix = name + ":"
    d = {k[len(prefix):]: torch.from_numpy(_GOLD[k]) for k in _GOLD.files if k.startswith(prefix)}
    assert d, name
    return d


@pytest.mark.parametrize("shape,mag", SOFTSPLAT)
def test_softsplat_sum_matches_reference_kernel(shape, mag):
    g = golden(case("softsplat_sum", shape, mag))
    got = ops_ref.softsplat_sum(g["x"], g["flow"])
    assert (got - g["out"]).abs().max().item() <= 1e-5


def test_softsplat_modes_on_top_of_the_reference_kernel():
    """softsplat() (cupy_ops/softsplat.py:382-435) = host arithmetic around softsplat_out; with the kernel being the
    reference's, 'avg' and 'soft' of the oracle must agree with that arithmetic done here."""
    g = golden("softsplat_modes")
    x, flow, metric = g["x"], g["flow"], g["metric"]
    o = g["avg"]
    norm = o[:, -1:].clone()
    norm[norm == 0.0] = 1.0
    assert (ops_ref.softsplat(x, flow, None, "avg") - o[:, :-1] / norm).abs().max().item() <= 2e-4  # small normalisers amplify fp32 rounding
    o = g["soft"]
    norm = o[:, -1:].clone()
    norm[norm == 0.0] = 1.0
    assert (ops_ref.softsplat(x, flow, metric, "soft") - o[:, :-1] / norm).abs().max().item() <= 2e-4  # small normalisers amplify fp32 rounding


@pytest.mark.parametrize("shape", COSTVOL)
def test_costvol_matches_reference_kernel(shape):
    g = golden(case("costvol", shape))
    assert (ops_ref.costvol_l1(g["one"], g["two"]) - g["out"]).abs().max().item() <= 1e-5


@pytest.mark.parametrize("k,hw", SEPCONV)
def test_sepconv_matches_reference_kernel(k, hw):
    g = golden(case("sepconv", k, hw))
    ref = g["out"]
    got = ops_ref.sepconv(g["x"], g["ver"], g["hor"])
    assert (got - ref).abs().max().item() <= 1e-4 * max(1.0, float(ref.abs().max()))


@pytest.mark.parametrize("shape", CORRELATION)
def test_correlation_dot_matches_reference_kernels(shape):
    """kernel_Correlation_rearrange + kernel_Correlation_updateOutput with blocks of 16 / 32 cooperating threads (fibers)."""
    g = golden(case("correlation", shape))
    assert (ops_ref.correlation_dot(g["a"], g["b"]) - g["out"]).abs().max().item() <= 1e-5


@pytest.mark.parametrize("f,dil", ADACOF)
def test_adacof_matches_reference_kernel(f, dil):
    g = golden(case("adacof", f, dil))
    ref = g["out"]
    assert (ops_ref.adacof(g["x"], g["w"], g["oi"], g["oj"], dil) - ref).abs().max().item() <= 2e-5 * max(1.0, float(ref.abs().max()))


def test_edt_matches_reference_kernel_and_scipy():
    g = golden("edt")
    img, data = g["img"], g["data"]
    diam2 = 9 ** 2 + 12 ** 2
    assert torch.equal(ops_ref.edt_pass(data, diam2), g["out"])
    from scipy import ndimage
    want = ndimage.distance_transform_edt(1 - img[0].numpy())
    assert abs(ops_ref.batch_edt(img)[0].numpy() - want).max() <= 1e-4
    assert float(ops_ref.batch_edt(img)[1].min()) == pytest.approx(diam2 ** 0.5)

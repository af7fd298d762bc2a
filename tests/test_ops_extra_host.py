"""csrc/ops_extra.cu (FunctionAdaCoF, the batch_edt pass) compiled for the HOST (tests/host_emu) and run against the oracle
restatements, which tests/test_ops_ref_pinned.py pins to the reference's own kernels."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from oracle import ops_ref
from ops_cases import ADACOF_SHAPES, adacof_inputs, first_mismatch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA_INC = "/usr/local/cuda/include"


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    if not (shutil.which("g++") and os.path.exists(os.path.join(CUDA_INC, "cuda_fp16.h"))):
        pytest.skip("g++ / CUDA headers not available")
    so = str(tmp_path_factory.mktemp("emu") / "libopsx.so")
    src = os.path.join(ROOT, "tests", "host_emu", "ops_extra_emu.cpp")
    r = subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-pthread", "-I" + CUDA_INC, "-o", so, src] + os.environ.get("VFI_EMU_CXXFLAGS", "").split(),
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return C.CDLL(so)


def vp(t):
    return C.c_void_p(t.data_ptr())


@pytest.mark.parametrize("f,dil,c", [(3, 1, 3), (5, 2, 11)])
def test_adacof_kernel(emu, f, dil, c):
    g = torch.Generator().manual_seed(f + c)
    n, ho, wo = 2, 6, 7
    hin, win = ho + (f - 1) * dil, wo + (f - 1) * dil
    x = torch.randn(n, c, hin, win, generator=g)
    w = torch.randn(n, f * f, ho, wo, generator=g)
    oi = torch.randn(n, f * f, ho, wo, generator=g) * 2.5
    oj = torch.randn(n, f * f, ho, wo, generator=g) * 2.5
    out = torch.zeros(n, c, ho, wo)
    assert emu.emu_adacof(vp(x), vp(w), vp(oi), vp(oj), vp(out), n, c, hin, win, f, dil, ho, wo) == 0
    ref = ops_ref.adacof(x, w, oi, oj, dil)
    assert (out - ref).abs().max().item() <= 2e-5 * max(1.0, float(ref.abs().max()))


def test_edt_pass_kernel(emu):
    g = torch.Generator().manual_seed(0)
    img = (torch.rand(3, 10, 17, generator=g) > 0.9).float()
    diam2 = float(10 ** 2 + 17 ** 2)
    data = ((1 - img) * diam2).contiguous()
    out = torch.zeros_like(data)
    assert emu.emu_edt_pass(vp(data), vp(out), 3, 10, 17, C.c_float(diam2)) == 0
    assert torch.equal(out, ops_ref.edt_pass(data, diam2))


@pytest.mark.parametrize("shape", ADACOF_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_adacof_exact(emu, shape):
    """dyadic inputs (tests/ops_cases.py), offsets in [-6, 6] with negative fractions: bit-exact against the oracle"""
    n, c, ho, wo, f, dil = shape
    x, w, oi, oj = adacof_inputs(n, c, ho, wo, f, dil, sum(shape))
    out = torch.full((n, c, ho, wo), float("nan"))
    assert emu.emu_adacof(vp(x), vp(w), vp(oi), vp(oj), vp(out), n, c, x.shape[2], x.shape[3], f, dil, ho, wo) == 0
    err = first_mismatch(out, ops_ref.adacof(x, w, oi, oj, dil))
    assert err is None, err

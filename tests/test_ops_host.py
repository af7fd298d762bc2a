"""csrc/ops.cu (the kernels behind vfi_softsplat_sum / vfi_costvol_l1 / vfi_corr_dot / vfi_sepconv, incl. the shared-memory
tiled ones) compiled for the HOST (tests/host_emu/cuda_shim_block.h: blocks on host threads, threads as fibers) against the
oracle restatements that tests/test_ops_ref_pinned.py pins to the reference's own kernels.  The same kernels are GPU-tested
in tests/test_gpu_ops.py; this keeps them under test where there is no GPU."""
import ctypes as C
import os
import shutil
import subprocess

import pytest
import torch

from oracle import ops_ref
from ops_cases import first_mismatch

# random (not dyadic) inputs of the weighted splat modes: the kernels and the oracle differ in summation order and in
# exp only, measured <= 4.8e-7 * max(1, max|ref|) on the host; untouched targets are 0 in both
WEIGHTED_TOL = 2e-6

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA_INC = "/usr/local/cuda/include"


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    if not (shutil.which("g++") and os.path.exists(os.path.join(CUDA_INC, "cuda_fp16.h"))):
        pytest.skip("g++ / CUDA headers not available")
    so = str(tmp_path_factory.mktemp("emu") / "libopsemu.so")
    src = os.path.join(ROOT, "tests", "host_emu", "ops_emu.cpp")
    r = subprocess.run(["g++", "-O2", "-std=c++20", "-shared", "-fPIC", "-pthread", "-I" + CUDA_INC, "-o", so, src] + os.environ.get("VFI_EMU_CXXFLAGS", "").split(),
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return C.CDLL(so)


def vp(t):
    return C.c_void_p(t.data_ptr())


def test_softsplat_kernel(emu):
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 5, 19, 23, generator=g)
    flow = (torch.rand(2, 2, 19, 23, generator=g) - 0.5) * 9
    out = torch.full_like(x, 7.0)   # the launcher zeroes the output itself
    assert emu.emu_softsplat(vp(x), vp(flow), vp(out), 2, 5, 19, 23) == 0
    assert (out - ops_ref.softsplat_sum(x, flow)).abs().max().item() <= 1e-4   # atomics: summation order differs


@pytest.mark.parametrize("dot", [0, 1])
def test_volume81_kernels(emu, dot):
    g = torch.Generator().manual_seed(dot)
    a, b = torch.randn(1, 20, 21, 37, generator=g), torch.randn(1, 20, 21, 37, generator=g)
    out = torch.zeros(1, 81, 21, 37)
    assert emu.emu_volume81(dot, vp(a), vp(b), vp(out), 1, 20, 21, 37) == 0
    ref = ops_ref.correlation_dot(a, b) if dot else ops_ref.costvol_l1(a, b)
    assert (out - ref).abs().max().item() <= 1e-4


def test_sepconv_tiled_kernel(emu):
    g = torch.Generator().manual_seed(3)
    h, w, k = 19, 45, 51                       # not multiples of the 16 x 32 tile
    x = torch.randn(1, 4, h + k - 1, w + k - 1, generator=g)
    ver, hor = torch.randn(1, k, h, w, generator=g), torch.randn(1, k, h, w, generator=g)
    out = torch.zeros(1, 4, h, w)
    assert emu.emu_sepconv(vp(x), vp(ver), vp(hor), vp(out), 1, 4, h, w, k, k) == 0
    ref = ops_ref.sepconv(x, ver, hor)
    assert (out - ref).abs().max().item() <= 2e-4 * max(1.0, float(ref.abs().max()))


@pytest.mark.parametrize("mode", ["avg", "linear", "soft", "soft-zeroeps", "linear-clipeps"])
def test_softsplat_fused_modes(emu, mode):
    """vfi_softsplat_weighted (two launches, no temporaries) == the reference's cat -> splat -> divide chain."""
    g = torch.Generator().manual_seed(len(mode))
    x = torch.randn(2, 6, 17, 21, generator=g)
    flow = (torch.rand(2, 2, 17, 21, generator=g) - 0.5) * 8
    metric = torch.rand(2, 1, 17, 21, generator=g) * 2 - (0.5 if mode.startswith("soft") else -0.2)
    base = mode.split("-")[0]
    m = {"avg": 0, "linear": 1, "soft": 2}[base]
    e = {"addeps": 0, "zeroeps": 1, "clipeps": 2}[mode.split("-")[1] if "-" in mode else "addeps"]
    out, norm = torch.full_like(x, 3.0), torch.full((2, 1, 17, 21), 3.0)
    assert emu.emu_softsplat_weighted(vp(x), vp(flow), None if m == 0 else vp(metric), m, e, vp(out), vp(norm), 2, 6, 17, 21) == 0
    ref = ops_ref.softsplat(x, flow, None if m == 0 else metric, mode)
    err = first_mismatch(out, ref, WEIGHTED_TOL * max(1.0, float(ref.abs().max())))   # measured: <= 4.8e-7 for every mode
    assert err is None, err


@pytest.mark.parametrize("mode", ["avg", "linear", "soft", "soft-zeroeps", "linear-clipeps"])
@pytest.mark.parametrize("c", [6, 3])
def test_softsplat_channel_last_modes(emu, mode, c):
    """the channel-last form behind vfi_softsplat_weighted since r02 (NCHW -> NHWC transpose, 16-byte vector atomics per four
    channels, normalise + transpose back) == the reference's chain; C = 3 exercises the channel padding"""
    g = torch.Generator().manual_seed(len(mode) + c)
    x = torch.randn(2, c, 17, 21, generator=g)
    flow = (torch.rand(2, 2, 17, 21, generator=g) - 0.5) * 8
    metric = torch.rand(2, 1, 17, 21, generator=g) * 2 - (0.5 if mode.startswith("soft") else -0.2)
    base = mode.split("-")[0]
    m = {"avg": 0, "linear": 1, "soft": 2}[base]
    e = {"addeps": 0, "zeroeps": 1, "clipeps": 2}[mode.split("-")[1] if "-" in mode else "addeps"]
    out, norm = torch.full_like(x, 3.0), torch.full((2, 1, 17, 21), 3.0)
    cp = (c + 3) // 4 * 4
    sa, sb = torch.full((2 * 17 * 21 * cp,), 5.0), torch.full((2 * 17 * 21 * cp,), 5.0)
    assert emu.emu_softsplat_weighted_nhwc(vp(x), vp(flow), None if m == 0 else vp(metric), m, e, vp(out), vp(norm), vp(sa), vp(sb), 2, c,
                                           17, 21) == 0
    ref = ops_ref.softsplat(x, flow, None if m == 0 else metric, mode)
    err = first_mismatch(out, ref, WEIGHTED_TOL * max(1.0, float(ref.abs().max())))
    assert err is None, err


@pytest.mark.parametrize("dot", [0, 1])
def test_volume81_warp_kernels(emu, dot):
    """the warp-per-pixel channel-last volume (shuffle reduction over the channels) == the oracle; C = 20 is not a multiple of
    32 (partial lane coverage) nor of 4 (channel padding), W = 37 not a multiple of the 8 pixels of a block"""
    g = torch.Generator().manual_seed(10 + dot)
    a, b = torch.randn(1, 20, 13, 37, generator=g), torch.randn(1, 20, 13, 37, generator=g)
    out = torch.zeros(1, 81, 13, 37)
    sa, sb = torch.zeros(13 * 37 * 20), torch.zeros(13 * 37 * 20)
    assert emu.emu_volume81_warp(dot, vp(a), vp(b), vp(out), vp(sa), vp(sb), 1, 20, 13, 37) == 0
    ref = ops_ref.correlation_dot(a, b) if dot else ops_ref.costvol_l1(a, b)
    assert (out - ref).abs().max().item() <= 1e-4


# ---- exact cases (tests/ops_cases.py): dyadic inputs, so every kernel form must equal the oracle bit for bit (soft mode:
# within SOFT_TOL), and every mismatch is reported with its first element

import ops_cases as K  # noqa: E402

_MODE = {"avg": 0, "linear": 1, "soft": 2}
_EPS = {"addeps": 0, "zeroeps": 1, "clipeps": 2}
NAN = float("nan")


def _mode_eps(mode):
    base, _, variant = mode.partition("-")
    return _MODE[base], _EPS[variant or "addeps"]


def _weight_plane(x, metric, mode):
    base = mode.split("-")[0]
    if base == "avg":
        return torch.ones(x.shape[0], 1, *x.shape[2:])
    return metric if base == "linear" else metric.exp()


def _guarded(shape):
    """A NaN-filled tensor of `shape` in the middle of a NaN-filled buffer three times its size: a launcher's write past
    either end lands in a guard band (_guard_err reports it) rather than in memory the test does not own."""
    numel = 1
    for d in shape:
        numel *= d
    buf = torch.full((3 * numel,), NAN)
    return buf, buf[numel:2 * numel].view(shape)


def _guard_err(name, buf):
    numel = buf.numel() // 3
    bands = torch.cat([buf[:numel], buf[2 * numel:]])
    err = K.first_mismatch(bands, torch.full_like(bands, NAN))
    return None if err is None else f"{name} written out of bounds (guard bands, flat): {err}"


def _emu_splat(emu, form, x, flow, metric, mode):
    """One splat through the emulated launcher of `form` ("nchw": the fused NCHW kernels, "nhwc": the channel-last form);
    outputs and scratch start as NaN, the launchers must zero what they accumulate into.  Returns (out, norm, errors
    of writes outside out / norm / scratch)."""
    n, c, h, w = x.shape
    bout, out = _guarded(x.shape)
    bufs = {"out": bout}
    if mode == "sum":
        assert emu.emu_softsplat(vp(x), vp(flow), vp(out), n, c, h, w) == 0
        norm = None
    else:
        m, e = _mode_eps(mode)
        bufs["norm"], norm = _guarded((n, 1, h, w))
        mp = None if metric is None else vp(metric)
        if form == "nchw":
            assert emu.emu_softsplat_weighted(vp(x), vp(flow), mp, m, e, vp(out), vp(norm), n, c, h, w) == 0
        else:
            cp = (c + 3) // 4 * 4
            (bufs["scratch a"], sa), (bufs["scratch b"], sb) = _guarded((n * h * w * cp,)), _guarded((n * h * w * cp,))
            assert emu.emu_softsplat_weighted_nhwc(vp(x), vp(flow), mp, m, e, vp(out), vp(norm), vp(sa), vp(sb), n, c, h,
                                                   w) == 0
    return out, norm, [err for name, b in bufs.items() if (err := _guard_err(name, b))]


def _splat_case(case, mode, seed):
    if case == "edge":
        return K.edge_splat_inputs(mode, seed)
    return K.splat_inputs(K.SPLAT_SHAPES[case], mode, seed)


@pytest.mark.parametrize("form", ["nchw", "nhwc"])
@pytest.mark.parametrize("case", list(range(len(K.SPLAT_SHAPES))) + ["edge"])
def test_softsplat_exact(emu, case, form):
    """every mode and eps variant of the splat on the shape / edge-flow table: out == oracle, and the norm plane == the
    summation splat of the weight plane"""
    bad = []
    for i, mode in enumerate(K.SPLAT_MODES):
        if mode == "sum" and form == "nhwc":
            continue  # "sum" is its own kernel, not a form of the weighted splat
        x, flow, metric = _splat_case(case, mode, 100 + i)
        out, norm, oob = _emu_splat(emu, form, x, flow, metric, mode)
        bad += [f"{mode}: {err}" for err in oob]
        ref = ops_ref.softsplat(x, flow, metric, mode)
        err = K.first_mismatch(out, ref, K.splat_tol(mode, ref))
        if err:
            bad.append(f"{mode} out: {err}")
        if norm is not None:
            nref = ops_ref.softsplat_sum(_weight_plane(x, metric, mode), flow)
            err = K.first_mismatch(norm, nref, K.splat_tol(mode, nref))
            if err:
                bad.append(f"{mode} norm: {err}")
    assert not bad, "\n".join(bad)


@pytest.mark.parametrize("shape", K.VOLUME_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_volume81_exact(emu, shape):
    """costvol and correlation in all three forms (shared-memory tiled, per-pixel, warp per pixel) on the shape table"""
    n, c, h, w = shape
    a, b = K.volume_inputs(shape, sum(shape))
    refs = {0: ops_ref.costvol_l1(a, b), 1: ops_ref.correlation_dot(a, b)}
    bad = []
    for dot in (0, 1):
        for form in ("tiled", "per-pixel", "warp"):
            bufs = {}
            bufs["out"], out = _guarded((n, 81, h, w))
            if form == "warp":
                cp = (c + 3) // 4 * 4
                (bufs["scratch a"], sa), (bufs["scratch b"], sb) = _guarded((n * h * w * cp,)), _guarded((n * h * w * cp,))
                assert emu.emu_volume81_warp(dot, vp(a), vp(b), vp(out), vp(sa), vp(sb), n, c, h, w) == 0
            else:
                assert emu.emu_volume81_form(int(form == "tiled"), dot, vp(a), vp(b), vp(out), n, c, h, w) == 0
            name = f"{'corr' if dot else 'costvol'} {form}"
            bad += [f"{name}: {err}" for nm, b in bufs.items() if (err := _guard_err(nm, b))]
            err = K.first_mismatch(out, refs[dot])
            if err:
                bad.append(f"{name}: {err}")
    assert not bad, "\n".join(bad)


@pytest.mark.parametrize("shape", K.SEPCONV_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_sepconv_exact(emu, shape):
    """sepconv on the shape table: K = 51 in every form (PY = 1, 2, 3 pixels per thread and the per-pixel kernel), other
    sizes (Kv != Kh included) through the generic kernel"""
    n, c, h, w, kv, kh = shape
    x, ver, hor = K.sepconv_inputs(n, c, h, w, kv, kh, sum(shape))
    ref = ops_ref.sepconv(x, ver, hor)
    bad = []
    for py in ((0, 1, 2, 3) if kv == kh == 51 else (2,)):
        buf, out = _guarded((n, c, h, w))
        assert emu.emu_sepconv_form(py, vp(x), vp(ver), vp(hor), vp(out), n, c, h, w, kv, kh) == 0
        for err in (_guard_err("out", buf), K.first_mismatch(out, ref)):
            if err:
                bad.append(f"py={py}: {err}")
    assert not bad, "\n".join(bad)


def test_big_batch_exact(emu):
    """N = 65536 (more images than grid.z holds): the NCHW splat, the per-pixel volume and the generic sepconv index
    batches past 2^16; the channel-last splat refuses the batch.  The batch is 8 distinct images repeated; the oracle runs
    on the 8 and its result is tiled."""
    n, d = K.BIG_N, K.BIG_DISTINCT
    bad = []
    x8, flow8, metric8 = K.splat_inputs((d, 2, 2, 3), "linear", 7)
    x, flow, metric = (K.tile_batch(t, n).contiguous() for t in (x8, flow8, metric8))
    for mode in ("sum", "linear"):
        out, _, oob = _emu_splat(emu, "nchw", x, flow, None if mode == "sum" else metric, mode)
        bad += [f"splat {mode}: {err}" for err in oob]
        err = K.first_mismatch(out, K.tile_batch(ops_ref.softsplat(x8, flow8, None if mode == "sum" else metric8, mode), n))
        if err:
            bad.append(f"splat {mode}: {err}")
    out, norm = torch.empty_like(x), torch.empty(n, 1, 2, 3)
    sa, sb = torch.empty(n * 6 * 4), torch.empty(n * 6 * 4)
    assert emu.emu_softsplat_weighted_nhwc(vp(x), vp(flow), vp(metric), 1, 0, vp(out), vp(norm), vp(sa), vp(sb), n, 2, 2, 3) != 0
    a8, b8 = K.volume_inputs((d, 3, 2, 3), 8)
    a, b = K.tile_batch(a8, n).contiguous(), K.tile_batch(b8, n).contiguous()
    for dot, fn in ((0, ops_ref.costvol_l1), (1, ops_ref.correlation_dot)):
        out = torch.full((n, 81, 2, 3), NAN)
        assert emu.emu_volume81_form(1, dot, vp(a), vp(b), vp(out), n, 3, 2, 3) == 0
        err = K.first_mismatch(out, K.tile_batch(fn(a8, b8), n))
        if err:
            bad.append(f"volume dot={dot}: {err}")
    x8, ver8, hor8 = K.sepconv_inputs(d, 2, 1, 2, 3, 5, 9)
    x, ver, hor = (K.tile_batch(t, n).contiguous() for t in (x8, ver8, hor8))
    out = torch.full((n, 2, 1, 2), NAN)
    assert emu.emu_sepconv_form(2, vp(x), vp(ver), vp(hor), vp(out), n, 2, 1, 2, 3, 5) == 0
    err = K.first_mismatch(out, K.tile_batch(ops_ref.sepconv(x8, ver8, hor8), n))
    if err:
        bad.append(f"sepconv: {err}")
    assert not bad, "\n".join(bad)

"""-m gpu: the op kernels (softsplat, costvol, correlation, sepconv, AdaCoF) bit-exactly against the oracle, on the dyadic
case table of tests/ops_cases.py that tests/test_ops_host.py and test_ops_extra_host.py run through the host build of the
same kernels.  On those inputs every summation order gives the same fp32 number, so any differing element is a wrong
element (soft mode: within ops_cases.SOFT_TOL), and each failure names the first one.

Besides the public cfi_b200.ops functions this covers, through the C ABI: outputs the library must zero itself, the norm
plane, scratch regrowth in one context, both sides of the N = 65535 / 65536 kernel switch, the caller's stream, two
streams sharing one context's scratch, and each kernel form that an environment variable selects (read once per process,
so each runs in a child process)."""
import ctypes as C
import os
import subprocess
import sys

import pytest
import torch

import ops_cases as K
from oracle import ops_ref as R

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
NAN = float("nan")
_MODE = {"avg": 0, "linear": 1, "soft": 2}
_EPS = {"addeps": 0, "zeroeps": 1, "clipeps": 2}


def _ops():
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    import __graft_entry__ as ge
    ge.load_package()
    import cfi_b200.ops as O
    return O


def _cuda(*ts):
    return [None if t is None else t.cuda() for t in ts]


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


# ---- the exact table through the public functions; each runner returns one line per mismatch


def run_splat(O, cases=None):
    bad = []
    for case in cases if cases is not None else list(range(len(K.SPLAT_SHAPES))) + ["edge"]:
        for i, mode in enumerate(K.SPLAT_MODES):
            x, flow, metric = (K.edge_splat_inputs(mode, 100 + i) if case == "edge"
                               else K.splat_inputs(K.SPLAT_SHAPES[case], mode, 100 + i))
            got = O.softsplat(*_cuda(x, flow, metric), mode)
            ref = R.softsplat(x, flow, metric, mode)
            err = K.first_mismatch(got, ref, K.splat_tol(mode, ref))
            if err:
                bad.append(f"splat {x.shape[0]}x{x.shape[1]}x{x.shape[2]}x{x.shape[3]} case {case} {mode}: {err}")
    return bad


def run_volumes(O, shapes=None):
    bad = []
    for shape in shapes or K.VOLUME_SHAPES:
        a, b = K.volume_inputs(shape, sum(shape))
        ga, gb = _cuda(a, b)
        for name, got, ref in (("costvol", O.costvol_func.apply(ga, gb), R.costvol_l1(a, b)),
                               ("corr", O.FunctionCorrelation(ga, gb), R.correlation_dot(a, b))):
            err = K.first_mismatch(got, ref)
            if err:
                bad.append(f"{name} {shape}: {err}")
    return bad


def run_sepconv(O, shapes=None):
    bad = []
    for shape in shapes or K.SEPCONV_SHAPES:
        x, ver, hor = K.sepconv_inputs(*shape, sum(shape))
        err = K.first_mismatch(O.sepconv_func.apply(*_cuda(x, ver, hor)), R.sepconv(x, ver, hor))
        if err:
            bad.append(f"sepconv {shape}: {err}")
    return bad


def run_adacof(O, shapes=None):
    bad = []
    for shape in shapes or K.ADACOF_SHAPES:
        n, c, ho, wo, f, dil = shape
        x, w, oi, oj = K.adacof_inputs(*shape, sum(shape))
        err = K.first_mismatch(O.FunctionAdaCoF.apply(*_cuda(x, w, oi, oj), dil), R.adacof(x, w, oi, oj, dil))
        if err:
            bad.append(f"adacof {shape}: {err}")
    return bad


RUNNERS = {"splat": run_splat, "volumes": run_volumes, "sepconv": run_sepconv, "adacof": run_adacof}


def child_main(op):
    """Entry point of a variant's child process: run one op's exact table, print every mismatch, exit 1 if any."""
    bad = RUNNERS[op](_ops())
    torch.cuda.synchronize()
    for line in bad:
        print(line)
    print(f"{op}: {len(bad)} mismatching cases")
    return 1 if bad else 0


@pytest.fixture(scope="module")
def O(pkg):
    return _ops()


@pytest.mark.parametrize("op", sorted(RUNNERS))
def test_exact_table(O, op):
    bad = RUNNERS[op](O)
    assert not bad, "\n".join(bad)


def test_callers_stream(O):
    """every op on a side stream, its inputs produced on that stream"""
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        bad = (run_splat(O, [0, "edge"]) + run_volumes(O, K.VOLUME_SHAPES[:2]) + run_sepconv(O, K.SEPCONV_SHAPES[:1]) +
               run_sepconv(O, K.SEPCONV_SHAPES[4:5]) + run_adacof(O, K.ADACOF_SHAPES[:2]))
    torch.cuda.synchronize()
    assert not bad, "\n".join(bad)


# ---- C ABI


@pytest.fixture
def ctx(O):
    """a fresh context, so that its scratch starts empty"""
    from cfi_b200._lib import check, lib
    h = C.c_void_p()
    check(lib().vfi_create(torch.cuda.current_device(), C.byref(h)))
    yield h
    torch.cuda.synchronize()
    check(lib().vfi_destroy(h))


def _capi_splat(ctx, x, flow, metric, mode, stream=None):
    """vfi_softsplat_weighted / vfi_softsplat_sum with out and norm filled with NaN: the library zeroes what it
    accumulates into.  Returns (out, norm) on the CPU."""
    from cfi_b200._lib import check, lib
    n, c, h, w = x.shape
    st = (stream or torch.cuda.current_stream()).cuda_stream
    gx, gf, gm = _cuda(x, flow, metric)
    out = torch.full_like(gx, NAN)
    if mode == "sum":
        check(lib().vfi_softsplat_sum(ctx, _p(gx), _p(gf), _p(out), n, c, h, w, st))
        return out.cpu(), None
    base, _, variant = mode.partition("-")
    norm = torch.full((n, 1, h, w), NAN, device="cuda")
    check(lib().vfi_softsplat_weighted(ctx, _p(gx), _p(gf), _p(gm), _MODE[base], _EPS[variant or "addeps"], _p(out),
                                       _p(norm), n, c, h, w, st))
    return out.cpu(), norm.cpu()


def _splat_checks(ctx, shape, modes, seed):
    bad = []
    for mode in modes:
        x, flow, metric = K.splat_inputs(shape, mode, seed)
        out, norm = _capi_splat(ctx, x, flow, metric, mode)
        ref = R.softsplat(x, flow, metric, mode)
        err = K.first_mismatch(out, ref, K.splat_tol(mode, ref))
        if err:
            bad.append(f"{shape} {mode} out: {err}")
        if norm is not None:
            base = mode.split("-")[0]
            wp = torch.ones(shape[0], 1, *shape[2:]) if base == "avg" else (metric if base == "linear" else metric.exp())
            nref = R.softsplat_sum(wp, flow)
            err = K.first_mismatch(norm, nref, K.splat_tol(mode, nref))
            if err:
                bad.append(f"{shape} {mode} norm: {err}")
    return bad


def test_capi_zeroes_outputs_and_fills_norm(ctx):
    """NaN-filled out / norm come back exact; norm is the summation splat of the weight plane"""
    bad = []
    for i, shape in enumerate(K.SPLAT_SHAPES[:4]):
        bad += _splat_checks(ctx, shape, K.SPLAT_MODES, 200 + i)
    assert not bad, "\n".join(bad)


def test_capi_other_ops_overwrite_nan(ctx):
    """volumes and sepconv write every output element (out starts as NaN)"""
    from cfi_b200._lib import check, lib
    st = torch.cuda.current_stream().cuda_stream
    bad = []
    for shape in K.VOLUME_SHAPES[:4]:
        n, c, h, w = shape
        a, b = K.volume_inputs(shape, sum(shape))
        ga, gb = _cuda(a, b)
        for name, fn, ref in (("costvol", lib().vfi_costvol_l1, R.costvol_l1(a, b)),
                              ("corr", lib().vfi_corr_dot, R.correlation_dot(a, b))):
            out = torch.full((n, 81, h, w), NAN, device="cuda")
            check(fn(ctx, _p(ga), _p(gb), _p(out), n, c, h, w, st))
            err = K.first_mismatch(out, ref)
            if err:
                bad.append(f"{name} {shape}: {err}")
    for shape in (K.SEPCONV_SHAPES[0], K.SEPCONV_SHAPES[6]):
        n, c, h, w, kv, kh = shape
        x, ver, hor = K.sepconv_inputs(*shape, sum(shape))
        gx, gv, gh = _cuda(x, ver, hor)
        out = torch.full((n, c, h, w), NAN, device="cuda")
        check(lib().vfi_sepconv(ctx, _p(gx), _p(gv), _p(gh), _p(out), n, c, h, w, kv, kh, st))
        err = K.first_mismatch(out, R.sepconv(x, ver, hor))
        if err:
            bad.append(f"sepconv {shape}: {err}")
    assert not bad, "\n".join(bad)


def test_capi_scratch_regrowth(ctx):
    """small, then large (C = 65, larger image: the context's scratch grows), then small again through one context"""
    bad = []
    for i, shape in enumerate([(1, 3, 5, 7), (2, 65, 48, 80), (1, 3, 5, 7), (2, 5, 9, 13)]):
        bad += _splat_checks(ctx, shape, ["avg", "linear-clipeps", "soft"], 300 + i)
    assert not bad, "\n".join(bad)


def test_capi_two_streams_share_scratch(ctx):
    """two splats through one context on two streams, not synchronised with each other: the second call must not
    overwrite the scratch the first one is still using"""
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    shape = (4, 64, 128, 160)
    a = K.splat_inputs(shape, "linear", 401)
    b = K.splat_inputs(shape, "linear", 402)
    _capi_splat(ctx, *a, "linear")  # the scratch reaches its size here: growing it waits on the host
    with torch.cuda.stream(s1):
        ga = _cuda(*a)
    with torch.cuda.stream(s2):
        gb = _cuda(*b)
    torch.cuda.synchronize()
    from cfi_b200._lib import check, lib
    n, c, h, w = shape
    outs = []
    for s, (gx, gf, gm) in ((s1, ga), (s2, gb)):
        with torch.cuda.stream(s):
            out, norm = torch.empty_like(gx), torch.empty(n, 1, h, w, device="cuda")
            check(lib().vfi_softsplat_weighted(ctx, _p(gx), _p(gf), _p(gm), 1, 0, _p(out), _p(norm), n, c, h, w, s.cuda_stream))
            outs.append(out)
    torch.cuda.synchronize()
    bad = [f"stream {i + 1}: {err}" for i, (out, inp) in enumerate(zip(outs, (a, b)))
           if (err := K.first_mismatch(out, R.softsplat(*inp, "linear")))]
    assert not bad, "\n".join(bad)


@pytest.mark.parametrize("n", [65535, K.BIG_N])
def test_batch_kernel_switch(O, n):
    """N = 65535 takes the grid.z kernels (channel-last splat, tiled volume, tiled sepconv), N = 65536 the others; the
    batch repeats 8 distinct images, whose oracle result is tiled"""
    d = K.BIG_DISTINCT
    bad = []
    x8, f8, m8 = K.splat_inputs((d, 2, 2, 3), "linear", 11)
    x, f, m = (K.tile_batch(t.cuda(), n).contiguous() for t in (x8, f8, m8))
    for mode in ("sum", "avg", "linear"):
        mm, mm8 = (None, None) if mode in ("sum", "avg") else (m, m8)
        err = K.first_mismatch(O.softsplat(x, f, mm, mode), K.tile_batch(R.softsplat(x8, f8, mm8, mode), n))
        if err:
            bad.append(f"splat {mode}: {err}")
    a8, b8 = K.volume_inputs((d, 3, 2, 3), 12)
    a, b = (K.tile_batch(t.cuda(), n).contiguous() for t in (a8, b8))
    for name, got, ref in (("costvol", O.costvol_func.apply(a, b), R.costvol_l1(a8, b8)),
                           ("corr", O.FunctionCorrelation(a, b), R.correlation_dot(a8, b8))):
        err = K.first_mismatch(got, K.tile_batch(ref, n))
        if err:
            bad.append(f"{name}: {err}")
    xs8, v8, h8 = K.sepconv_inputs(d, 1, 1, 1, 51, 51, 13)
    xs, v, h = (K.tile_batch(t.cuda(), n).contiguous() for t in (xs8, v8, h8))
    err = K.first_mismatch(O.sepconv_func.apply(xs, v, h), K.tile_batch(R.sepconv(xs8, v8, h8), n))
    if err:
        bad.append(f"sepconv: {err}")
    del xs, v, h
    assert not bad, "\n".join(bad)


# ---- kernel forms selected by environment variables (read once per process): one child process each

VARIANTS = [("VFI_SPLAT_NHWC", "0", "splat"), ("VFI_OPS_TILED", "0", "volumes"), ("VFI_VOLUME_WARP", "1", "volumes"),
            ("VFI_SEPCONV_PY", "0", "sepconv"), ("VFI_SEPCONV_PY", "1", "sepconv"), ("VFI_SEPCONV_PY", "3", "sepconv")]
_CHILD = ("import sys; sys.path[:0] = [{here!r}, {root!r}]; import test_gpu_ops_exact as T; "
          "sys.exit(T.child_main(sys.argv[1]))")


@pytest.mark.parametrize("var,val,op", VARIANTS, ids=[f"{v}={x}" for v, x, _ in VARIANTS])
def test_env_variant(pkg, var, val, op):
    env = dict(os.environ, **{var: val})
    r = subprocess.run([sys.executable, "-c", _CHILD.format(here=HERE, root=ROOT), op], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
    report = (r.stdout[-6000:] + "\n" + r.stderr[-3000:]).strip()
    assert r.returncode == 0, f"{var}={val} {op}: child exited {r.returncode}\n{report}"
    assert f"{op}: 0 mismatching cases" in r.stdout, report

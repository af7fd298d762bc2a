"""Cases shared by the exact op tests on the host (test_ops_host.py, test_ops_extra_host.py) and on the GPU
(test_gpu_ops_exact.py): seeded inputs on small dyadic grids, the shape tables, the edge-flow table and a report of the
first mismatching element.

On these grids every product and every partial sum the ops form is exact in fp32, so every summation order - atomics in
any order, shared-memory tiles, Kahan steps, the oracle's float64 sums - gives the same fp32 number, and FMA contraction
changes nothing either.  A kernel must then equal the oracle bit for bit (torch.equal).  The one exception is soft mode:
exp(metric) is not exact, and the device's expf and the CPU's exp may differ in the last bits, so soft mode is held to
SOFT_TOL * max(1, max|ref|).  The final division of the weighted modes is IEEE-rounded identically on both sides.
"""
import torch

# ---- dyadic grids: value ranges and steps keep every sum of products below 2^24 units of the finest step


def grid(gen, shape, step, lo, hi):
    """Uniform values of step * Z in [lo, hi] (seeded through gen)."""
    k0, k1 = round(lo / step), round(hi / step)
    return torch.randint(k0, k1 + 1, tuple(shape), generator=gen).float() * step


SPLAT_MODES = ["sum", "avg", "avg-zeroeps", "avg-clipeps", "linear", "linear-zeroeps", "linear-clipeps",
               "soft", "soft-zeroeps", "soft-clipeps"]
SOFT_TOL = 1e-6


def splat_inputs(shape, mode, seed):
    """x in 1/8 Z [-4, 4], flow in 1/4 Z [-8, 8]; metric in 1/4 Z [0.25, 2] (linear) or [-0.75, 1] (soft), None for
    sum / avg."""
    n, c, h, w = shape
    g = torch.Generator().manual_seed(seed)
    x = grid(g, (n, c, h, w), 0.125, -4, 4)
    flow = grid(g, (n, 2, h, w), 0.25, -8, 8)
    base = mode.split("-")[0]
    metric = None
    if base == "linear":
        metric = grid(g, (n, 1, h, w), 0.25, 0.25, 2)
    elif base == "soft":
        metric = grid(g, (n, 1, h, w), 0.25, -0.75, 1)
    return x, flow, metric


def splat_tol(mode, ref):
    """0 (bit-exact) except for soft mode."""
    return SOFT_TOL * max(1.0, float(ref.abs().max())) if mode.startswith("soft") else 0.0


# (N, C, H, W): W and H off the 32 x 32 transpose tiles, C = 1 / 3 / 4 / 5 / 65 (channel padding to a multiple of 4, one
# and three 32-channel transpose tiles), N = 1 / 2 / 3, a 1 x 1 image, a single row and a single column
SPLAT_SHAPES = [(2, 3, 37, 53), (2, 65, 24, 40), (3, 1, 5, 7), (1, 5, 1, 1), (1, 4, 1, 70), (2, 3, 9, 1), (1, 4, 32, 32)]

# ---- the edge-flow table: flows at the borders, flows that leave the image by far (on the GPU float -> int conversion
# saturates at |x| >= 2^31 where x86 returns INT_MIN), and non-finite flows (the pixel is dropped)
INF, NAN = float("inf"), float("nan")
BORDER_IN = [-0.0, -0.25, -0.5, -1.0, 0.0, 0.25]   # at x = 0 / y = 0: -1 lands one corner on the border with weight 0
BORDER_OUT = [0.0, 0.25, 0.5, 1.0, -0.0, -0.25]    # at x = W-1 / y = H-1
FAR = [1e6, -1e6, 2.0 ** 31, -2.0 ** 31, 3e9, -3e9, 1e30, -1e30, INF, -INF, NAN]
EDGE_SHAPE = (2, 5, 9, 13)


def edge_splat_inputs(mode, seed):
    """splat_inputs at EDGE_SHAPE with the edge-flow table written over the flow: the border values along the four
    borders, every FAR value once in x and once in y on interior pixels (the other component stays dyadic)."""
    x, flow, metric = splat_inputs(EDGE_SHAPE, mode, seed)
    _, _, h, w = EDGE_SHAPE
    for y in range(h):
        flow[:, 0, y, 0] = BORDER_IN[y % len(BORDER_IN)]
        flow[:, 0, y, w - 1] = BORDER_OUT[y % len(BORDER_OUT)]
    for xx in range(w):
        flow[:, 1, 0, xx] = BORDER_IN[xx % len(BORDER_IN)]
        flow[:, 1, h - 1, xx] = BORDER_OUT[xx % len(BORDER_OUT)]
    interior = [(y, xx) for y in range(1, h - 1) for xx in range(1, w - 1)]
    for i, v in enumerate(FAR):
        y, xx = interior[2 * i]
        flow[:, 0, y, xx] = v
        y, xx = interior[2 * i + 1]
        flow[:, 1, y, xx] = v
    return x, flow, metric


def volume_inputs(shape, seed):
    """Integers in [-8, 8] for both volumes (costvol L1 and dot correlation)."""
    g = torch.Generator().manual_seed(seed)
    return grid(g, shape, 1, -8, 8), grid(g, shape, 1, -8, 8)


# W and H off the 32 x 8 volume tile, C = 1 / 3 / 4 / 5 / 7 / 20 / 33 / 65 (partial and whole kVolCh = 8 channel chunks;
# 20 / 33 / 65 are not multiples of the 32 lanes of the warp form), N = 1 / 2 / 3, 1 x 1, one row, one column
VOLUME_SHAPES = [(2, 7, 13, 37), (1, 20, 9, 33), (3, 33, 5, 7), (1, 1, 1, 1), (1, 65, 10, 40), (2, 4, 1, 45),
                 (1, 3, 17, 1), (2, 5, 8, 32)]


def sepconv_inputs(n, c, h, w, kv, kh, seed):
    """x in 1/4 Z [-2, 2] (padded size), ver / hor in 1/16 Z [-1, 1]."""
    g = torch.Generator().manual_seed(seed)
    x = grid(g, (n, c, h + kv - 1, w + kh - 1), 0.25, -2, 2)
    ver = grid(g, (n, kv, h, w), 1 / 16, -1, 1)
    hor = grid(g, (n, kh, h, w), 1 / 16, -1, 1)
    return x, ver, hor


# (N, C, H, W, Kv, Kh).  K = 51 takes the tiled kernel: H off 8 * PY for PY = 1, 2, 3 (19, 25), W off 32, C = 1 / 3 / 4 / 5
# (one partial or whole four-channel pass, then a second pass); other sizes take the generic kernel, including Kv != Kh
SEPCONV_SHAPES = [(1, 4, 19, 45, 51, 51), (2, 5, 25, 33, 51, 51), (1, 1, 1, 1, 51, 51), (3, 3, 1, 40, 51, 51),
                  (2, 3, 9, 7, 5, 5), (1, 6, 8, 8, 13, 13), (2, 5, 7, 9, 5, 13), (1, 4, 6, 11, 13, 5), (1, 1, 1, 1, 3, 1)]


def adacof_inputs(n, c, ho, wo, f, dil, seed):
    """x in 1/8 Z [-4, 4], weights in 1/8 Z [-1, 1], offsets in 1/4 Z [-6, 6] (negative fractions: (int) truncates toward
    zero, so the kernel's fractions are negative there, as in the reference)."""
    g = torch.Generator().manual_seed(seed)
    hin, win = ho + (f - 1) * dil, wo + (f - 1) * dil
    x = grid(g, (n, c, hin, win), 0.125, -4, 4)
    w = grid(g, (n, f * f, ho, wo), 0.125, -1, 1)
    oi = grid(g, (n, f * f, ho, wo), 0.25, -6, 6)
    oj = grid(g, (n, f * f, ho, wo), 0.25, -6, 6)
    return x, w, oi, oj


# (N, C, Ho, Wo, F, dilation): C = 9 / 11 are one whole and one partial eight-channel sweep
ADACOF_SHAPES = [(2, 3, 6, 7, 3, 1), (2, 11, 6, 7, 5, 2), (1, 1, 1, 1, 3, 1), (3, 9, 5, 9, 4, 1)]

# more images than a grid's z dimension holds (65535): the splat, the volumes and the K = 51 sepconv switch kernels there
BIG_N = 65536
BIG_DISTINCT = 8


def tile_batch(t, n):
    """t's batch repeated, cut at n images: a big batch whose oracle is run on the few distinct images only."""
    return t.repeat(-(-n // t.shape[0]), *([1] * (t.dim() - 1)))[:n]


def first_mismatch(got, ref, tol=0.0):
    """None when got equals ref (tol = 0: bit for bit, NaN only against NaN) or is within tol everywhere; else one line
    naming the number of bad elements, the largest error and the first bad element (n, c, y, x) with both values."""
    got = got.detach().cpu()
    ref = ref.detach().cpu()
    if got.shape != ref.shape:
        return f"shape {tuple(got.shape)} != reference {tuple(ref.shape)}"
    both_nan = got.isnan() & ref.isnan()
    err = (got.double() - ref.double()).abs()
    bad = ~both_nan & ~(err <= tol)
    if tol == 0.0:
        bad = ~both_nan & (got != ref)
    if not bad.any():
        return None
    idx = tuple(int(i) for i in bad.nonzero()[0])
    finite = err[bad & err.isfinite()]
    worst = float(finite.max()) if finite.numel() else float("nan")
    return (f"{int(bad.sum())} of {bad.numel()} elements differ (tol {tol:.3g}), max |err| {worst:.6g}; first at "
            f"{idx}: got {float(got[idx])!r}, ref {float(ref[idx])!r}")

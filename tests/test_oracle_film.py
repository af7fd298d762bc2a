"""Pin the FILM oracle (oracle/film.py) to outputs of the unmodified reference (tests/golden/film_*.npz, made by
tools/make_golden_film.py in the build container)."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from make_golden_film import film_cases, film_inputs  # noqa: E402
from oracle import film as OF  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
pytestmark = pytest.mark.usefixtures("golden_cpu_threads")


@pytest.mark.parametrize("name", sorted(film_cases().keys()))
def test_film_oracle_matches_reference_output(name):
    cfg = film_cases()[name]
    gold = np.load(os.path.join(GOLD, name + ".npz"))
    ref = torch.from_numpy(gold["out"])
    sd = OF.synthetic_state_dict(cfg["seed"], cfg["flow_gain"])
    fr = film_inputs(cfg)
    if cfg["kind"] == "net":
        x = fr.permute(0, 3, 1, 2)
        dbg = {}
        out = OF.interpolator_forward(sd, x[0:1], x[1:2], torch.full((1, 1), 0.5), debug=dbg)
        for l in range(OF.FUSION_PYRAMID_LEVELS):
            assert (dbg["forward_flow"][l] - torch.from_numpy(gold[f"fwd_flow{l}"])).abs().max().item() <= 1e-5
            assert (dbg["backward_flow"][l] - torch.from_numpy(gold[f"bwd_flow{l}"])).abs().max().item() <= 1e-5
    else:
        out = OF.film_vfi(sd, fr, multiplier=cfg["multiplier"], states=cfg["states"])
    assert out.shape == ref.shape
    # same ATen CPU kernels in the same order
    assert (out - ref).abs().max().item() <= 1e-6
    if cfg["kind"] == "node":
        assert torch.equal(out[-1], fr[-1, ..., :3])  # film/__init__.py:104: the last frame is passed through


def test_film_state_dict_spec():
    spec = OF.state_dict_spec()
    assert len(spec) == 82
    assert sum(int(np.prod(s)) for _, s in spec) == 34436667  # SURVEY.md section 8 a10 / appendix B
    shapes = dict(spec)
    # the widest layers (film_arch.py:243-255: in_channels 1930 / 2442 / 1162 / 522 / 202)
    assert shapes["fuse.convs.0.0.weight"] == (512, 1930, 2, 2)
    assert shapes["fuse.convs.0.1.0.weight"] == (512, 2442, 3, 3)
    assert shapes["fuse.convs.3.1.0.weight"] == (64, 202, 3, 3)
    assert shapes["predict_flow._predictor._convs.0.0.weight"] == (256, 1920, 3, 3)
    assert shapes["predict_flow._predictors.2._convs.4.weight"] == (2, 16, 1, 1)


def test_film_inference_order():
    # film/__init__.py:12-42: 3 in-between frames = middle first, then the two quarters
    assert OF.inference_order(1) == [(0, 2, 1)]
    assert OF.inference_order(3) == [(0, 4, 2), (0, 2, 1), (2, 4, 3)]
    order = OF.inference_order(4)  # not a power of two: every new frame still comes from its current neighbours
    have = {0, 5}
    for lo, hi, new in order:
        assert lo in have and hi in have and lo < new < hi
        assert not any(lo < h < hi for h in have)
        have.add(new)
    assert have == set(range(6))


def test_film_warp_is_pixel_offset_sampling():
    # the normalisation of film_arch.py:704-723 reduces to sampling at (x + fx, y + fy) with border clamping
    g = torch.Generator().manual_seed(5)
    img = torch.rand(1, 3, 9, 13, generator=g)
    flow = torch.zeros(1, 2, 9, 13)
    flow[:, 0] = 2.0   # x
    flow[:, 1] = -1.0  # y
    out = OF.warp(img, flow)
    exp = torch.empty_like(img)
    for y in range(9):
        for x in range(13):
            exp[..., y, x] = img[..., min(max(y - 1, 0), 8), min(max(x + 2, 0), 12)]
    assert (out - exp).abs().max().item() <= 2e-6

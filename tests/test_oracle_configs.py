"""Pin the oracle at the sizes BASELINE.json quotes its numbers on: config 1 (the reference's demo pair at 540p through
the whole node) and the 1080p geometry of config 2 (padded 1088 x 1920) - against outputs of the UNMODIFIED reference
made by tools/make_golden_configs.py (16-bit fixed-point fixtures: half a quantisation step is 7.7e-6; on top of that
the 40-layer fp32 chain differs by up to ~6e-6 between oneDNN's batch-2 blocking, which made the fixture, and batch 1)."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from make_golden_configs import CFG1, CFG2, CROP, box8, crop_origins  # noqa: E402
from oracle import rife46 as O  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
pytestmark = pytest.mark.usefixtures("golden_cpu_threads")
QSTEP = 1.0 / 65535.0


def test_config1_demo_pair_540p():
    g = np.load(os.path.join(GOLD, "cfg1_anime_540p.npz"))
    fr = torch.from_numpy(g["frames_u8"]).float() / 255.0
    sd = O.synthetic_state_dict(CFG1["weight_seed"], CFG1["gain"], arch="4.6")
    out = O.rife_vfi(sd, fr, multiplier=CFG1["multiplier"])
    assert out.shape == (3, 540, 960, 3)
    assert torch.equal(out[0], fr[0]) and torch.equal(out[2], fr[1])
    ref = torch.from_numpy(g["mid_q16"].astype(np.float32)) * QSTEP
    assert (out[1] - ref).abs().max().item() <= 0.5 * QSTEP + 1e-5


def test_config2_geometry_1080p_arch46():
    g = np.load(os.path.join(GOLD, "cfg2_1080p_arch46.npz"))
    fr = O.synthetic_clip(2, CFG2["h"], CFG2["w"], seed=CFG2["clip_seed"])
    x = fr.permute(0, 3, 1, 2)
    sd = O.synthetic_state_dict(CFG2["weight_seed"], CFG2["gain"], arch="4.6")
    ts = torch.tensor(CFG2["ts"][:1], dtype=torch.float32).view(-1, 1, 1, 1)  # one timestep keeps the CPU suite short
    out = O.ifnet_forward("4.6", sd, x[0:1], x[1:2], ts).clamp(0, 1).permute(0, 2, 3, 1).numpy()
    crops = g["crops_q16"].astype(np.float32) * QSTEP
    for i, (y, x0) in enumerate(crop_origins(CFG2["h"], CFG2["w"])):
        assert np.abs(out[0, y:y + CROP, x0:x0 + CROP] - crops[0, i]).max() <= 0.5 * QSTEP + 1e-5, i
    assert np.abs(box8(out)[0] - g["box8_q16"][0].astype(np.float32) * QSTEP).max() <= 0.5 * QSTEP + 1e-5

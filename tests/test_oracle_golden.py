"""Pin the oracle: oracle/rife46.py vs outputs of the unmodified reference (tests/golden/*.npz,
made by tools/make_golden.py in the build container)."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from make_golden import cases, make_inputs  # noqa: E402
from oracle import rife46 as O  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
pytestmark = pytest.mark.usefixtures("golden_cpu_threads")


@pytest.mark.parametrize("name", sorted(cases().keys()))
def test_oracle_matches_reference_output(name):
    cfg = cases()[name]
    ref = torch.from_numpy(np.load(os.path.join(GOLD, name + ".npz"))["out"])
    arch = cfg.get("arch", "4.6")
    sd = O.synthetic_state_dict(cfg["seed"], cfg["gain"], arch=arch)
    fr = make_inputs(cfg)
    if cfg["kind"] == "ifnet":
        x = fr.permute(0, 3, 1, 2)
        b = len(cfg["ts"])
        ts = torch.tensor(cfg["ts"], dtype=torch.float32).view(-1, 1, 1, 1)
        sl = [v / cfg.get("scale_factor", 1.0) for v in O.SCALE_LIST[arch]]
        out = O.ifnet_forward(arch, sd, x[0:1].repeat(b, 1, 1, 1), x[1:2].repeat(b, 1, 1, 1), ts, sl)
    else:
        out = O.rife_vfi(sd, fr, multiplier=cfg["multiplier"], states=cfg["states"], arch=arch)
    assert out.shape == ref.shape
    # same ATen CPU kernels in the same order: agreement is at rounding level
    assert (out - ref).abs().max().item() <= 1e-6
    if cfg["kind"] == "node":
        # pass-through frames are bit exact (rife/__init__.py:227-230)
        assert torch.equal(out[0], fr[0, ..., :3])
        assert torch.equal(out[-1], fr[-1, ..., :3])


def test_state_dict_spec_matches_reference_layout():
    spec = O.state_dict_spec()
    assert len(spec) == 120
    assert sum(int(np.prod(s)) for _, s in spec) == 5306256  # SURVEY.md section 8 a4
    sd = O.synthetic_state_dict(0)
    assert list(sd.keys()) == [n for n, _ in spec]


def test_task_schedule():
    # rife/__init__.py:164-174
    tasks, mults = O.build_tasks(4, 3, ([1], True))
    assert mults == [3, 3, 3]
    assert tasks == [(0, 1 / 3), (0, 2 / 3), (2, 1 / 3), (2, 2 / 3)]
    tasks, mults = O.build_tasks(5, [2, 1, 3], None)
    assert mults == [2, 1, 3, 2]
    assert tasks == [(0, 0.5), (2, 1 / 3), (2, 2 / 3), (3, 0.5)]
    tasks, _ = O.build_tasks(4, 2, ([0, 2], False))
    assert [p for p, _ in tasks] == [0, 2]

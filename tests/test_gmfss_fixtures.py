"""GMFSS (SURVEY.md section 8 row a11) is not built yet; what exists are its target vectors: outputs of the unmodified
reference model on seeded weights (tools/make_golden_gmfss.py).  These tests keep the fixtures honest: the weight recipe is
deterministic and reference-free, the stored spec of the reference's five state_dicts agrees with the IFNet layout and the
stored flows / frames are finite and non-trivial."""
import os

import numpy as np
import pytest
import torch

from oracle import gmfss_weights as GW

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def test_weight_recipe_is_deterministic_and_complete():
    a, b = GW.synthetic_state_dicts(0), GW.synthetic_state_dicts(0)
    counts = {net: sum(v.numel() for v in a[net].values() if v.dtype == torch.float32) for net in GW.NETS}
    assert counts["ifnet"] == 5306256                       # IFNet("4.6"), SURVEY.md section 8 a4
    assert 4.6e6 < counts["flownet"] < 4.8e6 and 7.8e6 < counts["fusionnet"] < 7.9e6   # section 8 a11: 4.72 M, 7.84 M
    for net in GW.NETS:
        for k in a[net]:
            assert torch.equal(a[net][k], b[net][k])
    c = GW.synthetic_state_dicts(1)
    assert not torch.equal(a["feat_ext"][next(iter(a["feat_ext"]))], c["feat_ext"][next(iter(c["feat_ext"]))])


@pytest.mark.parametrize("name,shape", [("gmfss_96x128_t0.5", (1, 3, 96, 128)), ("gmfss_70x100_t0.3", (1, 3, 70, 100))])
def test_goldens_are_sane(name, shape):
    g = np.load(os.path.join(GOLD, name + ".npz"))
    assert g["out"].shape == shape and np.isfinite(g["out"]).all()
    assert g["out"].min() >= 0.0 and g["out"].max() <= 1.0 and g["out"].std() > 0.05      # clamped frame with structure
    ph, pw = ((shape[2] - 1) // 64 + 1) * 64, ((shape[3] - 1) // 64 + 1) * 64
    for k in ("flow01", "flow10"):
        assert g[k].shape == (1, 2, ph // 2, pw // 2) and np.isfinite(g[k]).all() and np.abs(g[k]).max() > 1.0
    for k in ("metric0", "metric1"):
        assert g[k].shape == (1, 1, ph // 2, pw // 2)


def test_spec_matches_the_reference_ifnet():
    """The ifnet entry of the spec must be the IFNet("4.6") layout this repo already runs on the GPU."""
    from oracle import rife46 as O
    spec = GW.load_spec()
    assert [(n, tuple(s)) for n, s, _ in spec["ifnet"]] == [(n, tuple(s)) for n, s in O.state_dict_spec("4.6")]

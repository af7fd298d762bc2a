"""CPU-side checks: the C-ABI library loads and exports every symbol include/vfi_b200.h declares; the node
surface matches the reference's; no compute calls (no GPU here)."""
import ctypes
import json
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol(pkg):
    from cfi_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "vfi_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(vfi_[a-z0-9_]+)\s*\(", hdr)))
    assert declared == sorted(_lib.SYMBOLS)
    L = ctypes.CDLL(_lib.LIB_PATH)
    for s in declared:
        assert hasattr(L, s), s
    assert b"sm_100a" in _lib.lib().vfi_version()


def test_no_gpu_is_a_loud_error(pkg):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from cfi_b200._lib import VfiError, lib
    from cfi_b200.engine import Rife46Engine
    with pytest.raises(VfiError):
        Rife46Engine({}, 0)
    ctx = ctypes.c_void_p()
    assert lib().vfi_create(0, ctypes.byref(ctx)) != 0
    assert len(lib().vfi_last_error()) > 0


def test_null_context_is_refused_before_any_cuda_call(pkg):
    """Error behaviour of the boundary without a GPU: every entry point that takes a context refuses a NULL one with
    VFI_E_INVALID (-1) and leaves a message; nothing is launched (include/vfi_b200.h: error convention)."""
    from cfi_b200._lib import lib
    L = lib()
    names = ["vfi_set_batch", "vfi_sync", "vfi_rife_load", "vfi_rife46_load", "vfi_rife46_forward", "vfi_rife46_interpolate_host",
             "vfi_warp_bilinear_border", "vfi_softsplat_sum", "vfi_softsplat_weighted", "vfi_costvol_l1", "vfi_corr_dot",
             "vfi_sepconv", "vfi_adacof", "vfi_edt_pass", "vfi_film_load", "vfi_film_forward", "vfi_sepconv_load",
             "vfi_sepconv_forward"]
    for name in names:
        fn = getattr(L, name)
        assert fn.argtypes, name
        args = []
        for t in fn.argtypes:                       # NULL for every pointer (the context first), 1 / 1.0 for scalars
            if t in (ctypes.c_float, ctypes.c_double):
                args.append(1.0)
            elif t in (ctypes.c_int, ctypes.c_int32, ctypes.c_int64, ctypes.c_size_t):
                args.append(1)
            else:
                args.append(None)
        rc = fn(*args)
        assert rc == -1, (name, rc)
        assert len(L.vfi_last_error()) > 0, name


def test_node_surface_matches_reference(pkg):
    """rife/__init__.py:36-75 and root __init__.py:23-47."""
    import cfi_b200 as P
    import cfi_b200.node as N
    assert P.NODE_CLASS_MAPPINGS["RIFE VFI"] is N.RIFE_VFI
    it = N.RIFE_VFI.INPUT_TYPES()
    assert list(it["required"].keys()) == ["ckpt_name", "frames", "clear_cache_after_n_frames", "multiplier",
                                           "fast_mode", "ensemble", "scale_factor", "dtype", "torch_compile",
                                           "batch_size"]
    assert it["required"]["frames"] == ("IMAGE",)
    assert it["required"]["clear_cache_after_n_frames"][1] == {"default": 10, "min": 1, "max": 1000}
    assert it["required"]["scale_factor"][0] == [0.25, 0.5, 1.0, 2.0, 4.0]
    assert it["required"]["dtype"][0] == ["float32", "float16", "bfloat16"]
    assert it["optional"] == {"optional_interpolation_states": ("INTERPOLATION_STATES",)}
    assert N.RIFE_VFI.RETURN_TYPES == ("IMAGE",) and N.RIFE_VFI.FUNCTION == "vfi"
    assert N.RIFE_VFI.CATEGORY == "ComfyUI-Frame-Interpolation/VFI"
    assert "rife46.pth" in it["required"]["ckpt_name"][0]


def test_task_builder_matches_oracle(pkg):
    import cfi_b200.node as N
    from oracle import rife46 as O
    for mult, states in [(3, ([1], True)), ([2, 1, 3], None), (2, ([0, 2], False)), (1, None), ([0, 4], None)]:
        st = None if states is None else N.InterpolationStateList(list(states[0]), states[1])
        assert N.build_tasks(4, mult, st) == O.build_tasks(5, mult, states)
    (lst,) = N.MakeInterpolationStateList().create_options("1, 2,3", True)
    assert lst.is_frame_skipped(2) and not lst.is_frame_skipped(0)
    assert N.FloatToInt().convert(2.7) == (2,) and N.FloatToInt().convert([1.2, 3.9]) == ([1, 3],)


def test_missing_checkpoint_is_an_error(pkg, monkeypatch, tmp_path):
    import cfi_b200.node as N
    monkeypatch.setenv("VFI_CKPT_DIR", str(tmp_path))
    with pytest.raises(Exception):
        N.load_file_from_github_release("rife", "rife46.pth")


def test_state_dict_layouts_agree(pkg):
    """The C header's tensor counts, the host's name lists and the oracle's reference-derived specs (checked against
    the unmodified reference by tools/make_golden.py's load_state_dict) describe the same checkpoints."""
    from cfi_b200.engine import ARCH_CODE, state_dict_names
    from oracle import rife46 as O
    hdr = open(os.path.join(ROOT, "include", "vfi_b200.h")).read()
    counts = {int(a): int(n) for a, n in re.findall(r"#define VFI_RIFE(\d+)_NUM_TENSORS (\d+)", hdr)}
    for arch, code in ARCH_CODE.items():
        spec = O.state_dict_spec(arch)
        assert state_dict_names(arch) == [n for n, _ in spec], arch
        assert counts[code] == len(spec), arch
    assert [c for _, c in O.BLOCK_SPECS_426] == [192, 128, 96, 64, 32]
    assert len(O.SCALE_LIST["4.26"]) == 5 and set(ARCH_CODE) == set(O.SCALE_LIST)


def test_ops_module_has_every_name_the_reference_exports(pkg):
    """vfi_models/ops/__init__.py:19-21: the twelve names the reference re-exports from its cupy / taichi backends (and its
    models import, e.g. gmfss_fortuna/GMFSS_Fortuna_union_arch.py:28, stmfnet/stmfnet_arch.py:28, eisai/eisai_arch.py:53);
    `sys.modules["vfi_models.ops"] = cfi_b200.ops` is the drop-in for those models (INTEGRATION.md section 6)."""
    import cfi_b200.ops as ops
    names = ["softsplat", "ModuleSoftsplat", "FunctionSoftsplat", "softsplat_func", "costvol_func", "sepconv_func", "init",
             "batch_edt", "FunctionAdaCoF", "ModuleCorrelation", "FunctionCorrelation", "_FunctionCorrelation"]
    for n in names:
        assert hasattr(ops, n), n
    with open(os.path.join(ROOT, "tests", "golden", "ops_exports.json")) as fh:   # the reference's list (tools/make_golden_ops.py)
        assert json.load(fh)["names"] == sorted(names)

#!/usr/bin/env python
"""Generate tests/golden/ops_ref_kernels.npz and tests/golden/ops_exports.json from the UNMODIFIED reference's op kernels.

    VFI_REFERENCE=<reference checkout> python tools/make_golden_ops.py

``oracle/ref_ops.py`` runs the reference's own cupy kernel strings on the CPU (its pre-processor, compiled behind
tests/host_emu).  Every case of ``tests/test_ops_ref_pinned.py`` is run through it here and its seeded inputs and the
kernel's output are stored as ``<case>:<name>`` arrays, so that test holds ``oracle/ops_ref.py`` to the reference
kernels without the reference being present.  ``ops_exports.json`` is the list of names the reference's
``vfi_models/ops/__init__.py`` re-exports (tests/test_capi_cpu.py).
"""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_ops  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
NPZ = os.path.join(GOLD, "ops_ref_kernels.npz")
EXPORTS = os.path.join(GOLD, "ops_exports.json")

# parameters of tests/test_ops_ref_pinned.py
SOFTSPLAT = [((1, 3, 9, 13), 1.5), ((2, 5, 8, 8), 6.0)]
COSTVOL = [(1, 8, 6, 7), (2, 3, 10, 5)]
SEPCONV = [(5, (6, 7)), (51, (4, 3))]
CORRELATION = [(1, 40, 5, 6), (2, 7, 4, 9)]
ADACOF = [(3, 1), (5, 2)]


def case(kind, *params) -> str:
    return kind + "_" + "_".join(str(p).replace(" ", "") for p in params)


def cases():
    """case name -> (seeded inputs, the reference kernel's outputs on them)."""
    out = {}
    for shape, mag in SOFTSPLAT:
        g = torch.Generator().manual_seed(shape[1])
        x = torch.randn(*shape, generator=g)
        flow = (torch.rand(shape[0], 2, shape[2], shape[3], generator=g) - 0.5) * 2 * mag   # some targets fall outside
        out[case("softsplat_sum", shape, mag)] = (dict(x=x, flow=flow), dict(out=ref_ops.softsplat_out(x, flow)))

    g = torch.Generator().manual_seed(1)
    x = torch.randn(1, 4, 7, 9, generator=g)
    flow = (torch.rand(1, 2, 7, 9, generator=g) - 0.5) * 5
    metric = torch.randn(1, 1, 7, 9, generator=g) * 0.3
    avg = ref_ops.softsplat_out(torch.cat([x, x.new_ones(1, 1, 7, 9)], 1), flow)
    soft = ref_ops.softsplat_out(torch.cat([x * metric.exp(), metric.exp()], 1), flow)
    out["softsplat_modes"] = (dict(x=x, flow=flow, metric=metric), dict(avg=avg, soft=soft))

    for shape in COSTVOL:
        g = torch.Generator().manual_seed(shape[2])
        one, two = torch.randn(*shape, generator=g), torch.randn(*shape, generator=g)
        out[case("costvol", shape)] = (dict(one=one, two=two), dict(out=ref_ops.costvol_out(one, two)))

    for k, hw in SEPCONV:
        g = torch.Generator().manual_seed(k)
        x = torch.randn(1, 4, hw[0] + k - 1, hw[1] + k - 1, generator=g)
        ver, hor = torch.randn(1, k, *hw, generator=g), torch.randn(1, k, *hw, generator=g)
        out[case("sepconv", k, hw)] = (dict(x=x, ver=ver, hor=hor), dict(out=ref_ops.sepconv_out(x, ver, hor)))

    for shape in CORRELATION:
        g = torch.Generator().manual_seed(shape[1])
        a, b = torch.randn(*shape, generator=g), torch.randn(*shape, generator=g)
        out[case("correlation", shape)] = (dict(a=a, b=b), dict(out=ref_ops.correlation(a, b)))

    for f, dil in ADACOF:
        g = torch.Generator().manual_seed(f)
        n, c, ho, wo = 2, 3, 6, 7
        x = torch.randn(n, c, ho + (f - 1) * dil, wo + (f - 1) * dil, generator=g)
        w = torch.randn(n, f * f, ho, wo, generator=g)
        oi = torch.randn(n, f * f, ho, wo, generator=g) * 2.5      # negative offsets: (int) truncation != floor
        oj = torch.randn(n, f * f, ho, wo, generator=g) * 2.5
        out[case("adacof", f, dil)] = (dict(x=x, w=w, oi=oi, oj=oj), dict(out=ref_ops.adacof(x, w, oi, oj, dil)))

    g = torch.Generator().manual_seed(2)
    img = (torch.rand(2, 9, 12, generator=g) > 0.85).float()
    img[1] = 0                                                   # empty image: defaults to the diameter
    diam2 = 9 ** 2 + 12 ** 2
    data = (1 - img) * diam2
    out["edt"] = (dict(img=img, data=data), dict(out=ref_ops.edt_pass(data, diam2)))
    return out


def exported_op_names():
    """The names vfi_models/ops/__init__.py re-exports from its cupy backend."""
    with open(os.path.join(ref_ops.REF, "vfi_models", "ops", "__init__.py")) as fh:
        line = [ln for ln in fh if "from .cupy_ops import" in ln][0]
    return sorted(x.strip() for x in line.split("import", 1)[1].split(","))


def main():
    if not ref_ops.available():
        sys.exit(f"reference op kernels not found under {ref_ops.REF} (set VFI_REFERENCE)")
    arrays = {}
    for name, (inputs, outputs) in cases().items():
        for k, v in {**inputs, **outputs}.items():
            arrays[f"{name}:{k}"] = v.numpy()
    np.savez_compressed(NPZ, **arrays)
    with open(EXPORTS, "w") as fh:
        json.dump({"source": "vfi_models/ops/__init__.py", "names": exported_op_names()}, fh, indent=1)
        fh.write("\n")
    print(NPZ, len(arrays), "arrays;", EXPORTS)


if __name__ == "__main__":
    main()

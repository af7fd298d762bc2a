"""The reference's OWN op kernels, executed on the CPU.  TEST INFRASTRUCTURE ONLY (build container only).

The reference's custom ops are CUDA C strings launched through cupy (``vfi_models/ops/cupy_ops/{softsplat,costvol,
sepconv}.py``); neither cupy nor a GPU exists in the build container, which left ``oracle/ops_ref.py`` (the CPU
restatements the GPU tests check the sm_100a op kernels against) pinned only to a reading of those strings.  This module
closes that gap without copying any reference source into the repo:

  1. the reference modules are imported from ``/root/reference`` as they are (with a stub ``cupy`` module: only
     ``import cupy`` has to succeed) and the reference's own pre-processor ``cupy_ops/utils.py:cuda_kernel`` specialises the
     reference's own kernel string for the given tensors (sizes and strides are baked into the source, :124-209);
  2. that source - plain C with a grid-stride loop over ``blockIdx / blockDim / gridDim`` - is written to
     ``oracle/_ref/<kernel>_<hash>.cpp`` behind ``tests/host_emu/cuda_shim.h`` and compiled with g++ into
     ``oracle/_ref/`` (git-ignored build products, like the task's recipe for compiled references asks);
  3. the kernel runs on CPU tensors through ctypes exactly as ``cuda_launch`` would run it on the device
     (``args = [n, data pointers...]``, one emulated thread walking the whole grid-stride range).

``tools/make_golden_ops.py`` stores these outputs in ``tests/golden/ops_ref_kernels.npz`` and
``tests/test_ops_ref_pinned.py`` holds ``oracle/ops_ref.py`` to them, which makes the chain
reference kernel source -> oracle -> sm_100a kernels (GPU tests) complete for softsplat_out, costvol_out and sepconv_out.
``kernel_Correlation_rearrange`` / ``_updateOutput`` (blocks of cooperating threads, shared memory, ``__syncthreads``) run
through a second shim, ``tests/host_emu/block_emu.h``: every thread of a block is a fiber and ``__syncthreads()`` yields to
a round-robin scheduler, i.e. the block advances barrier phase by barrier phase in thread order (warp lock-step).
Nothing here runs on the GPU box (``/root/reference`` does not exist there) and nothing here is product code.
"""
from __future__ import annotations

import ctypes
import hashlib
import importlib
import os
import subprocess
import sys
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("VFI_REFERENCE", "/root/reference")
OUT = os.path.join(ROOT, "oracle", "_ref")
SHIM = os.path.join(ROOT, "tests", "host_emu", "cuda_shim.h")
CUDA_INC = "/usr/local/cuda/include"
_mods = {}


def available() -> bool:
    return os.path.isdir(os.path.join(REF, "vfi_models", "ops", "cupy_ops")) and os.path.exists(
        os.path.join(CUDA_INC, "cuda_runtime.h"))


def _ref_module(name: str):
    """vfi_models/ops/cupy_ops/<name>.py of the reference, unmodified."""
    if name in _mods:
        return _mods[name]
    if "cupy" not in sys.modules:                       # `import cupy` at cupy_ops/utils.py:1 - never called here
        stub = types.ModuleType("cupy")
        stub.int32 = int
        stub.float32 = float
        stub.memoize = lambda **kw: (lambda f: f)        # decorator at cupy_ops/utils.py:228 (cuda_launch; never called)
        sys.modules["cupy"] = stub
    if "comfy.model_management" not in sys.modules:     # cupy_ops/__init__.py:6
        comfy = types.ModuleType("comfy")
        mm = types.ModuleType("comfy.model_management")
        mm.get_torch_device = lambda: torch.device("cpu")
        mm.soft_empty_cache = lambda *a, **k: None
        mm.is_nvidia = lambda: False
        mm.get_torch_device_name = lambda d: str(d)
        comfy.model_management = mm
        sys.modules["comfy"] = comfy
        sys.modules["comfy.model_management"] = mm
    ops_dir = os.path.join(REF, "vfi_models", "ops")
    if ops_dir not in sys.path:
        sys.path.insert(0, ops_dir)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        _mods[name] = importlib.import_module("cupy_ops." + name)
    utils = importlib.import_module("cupy_ops.utils")
    utils.objCudacache.setdefault("device", "host-emulation")   # cuda_kernel asks torch.cuda for a name otherwise (:29-31)
    return _mods[name]


def _compile(kernel_name: str, source: str) -> ctypes.CDLL:
    os.makedirs(OUT, exist_ok=True)
    tag = hashlib.sha1(source.encode()).hexdigest()[:12]
    base = os.path.join(OUT, f"{kernel_name}_{tag}")
    if not os.path.exists(base + ".so"):
        with open(base + ".cpp", "w") as fh:
            fh.write(f'#include "{SHIM}"\n#include <cassert>\n#define __launch_bounds__(...)\n'
                     "using std::abs; using std::floor; using std::isfinite;\n"
                     "static inline float atomicAdd(float* p, float v) { const float o = *p; *p += v; return o; }\n"
                     + source)
        r = subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-pthread", "-I" + CUDA_INC, "-o", base + ".so",
                            base + ".cpp"], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("g++ failed on the specialised reference kernel:\n" + r.stderr[-3000:])
    return ctypes.CDLL(base + ".so")


def _run(module: str, kernel_name: str, variables: dict, order, out_name: str) -> torch.Tensor:
    mod = _ref_module(module)
    utils = importlib.import_module("cupy_ops.utils")
    key = utils.cuda_kernel(kernel_name, getattr(mod, kernel_name), variables)   # the reference's own pre-processor
    lib = _compile(kernel_name, utils.objCudacache[key]["strKernel"])
    fn = getattr(lib, kernel_name)
    out = variables[out_name]
    args = [ctypes.c_int(out.nelement())] + [ctypes.c_void_p(variables[n].data_ptr()) for n in order]
    fn(*args)   # blockIdx = 0, blockDim = gridDim = 1: the kernel's grid-stride loop walks [0, n)
    return out


def softsplat_out(ten_in: torch.Tensor, ten_flow: torch.Tensor) -> torch.Tensor:
    """softsplat_func.forward, cupy_ops/softsplat.py:199-224: out = zeros; launch softsplat_out(n, in, flow, out)."""
    ten_in, ten_flow = ten_in.contiguous().float(), ten_flow.contiguous().float()
    out = ten_in.new_zeros(ten_in.shape)
    return _run("softsplat", "softsplat_out", {"tenIn": ten_in, "tenFlow": ten_flow, "tenOut": out},
                ("tenIn", "tenFlow", "tenOut"), "tenOut")


def costvol_out(one: torch.Tensor, two: torch.Tensor) -> torch.Tensor:
    """costvol_func.forward, cupy_ops/costvol.py:134-170: out [N,81,H,W]; n = N*H*W threads."""
    one, two = one.contiguous().float(), two.contiguous().float()
    out = one.new_empty([one.shape[0], 81, one.shape[2], one.shape[3]])
    mod = _ref_module("costvol")
    utils = importlib.import_module("cupy_ops.utils")
    variables = {"intChans": one.shape[1], "tenOne": one, "tenTwo": two, "tenOut": out}
    key = utils.cuda_kernel("costvol_out", mod.costvol_out, variables)
    lib = _compile("costvol_out", utils.objCudacache[key]["strKernel"])
    n = one.shape[0] * one.shape[2] * one.shape[3]   # :157-160: one thread per (n, y, x)
    lib.costvol_out(ctypes.c_int(n), ctypes.c_void_p(one.data_ptr()), ctypes.c_void_p(two.data_ptr()),
                    ctypes.c_void_p(out.data_ptr()))
    return out


def sepconv_out(ten_in: torch.Tensor, ver: torch.Tensor, hor: torch.Tensor) -> torch.Tensor:
    """sepconv_func.forward, cupy_ops/sepconv.py:158-190: out [N,C,H,W] with H = min(ver, hor) sizes."""
    ten_in, ver, hor = ten_in.contiguous().float(), ver.contiguous().float(), hor.contiguous().float()
    out = ten_in.new_empty([ten_in.shape[0], ten_in.shape[1], ver.shape[2] and hor.shape[2], ver.shape[3] and hor.shape[3]])
    return _run("sepconv", "sepconv_out", {"tenIn": ten_in, "tenVer": ver, "tenHor": hor, "tenOut": out},
                ("tenIn", "tenVer", "tenHor", "tenOut"), "tenOut")


def correlation(first: torch.Tensor, second: torch.Tensor) -> torch.Tensor:
    """_FunctionCorrelation.forward, cupy_ops/correlation.py:231-296: two rearrange launches (grid (ceil(HW/16), C, N), block
    16) into zero-initialised padded NHWC buffers, then updateOutput (grid (W, H, N), block 32, C * 4 bytes of dynamic
    shared memory)."""
    first, second = first.contiguous().float(), second.contiguous().float()
    n_, c, h, w = first.shape
    rbot0 = first.new_zeros([n_, h + 8, w + 8, c])
    rbot1 = first.new_zeros([n_, h + 8, w + 8, c])
    out = first.new_zeros([n_, 81, h, w])
    mod = _ref_module("correlation")
    utils = importlib.import_module("cupy_ops.utils")
    src = ""
    for name, var in (("kernel_Correlation_rearrange", {"input": first, "output": rbot0}),
                      ("kernel_Correlation_updateOutput", {"rbot0": rbot0, "rbot1": rbot1, "top": out})):
        key = utils.cuda_kernel(name, getattr(mod, name), var)      # the reference's own pre-processor
        src += utils.objCudacache[key]["strKernel"]
    # the only textual change: CUDA's dynamic shared memory declaration becomes the emulation's buffer
    src = src.replace("extern __shared__ char patch_data_char[];", "char* patch_data_char = emu_dyn_smem;")
    driver = """
extern "C" void emu_correlation(int N, int C, int H, int W, const float* first, const float* second, float* rbot0,
                                float* rbot1, float* out) {
  const int n = H * W;
  blockDim.x = 16;
  gridDim.x = (n + 15) / 16; gridDim.y = C; gridDim.z = N;
  for (int pass = 0; pass < 2; ++pass)
    for (unsigned z = 0; z < gridDim.z; ++z)
      for (unsigned y = 0; y < gridDim.y; ++y)
        for (unsigned x = 0; x < gridDim.x; ++x)
          for (unsigned t = 0; t < 16; ++t) {
            blockIdx.x = x; blockIdx.y = y; blockIdx.z = z; threadIdx.x = t;
            kernel_Correlation_rearrange(n, pass ? second : first, pass ? rbot1 : rbot0);
          }
  std::vector<char> smem((size_t)C * 4);
  emu_dyn_smem = smem.data();
  blockDim.x = 32;
  gridDim.x = W; gridDim.y = H; gridDim.z = N;
  for (unsigned z = 0; z < gridDim.z; ++z)
    for (unsigned y = 0; y < gridDim.y; ++y)
      for (unsigned x = 0; x < gridDim.x; ++x) {
        blockIdx.x = x; blockIdx.y = y; blockIdx.z = z;
        block_emu::run_block(32, [&]() { kernel_Correlation_updateOutput(81 * H * W, rbot0, rbot1, out); });
      }
}
"""
    os.makedirs(OUT, exist_ok=True)
    tag = hashlib.sha1((src + driver).encode()).hexdigest()[:12]
    base = os.path.join(OUT, f"correlation_{tag}")
    if not os.path.exists(base + ".so"):
        with open(base + ".cpp", "w") as fh:
            fh.write(f'#include "{os.path.join(ROOT, "tests", "host_emu", "block_emu.h")}"\n' + src + driver)
        r = subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-o", base + ".so", base + ".cpp"],
                           capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("g++ failed on the specialised reference kernel:\n" + r.stderr[-3000:])
    lib = ctypes.CDLL(base + ".so")
    vp = ctypes.c_void_p
    lib.emu_correlation(n_, c, h, w, vp(first.data_ptr()), vp(second.data_ptr()), vp(rbot0.data_ptr()), vp(rbot1.data_ptr()),
                        vp(out.data_ptr()))
    return out


def adacof(inp, weight, off_i, off_j, dilation: int) -> torch.Tensor:
    """FunctionAdaCoF.forward, cupy_ops/adacof.py:259-330: kernel_AdaCoF_updateOutput with F_SIZE / DILATION substituted."""
    inp, weight, off_i, off_j = [t.contiguous().float() for t in (inp, weight, off_i, off_j)]
    out = inp.new_zeros(inp.shape[0], inp.shape[1], weight.shape[2], weight.shape[3])
    mod = _ref_module("adacof")
    utils = importlib.import_module("cupy_ops.utils")
    f = int(round(weight.shape[1] ** 0.5))
    var = {"input": inp, "weight": weight, "offset_i": off_i, "offset_j": off_j, "output": out}
    key = utils.cuda_kernel("kernel_AdaCoF_updateOutput", mod.kernel_AdaCoF_updateOutput, var, F_SIZE=str(f),
                            DILATION=str(dilation))
    lib = _compile("kernel_AdaCoF_updateOutput", utils.objCudacache[key]["strKernel"])
    vp = ctypes.c_void_p
    lib.kernel_AdaCoF_updateOutput(ctypes.c_int(out.nelement()), vp(inp.data_ptr()), vp(weight.data_ptr()), vp(off_i.data_ptr()),
                                   vp(off_j.data_ptr()), vp(out.data_ptr()))
    return out


def edt_pass(data: torch.Tensor, diam2: float) -> torch.Tensor:
    """kernel_dt, cupy_ops/batch_edt.py:9-41 (a raw string, no pre-processing; one thread per element, no stride loop:
    every element index is emulated as its own block)."""
    mod = _ref_module("batch_edt")
    name, src = mod._batch_edt_kernel
    data = data.contiguous().float()
    bs, h, w = data.shape
    out = torch.zeros_like(data)
    driver = ("\nextern \"C\" void emu_dt(int bs, int h, int w, float diam2, float* data, float* out) {\n"
              "  blockDim.x = 1; gridDim.x = bs * h * w; threadIdx.x = 0;\n"
              "  for (int i = 0; i < bs * h * w; ++i) { blockIdx.x = i; kernel_dt(bs, h, w, diam2, data, out); }\n}\n")
    lib = _compile(name, src + driver)
    lib.emu_dt(bs, h, w, ctypes.c_float(diam2), ctypes.c_void_p(data.data_ptr()), ctypes.c_void_p(out.data_ptr()))
    return out

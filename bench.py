#!/usr/bin/env python
"""bench.py - interpolated frames/s of the RIFE-4.6 2x path at 1080p (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

One "step" = one pass of the hot path over one synthetic 64-frame 1080p clip per GPU (63 frame pairs, 2x ->
63 interpolated frames; SURVEY.md section 8d config 2 / BASELINE.json configs[1]).  Weak scaling: every rank
interpolates its own 64-frame shard of a (63*N+1)-frame clip (frame pairs are independent, one-frame halo),
and for N > 1 the interpolated frames are gathered on rank 0 over NCCL inside the timed region (the path's
only exchange step).
  value : whole-job interpolated frames/s with the clip already resident in HBM (CUDA events, max over ranks)
  e2e   : same metric through the plugin call a ComfyUI user makes - RIFE_VFI().vfi(ckpt, frames, multiplier=2) - with a
          PAGEABLE [64,1080,1920,3] fp32 input tensor and the node's own output tensor; H2D + D2H (and the host-side
          staging and pass-through copies) inside the timed region.  e2e_capi is the same through the bare C-ABI call
          on pre-pinned buffers (the r01 figure).
  roofline     : the dominant kernel (tcgen05 tap-conv, block-3 ResConv layer) timed alone, against the measured
                 bf16 tensor peak in MEASURED_PEAKS.json
  roofline_hbm : the HBM-bound kernels the step actually runs (block-3 / block-2 `front`, `final`), timed with CUDA
                 events on their launching stream inside real passes (vfi_rife_profile), against measured HBM bandwidth
  psnr_db      : the GPU's interpolated frames against the CPU leg's output on the CPU leg's sample of the same clip
  cpu_baseline : the CPU oracle port (oracle/rife46.py == the reference's PyTorch-CPU path, SURVEY.md F2) on the
                 host cores, on a bounded sample of the same clip (rank 0, N = 1 only)
--impl reference times that CPU port alone (all host threads), same metric / config.
--dump-outputs DIR writes the interpolated frames of the last timed step (every rank's, in rank order) to
DIR/interpolated_frames.npy: float32 [frames, pixels, 3] at the same seeded sample of pixel positions in every frame, so
that two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W, NFRAMES = 1080, 1920, 64
METRIC = "interpolated frames/sec @1080p RIFE-4.6 2x"
UNIT = "frames/s"
FLOPS_PER_FRAME = 175.245e9          # SURVEY.md section 8d (87.62 GMAC)
CPU_SAMPLE_FRAMES = 3                # 2 pairs of the same clip for the CPU legs (bounded sample)
CPU_ARCH = "4.6"
# N > 1: the shard's 63 pairs leave for rank 0 in this many chunks, each behind the kernels that produce it.  8 chunks = one
# internal pass of 8 pairs per chunk (r02: 16 chunks of 4 pairs made every pass half as wide - the latency-bound blocks 0 / 1
# cost the same per pass - and the step 4.7 ms slower than N = 1, whatever the transport)
GATHER_CHUNKS = int(os.environ.get("VFI_GATHER_CHUNKS", "8"))
DUMP_BYTES = 60_000_000              # --dump-outputs: size bound of the written sample (a 64-frame clip is 1.6 GB)
DUMP_SEED = 0


def frame_sample(frames, npix):
    """[n, H, W, 3] -> float32 CPU [n, npix, 3]: the same seeded pixel positions (raster order) of every frame."""
    import torch
    n, h, w, c = frames.shape
    pos = torch.randperm(h * w, generator=torch.Generator().manual_seed(DUMP_SEED))[:npix].sort().values
    return frames.reshape(n, h * w, c).index_select(1, pos.to(frames.device)).float().cpu()


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tflops=d["bf16_tflops"], tflops_sustained=d.get("bf16_tflops_sustained"),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, tflops=1590.0, tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            cells = [c.strip() for c in line.split(",")]
            try:  # nvidia-smi's own time stamp (local time), not the arrival time of a possibly buffered pipe
                import datetime
                ts = datetime.datetime.strptime(cells[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except Exception:
                ts = time.time()
            self.rows.append((ts, cells))

    def wait_first(self, timeout=3.0):
        """nvidia-smi needs ~1 s before its first row: block until the sampler is actually sampling."""
        t0 = time.time()
        while self.proc and not self.rows and time.time() - t0 < timeout:
            time.sleep(0.02)

    def stop(self, t_begin=None, t_end=None):
        """Median SM clock and throttle reasons of the samples taken inside [t_begin, t_end] (the timed region)."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        rows = [r for ts, r in self.rows if t_begin is None or t_begin <= ts <= t_end + 0.03]
        scope = "timed region"
        if not rows:  # region shorter than the sampling period: fall back to every sample of the run
            rows, scope = [r for _, r in self.rows], "whole run (no sample fell inside the timed region)"
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        # "under load" = samples above the idle clock
        load = [v for v in sm if v > 0.5 * max(sm)] if sm else []
        return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "scope": scope}


def _pick_threads(sd):
    """Host thread count for the CPU legs: the fastest of a few candidates on a small (270x480) pair.  "All the
    host threads it can use" is not os.cpu_count() on these boxes: oneDNN conv with 128 threads on a shared /
    cgroup-limited host is >10x slower than with 16-32 (measured r01), so the count is calibrated, then stated."""
    import torch
    from oracle import rife46 as O
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    cands = sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu})
    small = O.synthetic_clip(2, 270, 480, seed=7)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        O.rife_vfi(sd, small, multiplier=2, arch=CPU_ARCH)
        t0 = time.perf_counter()
        O.rife_vfi(sd, small, multiplier=2, arch=CPU_ARCH)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    return best, ncpu


def bind_to_gpu_numa_node(local_rank):
    """Multi-process runs: pin this rank's threads (and, by first touch, its host buffers) to the NUMA node its GPU hangs
    off.  r01: eight unbound ranks streaming pinned H2D + D2H at once reached 14.9 GB/s per direction per GPU against 41
    alone (GPU0-3 sit on node 0, GPU4-7 on node 1).  Returns a description for the JSON line, or None."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local_rank)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        if node < 0:
            return None
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus += list(range(int(lo), int(hi or lo) + 1))
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return {"gpu": local_rank, "pci": bdf, "numa_node": node, "cpus": len(allowed)}
    except Exception:
        return None


def cpu_port_fps(clip, sd, steps, warmup, min_seconds=0.0, keep=None):
    """The CPU restatement of the reference path (== reference PyTorch-CPU eager, fp32) on the host cores.
    Runs `steps` timed repetitions, and more until `min_seconds` of timed CPU work (at most 16 repetitions)."""
    import torch
    from oracle import rife46 as O
    threads, ncpu = _pick_threads(sd)
    torch.set_num_threads(threads)
    sample = clip[:CPU_SAMPLE_FRAMES].contiguous()
    times = []
    i = 0
    while i < warmup + steps or (sum(times) < min_seconds and len(times) < 16):
        t0 = time.perf_counter()
        res = O.rife_vfi(sd, sample, multiplier=2, arch=CPU_ARCH)
        dt = time.perf_counter() - t0
        if keep is not None:
            keep["out"] = res
        if i >= warmup:
            times.append(dt)
        i += 1
    n = CPU_SAMPLE_FRAMES - 1
    return n * len(times) / sum(times), sum(times) / len(times), threads, ncpu, len(times)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=8, help="pairs per internal pass (scheduling only)")
    ap.add_argument("--dtype", default="float32", help="node dtype: float32/float16 -> fp16 operands, bfloat16 -> bf16")
    ap.add_argument("--frames", type=int, default=NFRAMES)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--workload", default="rife", choices=["rife", "film", "sepconv", "gmfss"],
                    help="rife = the BASELINE.json metric (default).  film / sepconv: the side workloads of BASELINE configs[2] / "
                         "[4] through tools/bench_film.py / tools/bench_sepconv.py (same JSON-line contract, own metric name)")
    ap.add_argument("--arch", default="4.6", choices=["4.6", "4.7", "4.17", "4.26"],
                    help="RIFE arch (default 4.6 = the BASELINE.json metric; the others are side measurements)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a seeded sample of the last timed step's interpolated frames to DIR/interpolated_frames.npy")
    a, extra = ap.parse_known_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.workload != "rife" or a.impl != "b200"):
        ap.error("--dump-outputs is implemented for the default workload (--workload rife --impl b200)")
    if a.workload != "rife":  # the other model families keep their own harness; same launch convention (torchrun for N > 1)
        import runpy
        tool = {"film": "bench_film.py", "sepconv": "bench_sepconv.py", "gmfss": "bench_gmfss.py"}[a.workload]
        fwd = ["--steps", str(a.steps), "--warmup", str(a.warmup)] + (["--no-cpu"] if a.no_cpu else [])
        if a.workload != "gmfss" and a.frames != NFRAMES:
            fwd += ["--frames", str(a.frames)]
        sys.argv = [os.path.join(ROOT, "tools", tool)] + fwd + extra
        runpy.run_path(sys.argv[0], run_name="__main__")
        return
    if extra:
        ap.error("unrecognised arguments: " + " ".join(extra))

    import torch
    from oracle import rife46 as O

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.gpus != world and world > 1:
        a.gpus = world
    config = {"workload": f"RIFE {a.arch}, 2x multiplier, {a.frames}-frame synthetic 1080p clip per GPU (BASELINE configs[1])",
              "resolution": [H, W], "frames_per_gpu": a.frames, "pairs_per_gpu": a.frames - 1,
              "padded": [1088, 1920], "weights": "seeded synthetic (oracle.synthetic_state_dict(0)); no checkpoint ships",
              "parallelism": (f"frame-pair shards x{a.gpus}; each rank's output frames land on rank 0 over NVLink in {GATHER_CHUNKS} chunks behind the kernels that "
                              f"produce them ({'NCCL send/recv' if os.environ.get('VFI_GATHER', 'nccl') != 'push' else 'copy-engine pushes into an IPC-shared buffer, NCCL for the handle and the barriers'})")
              if a.gpus > 1 else "1 GPU",
              "l2": "inputs larger than L2 (1.6 GB clip, 1.6 GB output per step)", "batch": a.batch}

    sd = O.synthetic_state_dict(0, arch=a.arch)
    global CPU_ARCH
    CPU_ARCH = a.arch

    # ------------------------------------------------------------------ reference arm: CPU port only
    if a.impl == "reference":
        if rank != 0:
            return
        clip = O.synthetic_clip(CPU_SAMPLE_FRAMES, H, W, seed=1234)
        fps, sec, cores, ncpu, _reps = cpu_port_fps(clip, sd, max(a.steps, 1), max(a.warmup, 1))
        line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": 0, "steps": a.steps,
                "warmup": a.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": fps, "unit": UNIT, "cores": cores, "kind": "port",
                                 "sample": f"{CPU_SAMPLE_FRAMES - 1} pairs of the 1080p clip per step (bounded sample), "
                                           f"oracle/rife46.py = reference PyTorch-CPU path, {cores} threads (fastest of 8..{ncpu})"},
                "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ B200 arm
    import __graft_entry__ as ge
    ge.load_package()
    from cfi_b200.engine import Rife46Engine
    from cfi_b200 import _lib as cfi_lib

    torch.cuda.set_device(local_rank)
    # every rank (also the single one) runs on the cores of its GPU's NUMA node: host staging copies and the pinned
    # buffers then stay local to the PCIe root the GPU hangs off (what `numactl --cpunodebind` would do for a ComfyUI worker)
    numa = bind_to_gpu_numa_node(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    if rank == 0 and world > 1 and os.environ.get("VFI_NUM_SMS_RANK0"):
        # the gathering rank leaves a few SMs to NCCL's receive kernels (its persistent grids are sized for the rest)
        os.environ["VFI_NUM_SMS"] = os.environ["VFI_NUM_SMS_RANK0"]
    nf = a.frames
    clip = O.synthetic_clip(nf, H, W, seed=1234 + rank)            # this rank's shard (own content, same shape)
    eng = Rife46Engine(sd, device=local_rank, dtype=a.dtype, batch=a.batch, arch=a.arch)
    f0 = list(range(nf - 1))
    f1 = list(range(1, nf))
    ts = [0.5] * (nf - 1)
    npairs = nf - 1

    # ---- device-resident throughput ("value")
    dev_clip = clip.cuda()
    dev_out = torch.empty((npairs, H, W, 3), dtype=torch.float32, device="cuda")
    gather_list = None
    if dist is not None and rank == 0:
        gather_list = [torch.empty_like(dev_out) for _ in range(world)]
    if dist is not None:
        from cfi_b200 import shard

    def run_slice(lo, hi):
        eng.forward(dev_clip, f0[lo:hi], f1[lo:hi], ts[lo:hi], out=dev_out[lo:hi])

    # the only exchange of the path, inside the timed region for N > 1: every rank's interpolated frames end up on rank 0.
    # Default: chunked dist.gather (NCCL send / recv kernels over NVLink, 595 GB/s alone at N = 2).  VFI_GATHER=push: copy-engine
    # pushes into an IPC-shared buffer on rank 0 (shard.PushGather) - measured r02 on this pool: 35 GB/s, i.e. the IPC mapping
    # gets no peer access inside these containers and the copy is staged through the host, so it stays an option only.
    pusher = None
    if dist is not None and os.environ.get("VFI_GATHER", "nccl") == "push":
        pusher = shard.PushGather(npairs, (H, W, 3), torch.float32, dist, dst=0)
        gather_list = None

    def step_device():
        if dist is None:
            eng.forward(dev_clip, f0, f1, ts, out=dev_out)
        elif pusher is not None:
            shard.forward_and_push(run_slice, dev_out, npairs, pusher, nchunks=GATHER_CHUNKS)
        else:  # chunks of the shard are gathered to rank 0 while the next chunk computes (shard.forward_and_gather)
            shard.forward_and_gather(run_slice, dev_out, [npairs] * world, dist, dst=0, nchunks=GATHER_CHUNKS, gathered=gather_list)

    for _ in range(a.warmup):
        step_device()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        sampler.wait_first()
    barrier()
    step_device()  # one more untimed step on every rank: the GPUs are under load again when the sampled region starts
    barrier()
    l0 = eng.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_begin = time.time()
    e0.record()
    for _ in range(a.steps):
        step_device()
    e1.record()
    barrier()
    t_end = time.time()
    launches = eng.launch_count() - l0
    ms_dev = e0.elapsed_time(e1)
    clocks = sampler.stop(t_begin, t_end) if rank == 0 else None
    if a.dump_outputs and rank == 0:   # what a caller of the timed path receives: every rank's frames, in rank order
        import numpy as np
        shards = [dev_out] if dist is None else list(pusher.buffer if pusher is not None else gather_list)
        npix = min(H * W, DUMP_BYTES // (len(shards) * npairs * 3 * 4))
        os.makedirs(a.dump_outputs, exist_ok=True)
        np.save(os.path.join(a.dump_outputs, "interpolated_frames.npy"),
                torch.cat([frame_sample(s, npix) for s in shards]).numpy())
    gather_ok = None
    if dist is not None:  # what landed on rank 0 is what every rank computed (sums of each rank's first and last frame)
        mine = torch.stack([dev_out[0].double().sum(), dev_out[-1].double().sum()])
        sums = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(sums, mine)
        if rank == 0:
            got = pusher.buffer if pusher is not None else torch.stack(gather_list)
            gather_ok = all(bool(torch.equal(torch.stack([got[r][0].double().sum(), got[r][-1].double().sum()]), sums[r]))
                            for r in range(world))

    # ---- end to end through the bare C-ABI call on pre-pinned buffers ("e2e_capi", the r01 figure)
    host_in = clip.contiguous().pin_memory()
    host_out = torch.empty((npairs, H, W, 3), dtype=torch.float32).pin_memory()
    for _ in range(max(1, min(a.warmup, 2))):
        eng.interpolate_host(host_in, f0, f1, ts, host_out)
    barrier()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        eng.interpolate_host(host_in, f0, f1, ts, host_out)
    barrier()
    sec_capi = time.perf_counter() - t0
    # parity spot check inside the bench: host path == device path on this rank's data
    same = bool(torch.equal(host_out[:2], dev_out[:2].cpu()))
    del host_in, host_out

    # ---- per-kernel-group device times inside real passes (CUDA events on the launching stream, one profiled step)
    prof = None
    if rank == 0:
        eng.profile(True)
        eng.forward(dev_clip, f0, f1, ts, out=dev_out)
        prof = eng.profile_read()
        eng.profile(False)

    # ---- end to end through the plugin call ("e2e"): pageable input tensor, node-owned output tensor
    import tempfile
    from cfi_b200 import node as N
    ckpt = {"4.6": "rife46.pth", "4.7": "rife47.pth", "4.17": "rife417.pth", "4.26": "rife426.pth"}[a.arch]
    ckpt_dir = tempfile.mkdtemp(prefix="vfi_bench_ckpt_")
    os.makedirs(os.path.join(ckpt_dir, "rife"), exist_ok=True)
    torch.save(sd, os.path.join(ckpt_dir, "rife", ckpt))
    os.environ["VFI_CKPT_DIR"] = ckpt_dir
    node = N.RIFE_VFI()
    pageable = clip.contiguous()          # an ordinary CPU tensor, as ComfyUI hands an IMAGE over
    assert not pageable.is_pinned()
    res = None
    for _ in range(max(2, min(a.warmup, 3))):   # (two warm-ups: the output blocks of the caching host allocator exist)
        (res,) = node.vfi(ckpt, pageable, multiplier=2, dtype=a.dtype, batch_size=a.batch)
    barrier()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        (res,) = node.vfi(ckpt, pageable, multiplier=2, dtype=a.dtype, batch_size=a.batch)
    barrier()
    sec_e2e = time.perf_counter() - t0
    node_ok = bool(tuple(res.shape) == (2 * nf - 1, H, W, 3) and torch.equal(res[1], dev_out[0].cpu())
                   and torch.equal(res[0], clip[0]) and torch.equal(res[2], clip[1]))
    node_out_pinned = bool(res.is_pinned())
    del res
    N.clear_model_cache()

    # ---- reduce timings: max over ranks
    tt = torch.tensor([ms_dev, sec_e2e * 1e3, sec_capi * 1e3], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e, ms_capi = tt.tolist()

    if rank == 0:
        peaks = _peaks()
        total = npairs * world
        value = total * a.steps / (ms_dev / 1e3)
        e2e = total * a.steps / (ms_e2e / 1e3)
        e2e_capi = total * a.steps / (ms_capi / 1e3)

        # ---- roofline of the dominant kernel, timed alone with CUDA events (flush L2 between launches)
        tdt = torch.bfloat16 if a.dtype == "bfloat16" else torch.float16
        B = a.batch
        x = (0.1 * torch.randn(B, 272, 480, 64, device="cuda")).to(tdt)
        y = torch.empty_like(x)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
        pl = eng.layer_plan(3, 2)
        tl = []
        for i in range(13):
            flush.zero_()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            eng.debug_layer(3, 2, x, y)
            a1.record()
            torch.cuda.synchronize()
            if i >= 3:
                tl.append(a0.elapsed_time(a1))
        k_ms = sum(tl) / len(tl)
        k_flops = 2.0 * pl["macs_per_cell"] * B * 272 * 480
        achieved = k_flops / (k_ms * 1e-3) / 1e12
        roofline = {"kernel": "tapconv_kernel (block-3 ResConv 64->64, 272x480 cells, tcgen05)", "bound": "tensor",
                    "achieved": achieved, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": achieved / peaks["tflops"],
                    # dram__bytes_read.sum + dram__bytes_write.sum of this launch (batch 8) in the committed capture
                    # profiles/r02_c_resconv_b3.ncu-rep: 133.8 MB + 90.6 MB against 2 x 133.7 MB of algorithmic
                    # activation bytes (part of the output is still in L2 when the kernel ends); not re-measured here
                    "traffic": (224.4e6 if B == 8 else None), "traffic_source": "ncu profiles/r02_c_resconv_b3 (133.8 MB read + 90.6 MB written)",
                    "algorithmic_bytes": 2.0 * B * 272 * 480 * 64 * 2,
                    "peak_source": peaks["source"] + ", burst figure (kernel timed alone)",
                    "launch_ms": k_ms, "flops_per_launch": k_flops}
        # HBM-bound kernels ON the path, from the profiled step (ids: 10 * block + 0 = front, 90 = final).  Bytes per
        # padded pixel and task that the kernel has to move in this schedule (DESIGN.md section 4.2): block-3 front =
        # two half4 image gathers (16) + accumulated flow / mask read (20) and written back with the block-2 level
        # folded in (20) + that level at 1/4 of the pixels (5) + the 16-channel 16-bit block input (32); block-2 front =
        # the image gathers at full resolution (16) + the two coarse levels (1.56) + the block input at half resolution
        # (32 / 4) + the accumulated flow / mask it stores (20); final = flow / mask (20) + block-3 level (20) + two float4
        # image gathers (32) + RGB out (12, on the cropped frame).
        px = 1088 * 1920
        passes = {k: v[1] for k, v in prof.items()}
        def per_pair_ms(gid):
            return prof[gid][0] / npairs if gid in prof else None
        hbm_rows = []
        if a.arch == "4.6":
            # traffic: dram__bytes_read.sum + dram__bytes_write.sum of the same kernels in the committed capture
            # profiles/r02_i_elementwise.ncu-rep (one pass of 8 pairs: 1497 / 1382 / 645 MB), per pair
            for gid, name, bpp, traffic in (
                    (30, "front<block 3> (flow up-sample + 2 warps + resample + concat -> conv0.0 input)", 16 + 20 + 20 + 5 + 32, 1497e6 / 8),
                    (90, "final (flow up-sample + 2 warps + sigmoid blend + crop + clamp)", 20 + 20 + 32 + 12 * (H * W) / px, 1382e6 / 8),
                    (20, "front<block 2> (same at scale 2; stores the accumulated flow plane)", 16 + 1.5625 + 32 / 4 + 20, 645e6 / 8)):
                ms = per_pair_ms(gid)
                if ms:
                    gbs = bpp * px / (ms * 1e-3) / 1e9
                    hbm_rows.append({"kernel": name, "ms_per_pair": ms, "bytes_per_pair": bpp * px, "achieved": gbs,
                                     "frac": gbs / peaks["hbm_gbs"], "traffic": traffic if a.batch == 8 else None})
        roofline_hbm = {"bound": "hbm", "unit": "GB/s", "peak": peaks["hbm_gbs"], "peak_source": peaks["source"],
                        "how": "CUDA events on the launching stream around each launch inside one profiled 63-pair step "
                               "(vfi_rife_profile); bytes = what the kernel must read + write per pair in this schedule",
                        "kernels": hbm_rows,
                        "achieved": hbm_rows[0]["achieved"] if hbm_rows else None,
                        "frac": hbm_rows[0]["frac"] if hbm_rows else None,
                        "kernel": hbm_rows[0]["kernel"] if hbm_rows else None,
                        "traffic": hbm_rows[0]["traffic"] if hbm_rows else None,
                        "traffic_source": "ncu profiles/r02_i_elementwise.ncu-rep (per pair = per-launch bytes / 8)"}
        groups = {str(k): {"ms_per_pair": v[0] / npairs, "spans": v[1]} for k, v in sorted(prof.items())}
        del x, y, flush

        cpu = None
        psnr_db = None
        if world == 1 and not a.no_cpu:
            keep = {}
            fps, sec, cores, ncpu, reps = cpu_port_fps(clip, sd, 0, 1, min_seconds=10.0, keep=keep)
            # parity at the quoted configuration: the CPU leg's interpolated frames (fp32 oracle = reference CPU path)
            # against the GPU's frames for the same two pairs of the same clip
            mids = keep["out"][1::2][: CPU_SAMPLE_FRAMES - 1]
            psnr_db = float(O.psnr(dev_out[: CPU_SAMPLE_FRAMES - 1].cpu(), mids))
            cpu = {"value": fps, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": f"{CPU_SAMPLE_FRAMES - 1} pairs of the same 1080p clip, 1 warm-up + {reps} timed repetitions "
                             f"({sec * reps:.1f} s of CPU work), oracle/rife46.py == reference PyTorch-CPU path, {cores} "
                             f"threads (fastest of 8..{ncpu} on this host)"}

        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": ms_dev / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "bf16" if a.dtype == "bfloat16" else "f16",
                "dtype_note": "conv operands 16-bit, fp32 accumulate (TMEM); flow/mask/warp/blend fp32; PSNR>=50 dB "
                              "vs fp32 oracle enforced by tests/test_gpu_forward.py",
                "data": "synthetic", "config": config,
                "e2e": {"value": e2e, "unit": UNIT, "ms_per_step": ms_e2e / a.steps, "via": "RIFE_VFI.vfi (node call)",
                        "input": "pageable CPU tensor [64,1080,1920,3] fp32", "output": "node-allocated" + (" (page-locked, torch caching host allocator)" if node_out_pinned else " (pageable)"),
                        "h2d_bytes_per_step": nf * H * W * 3 * 4, "d2h_bytes_per_step": npairs * H * W * 3 * 4,
                        "node_output_matches_device_path": node_ok},
                "e2e_capi": {"value": e2e_capi, "unit": UNIT, "ms_per_step": ms_capi / a.steps,
                             "via": "vfi_rife46_interpolate_host on pre-pinned buffers", "host_equals_device_path": same},
                "psnr_db": psnr_db, "numa": numa, "gather_verified": gather_ok, "kernel_groups": groups,
                "gpu_launches": launches, "lib": cfi_lib.lib().vfi_version().decode(), "clocks": clocks,
                "model_tflops": value * FLOPS_PER_FRAME / 1e12 if a.arch == "4.6" else None,
                "roofline": roofline, "roofline_hbm": roofline_hbm, "cpu_baseline": cpu}
        print(json.dumps(line))
    eng.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

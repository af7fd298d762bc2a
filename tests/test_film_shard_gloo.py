"""FILM N>1 host logic on CPU: world_size-2 gloo run of the pair sharding + output gather against the unsharded node."""
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


class MidEngine:
    """Stand-in engine (tests only): order- and content-sensitive 'midpoint' so that a wrong pair / order shows."""
    torch_device = torch.device("cpu")

    def forward(self, frames, f0, f1, clamp=False, out=None):
        return torch.stack([0.25 * frames[a] + 0.75 * frames[b] + 0.1 * (frames[a] - frames[b]).abs() for a, b in zip(f0, f1)])


def _clip(n):
    g = torch.Generator().manual_seed(17)
    return torch.rand(n, 8, 10, 4, generator=g)


CASES = [dict(n=6, multiplier=4, states=None), dict(n=7, multiplier=[2, 5, 3], states=([2], True)),
         dict(n=5, multiplier=3, states=([0, 3], False)), dict(n=2, multiplier=2, states=None)]


def _worker(rank, world, port, q):
    # host logic only: the stand-in engines run on the CPU, so the nodes' GPU paths (Sepconv's pipelined multiplier-2
    # path) must not engage when the machine has a GPU
    os.environ["CUDA_VISIBLE_DEVICES"] = ""
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import __graft_entry__ as ge
    ge.load_package()
    from cfi_b200 import shard
    import cfi_b200.film_node as FN
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    eng = MidEngine()

    def run_node(sub, mults, st):
        s = None if st is None else FN.InterpolationStateList(list(st[0]), st[1])
        return FN.FILM_VFI().vfi("film_net_fp32.pt", sub, multiplier=list(mults), optional_interpolation_states=s,
                                 _engine=eng)[0]

    ok = True
    for c in CASES:
        fr = _clip(c["n"])
        got = shard.film_vfi_sharded(run_node, fr, c["multiplier"], c["states"], dist)
        if rank == 0:
            s = None if c["states"] is None else FN.InterpolationStateList(list(c["states"][0]), c["states"][1])
            ref = FN.FILM_VFI().vfi("film_net_fp32.pt", fr, multiplier=c["multiplier"], optional_interpolation_states=s,
                                    _engine=eng)[0]
            ok = ok and got.shape == ref.shape and torch.equal(got, ref)
    # Sepconv node (generic_frame_loop, recursive bisection) sharded the same way
    import cfi_b200.sepconv_node as SN

    class Mid:
        def middle_frame(self, a, b):
            return 0.25 * a + 0.75 * b + 0.1 * (a - b).abs()

    def run_sep(sub, m, st):
        s = None if st is None else FN.InterpolationStateList(list(st[0]), st[1])
        return SN.SepconvVFI().vfi("sepconv.pth", sub, multiplier=m, optional_interpolation_states=s, _engine=Mid())[0]

    for c in [dict(n=6, multiplier=4, states=None), dict(n=5, multiplier=3, states=([1, 2], True)),
              dict(n=4, multiplier=2, states=([0], False))]:
        fr = _clip(c["n"])
        got = shard.generic_vfi_sharded(run_sep, fr, c["multiplier"], c["states"], dist)
        if rank == 0:
            ref = run_sep(fr, c["multiplier"], c["states"])
            ok = ok and got.shape == ref.shape and torch.equal(got, ref)
    if rank == 0:
        q.put(ok)
    dist.destroy_process_group()


def test_film_sharded_equals_unsharded_world2():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    ps = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in ps:
        p.start()
    ok = q.get(timeout=120)
    for p in ps:
        p.join(timeout=60)
    assert ok


def test_shard_pairs_by_cost():
    import __graft_entry__ as ge
    ge.load_package()
    from cfi_b200.shard import shard_pairs_by_cost
    for costs, world in [([3] * 8, 4), ([3, 0, 3, 1, 1, 7, 0, 2], 3), ([1], 4), ([], 2), ([5, 1, 1, 1, 1, 1], 2)]:
        sl = shard_pairs_by_cost(costs, world)
        assert len(sl) == world and sl[0][0] == 0 and sl[-1][1] == len(costs)
        assert all(a[1] == b[0] for a, b in zip(sl, sl[1:])) and all(lo <= hi for lo, hi in sl)
    assert shard_pairs_by_cost([3] * 8, 4) == [(0, 2), (2, 4), (4, 6), (6, 8)]
    assert shard_pairs_by_cost([5, 1, 1, 1, 1, 1], 2) == [(0, 1), (1, 6)]

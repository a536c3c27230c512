"""N>1 gradient path on CPU: unite_b200.ddp.GradSync over gloo, world_size 2 (the NCCL path runs the same code on CUDA
tensors).  Checks (a) the overlapped range-by-range all-reduce + final flush equals one flat all-reduce, (b) the returned
scale turns the SUM into DDP's MEAN (run_stage1.py:809), (c) ranges may be announced in any increasing order."""
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


def _cpu_rank_env(rank, world, port):
    # the ranks stay on the CPU even on a GPU box: with CUDA visible, init_distributed_from_env binds cuda:LOCAL_RANK, and a box
    # with one GPU has no cuda:1
    os.environ.update(CUDA_VISIBLE_DEVICES="", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))


def _worker(rank, world, port, q):
    _cpu_rank_env(rank, world, port)
    from unite_b200.ddp import GradSync, init_distributed_from_env
    r, _, w = init_distributed_from_env(backend="gloo")
    assert (r, w) == (rank, world)
    g = torch.Generator().manual_seed(100 + rank)
    n = 10_000
    flat = torch.randn(n, generator=g)
    mine = flat.clone()
    gs = GradSync()
    # backward announces growing prefixes of the decay segment as blocks finish; the tail is flushed by all_reduce()
    for hi in (1000, 1000, 4096, 7000):
        gs.range_ready(flat, hi)
    scale = gs.all_reduce(flat)
    assert abs(scale - 1.0 / world) < 1e-12
    others = [torch.randn(n, generator=torch.Generator().manual_seed(100 + k)) for k in range(world)]
    expect = sum(others)
    ok = torch.allclose(flat, expect, atol=1e-6) and gs.calls == 4 and not torch.equal(flat, mine)
    # second step re-uses the object: state must have been reset
    flat2 = torch.full((n,), float(rank + 1))
    gs.range_ready(flat2, 5000)
    gs.all_reduce(flat2)
    ok = ok and torch.allclose(flat2, torch.full((n,), float(sum(range(1, world + 1)))))
    q.put((rank, bool(ok)))
    dist.barrier()
    dist.destroy_process_group()


def test_gradsync_world2_gloo():
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert sorted(res) == [(0, True), (1, True)]


def test_gradsync_single_process_is_identity():
    from unite_b200.ddp import GradSync
    gs = GradSync()
    x = torch.arange(10.0)
    gs.range_ready(x, 4)
    assert gs.all_reduce(x) == 1.0 and torch.equal(x, torch.arange(10.0)) and gs.calls == 0


def test_nvls_shards_tile_the_decay_segment():
    """ddp.NvlsShardedStep.shard_of mirrors the kernel's slice arithmetic: disjoint, ordered, covering, 8-element aligned."""
    from unite_b200.ddp import NvlsShardedStep
    for n_decay in (0, 8, 64, 87_949_272, 8 * 1001):
        for world in (1, 2, 3, 4, 8):
            edges = [NvlsShardedStep.shard_of(n_decay, r, world) for r in range(world)]
            assert edges[0][0] == 0 and edges[-1][1] == n_decay
            for (lo, hi), (lo2, _) in zip(edges, edges[1:] + [(n_decay, n_decay)]):
                assert lo <= hi == lo2 and lo % 8 == 0 and hi % 8 == 0


def _consolidate_worker(rank, world, port, q):
    import types
    _cpu_rank_env(rank, world, port)
    from unite_b200.ddp import NvlsShardedStep, init_distributed_from_env
    init_distributed_from_env(backend="gloo")
    n, n_decay = 4096, 4096 - 72
    full = [torch.arange(n, dtype=torch.float32) * (k + 1) for k in range(3)]          # what a replicated optimizer would hold
    lo, hi = NvlsShardedStep.shard_of(n_decay, rank, world)
    mine = []
    for t in full:                                                                      # sharded: only my slice + no-decay tail are live
        x = torch.full((n,), -1.0)
        x[lo:hi] = t[lo:hi]
        x[n_decay:] = t[n_decay:]
        mine.append(x)
    step = object.__new__(NvlsShardedStep)                                              # host-side gather only; no symmetric memory on CPU
    step.arena = types.SimpleNamespace(params=mine[0], n_decay=n_decay)
    step.opt = types.SimpleNamespace(exp_avg=mine[1], exp_avg_sq=mine[2])
    step.pg, step.rank, step.world = dist.group.WORLD, rank, world
    step.check = lambda: None
    step.consolidate()
    q.put((rank, all(torch.equal(a, b) for a, b in zip(mine, full))))
    dist.barrier()
    dist.destroy_process_group()


def test_nvls_consolidate_gathers_sharded_state_world2_gloo():
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_consolidate_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert sorted(res) == [(0, True), (1, True)]

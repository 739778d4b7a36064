"""Multi-process logic of the data-parallel path on the CPU: world_size 2, gloo backend.
Covers what `bench.py --gpus N` relies on: ray sharding, the flat gradient arena and its single all-reduce."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from neuradar_b200.dist import GradArena, shard_bounds


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank: int, world: int, port: int, out_dir: str) -> None:
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.manual_seed(0)  # replicated parameters
        net = torch.nn.Sequential(torch.nn.Linear(6, 5), torch.nn.ReLU(), torch.nn.Linear(5, 3))
        frozen = torch.nn.Linear(2, 2)  # a parameter that never receives a gradient (cf. proposal_fields[0])
        params = list(net.parameters()) + list(frozen.parameters())
        arena = GradArena(params)
        assert arena.flat.numel() % 4 == 0 and all(p.grad.data_ptr() >= arena.flat.data_ptr() for p in params)
        # the global batch, identical on every rank; each rank takes its contiguous slice of whole 4-ray granules
        g = torch.Generator().manual_seed(1)
        x = torch.randn((32, 6), generator=g)
        lo, hi = shard_bounds(32, world, rank, granule=4)
        arena.zero()
        net(x[lo:hi]).pow(2).mean().backward()  # per-rank mean over its own rays, as DDP does
        arena.all_reduce(average=True)
        torch.save({"flat": arena.flat.clone(), "bounds": (lo, hi)}, os.path.join(out_dir, f"rank{rank}.pt"))
    finally:
        dist.destroy_process_group()


def test_arena_allreduce_matches_full_batch(tmp_path):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    r0 = torch.load(tmp_path / "rank0.pt")
    r1 = torch.load(tmp_path / "rank1.pt")
    assert r0["bounds"] == (0, 16) and r1["bounds"] == (16, 32)
    assert torch.equal(r0["flat"], r1["flat"]), "every rank must hold the same averaged gradient"
    # equal shards: the average of per-rank means is the full-batch mean
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Linear(6, 5), torch.nn.ReLU(), torch.nn.Linear(5, 3))
    frozen = torch.nn.Linear(2, 2)
    g = torch.Generator().manual_seed(1)
    x = torch.randn((32, 6), generator=g)
    net(x).pow(2).mean().backward()
    want = torch.cat([p.grad.flatten() for p in net.parameters()])
    got = r0["flat"]
    # arena views are padded to multiples of 4 floats; compare view by view
    off = 0
    for p in list(net.parameters()) + list(frozen.parameters()):
        n = p.numel()
        ref = p.grad.flatten() if p.grad is not None else torch.zeros(n)
        torch.testing.assert_close(got[off : off + n], ref, rtol=1e-6, atol=1e-7)
        off += (n + 3) // 4 * 4
    assert want.numel() > 0


def test_arena_single_process_is_a_noop():
    p = torch.nn.Parameter(torch.ones(5))
    arena = GradArena([p])
    p.sum().backward()
    arena.all_reduce()  # no process group: must not raise
    assert torch.equal(p.grad, torch.ones(5))
    arena.zero()
    assert float(p.grad.abs().sum()) == 0.0
    with pytest.raises(ValueError):
        GradArena([])


def test_arena_relinks_after_zero_grad_set_to_none():
    """`optimizer.zero_grad()` / `module.zero_grad()` default to set_to_none=True and detach the gradients from the arena;
    `all_reduce()` / `zero()` must bring them back (ADVICE round 1)."""
    torch.manual_seed(0)
    net = torch.nn.Linear(4, 3)
    arena = GradArena(list(net.parameters()))
    net.zero_grad(set_to_none=True)
    assert all(p.grad is None for p in net.parameters())
    net(torch.ones(2, 4)).sum().backward()  # autograd allocates fresh gradient tensors
    want = [p.grad.clone() for p in net.parameters()]
    assert all(p.grad.data_ptr() != v.data_ptr() for p, v in zip(arena.params, arena._views))
    arena.all_reduce()  # single process: only the re-link happens
    for p, v, w in zip(arena.params, arena._views, want):
        assert p.grad.data_ptr() == v.data_ptr()
        assert torch.equal(p.grad, w)
    off = 0
    for w in want:
        assert torch.equal(arena.flat[off : off + w.numel()], w.flatten())
        off += (w.numel() + 3) // 4 * 4
    net.zero_grad(set_to_none=True)
    arena.zero()
    assert all(p.grad is not None and float(p.grad.abs().sum()) == 0.0 for p in net.parameters())
    assert arena.relink() == 0


def _early_worker(rank: int, world: int, port: int, out_dir: str) -> None:
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        table = torch.nn.Parameter(torch.zeros(37, 2))   # stands for the main hash table: gradient final early
        other = torch.nn.Parameter(torch.zeros(5))
        last = torch.nn.Parameter(torch.zeros(3, 3))
        arena = GradArena([other, table, last], direct_scatter=True, early=[table])
        assert arena.params[0] is table, "early parameters lead the flat buffer"
        assert arena.reducer.n_early == 76  # 74 floats padded to a multiple of 4
        for step in range(2):  # the second step checks that the reducer re-arms
            arena.zero()
            # what a backward kernel with a direct sink does: add into the sink, then signal (functional._sink_written)
            table._nrb_grad_sink.add_(float(rank + 1 + step))
            table._nrb_grad_ready()
            assert arena.reducer._work is not None, "the early all-reduce must be in flight"
            other._nrb_grad_sink.add_(10.0 * (rank + 1))
            last.grad.add_(100.0 * (rank + 1))
            arena.all_reduce(average=True)
            assert arena.reducer._work is None
        torch.save({"flat": arena.flat.clone()}, os.path.join(out_dir, f"early{rank}.pt"))
    finally:
        dist.destroy_process_group()


def test_early_overlapped_reduce_matches_single_collective(tmp_path):
    world = 2
    mp.spawn(_early_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    f0 = torch.load(tmp_path / "early0.pt")["flat"]
    f1 = torch.load(tmp_path / "early1.pt")["flat"]
    assert torch.equal(f0, f1)
    assert torch.allclose(f0[:74], torch.full((74,), (2.0 + 3.0) / 2))       # step 1: ranks added 2 and 3
    assert float(f0[74:76].abs().sum()) == 0.0                                # padding stays zero
    assert torch.allclose(f0[76:81], torch.full((5,), 15.0))
    assert torch.allclose(f0[84:93], torch.full((9,), 150.0))


def _misuse_worker(rank: int, world: int, port: int, out_dir: str) -> None:
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from neuradar_b200._lib import NeuradarB200Error

        table = torch.nn.Parameter(torch.zeros(8))
        other = torch.nn.Parameter(torch.zeros(4))
        arena = GradArena([other, table], direct_scatter=True, early=[table])
        arena.zero()
        # two backward passes per reduce (gradient accumulation, or two losses with retain_graph): the second write to
        # the early region lands after its collective was launched and would never be exchanged
        table._nrb_grad_sink.add_(float(rank + 1))
        table._nrb_grad_ready()
        table._nrb_grad_sink.add_(float(rank + 1))
        with pytest.raises(NeuradarB200Error, match="gradient accumulation"):
            table._nrb_grad_ready()
        arena.all_reduce(average=True)  # joins the first collective; the reducer is idle again
        assert arena.reducer._work is None
        subgroup = dist.new_group([0, 1])  # the same ranks, but not the default group
        with pytest.raises(ValueError):
            arena.all_reduce(group=subgroup)
    finally:
        dist.destroy_process_group()


def test_second_early_write_per_reduce_raises(tmp_path):
    world = 2
    mp.spawn(_misuse_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)


def test_single_process_early_writes_accumulate():
    """Without data parallelism the early callback does nothing, so gradient accumulation keeps working."""
    table = torch.nn.Parameter(torch.zeros(6))
    arena = GradArena([table], direct_scatter=True, early=[table])
    for k in (1.0, 2.0):
        table._nrb_grad_sink.add_(k)
        table._nrb_grad_ready()
    arena.all_reduce()
    assert torch.equal(table.grad, torch.full((6,), 3.0))


def test_arena_keeps_an_existing_grad():
    p = torch.nn.Parameter(torch.zeros(5))
    p.grad = torch.arange(5.0)
    arena = GradArena([p])
    assert p.grad.data_ptr() == arena.flat.data_ptr()
    assert torch.equal(p.grad, torch.arange(5.0))

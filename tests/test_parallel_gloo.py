"""world_size-2 gloo (CPU) checks of the multi-GPU host logic (SURVEY §8e): shard ranges, the padded all-gather that
restores global net order for uneven shards, and the identity behind arg-min routing (the partial dL/da of the ranks
sum to the single-process gradient).  No CUDA involved: the exchanged tensors are plain torch tensors."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from super_sac_b200 import parallel


def test_local_range_partitions():
    for n, world in [(10, 8), (10, 4), (10, 2), (5, 2), (2, 2), (7, 3)]:
        ranges = [parallel.local_range(n, world, r) for r in range(world)]
        assert ranges[0][0] == 0 and ranges[-1][1] == n
        assert all(ranges[r][1] == ranges[r + 1][0] for r in range(world - 1))
        sizes = [hi - lo for lo, hi in ranges]
        assert max(sizes) - min(sizes) <= 1 and sorted(sizes, reverse=True) == sizes
    assert [parallel.local_range(10, 8, r) for r in range(3)] == [(0, 2), (2, 4), (4, 5)]


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, n_global, out_q):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        lo, hi = parallel.enable_critic_sharding(n_global)
        B, A = 6, 3
        gen = torch.Generator().manual_seed(0)                     # replicated "Philox": same numbers on every rank
        q_full = torch.randn(n_global, B, 1, generator=gen)
        dx_full = torch.randn(n_global, B, A, generator=gen)       # per-net dQ/da if that net were the arg-min
        q_all = parallel.all_gather_q(q_full[lo:hi].clone())
        assert torch.equal(q_all, q_full), "all_gather_q must restore global net order"
        arg = q_all.squeeze(-1).argmin(0)                          # [B] identical on every rank
        onehot = torch.zeros(n_global, B)
        onehot[arg, torch.arange(B)] = 1.0
        da_local = (onehot[lo:hi, :, None] * dx_full[lo:hi]).sum(0)  # only rows whose arg-min critic is local
        da = parallel.all_reduce_sum_(da_local.clone())
        want = dx_full[arg, torch.arange(B)]
        assert torch.allclose(da, want), "sum of routed partial gradients == single-process gradient"
        loss = parallel.all_reduce_sum_(torch.tensor([float(hi - lo)]))
        assert float(loss) == n_global
        # global-norm clipping under sharding (learning.py critic_clip): sum ||g||^2 over every rank's critics
        g_full = torch.randn(n_global, 7, generator=gen)
        gsq = parallel.all_reduce_sum_((g_full[lo:hi] ** 2).sum().reshape(1), site="critic_gnorm")
        assert torch.allclose(gsq, (g_full ** 2).sum().reshape(1))
        # DR3 under sharding: every rank adds its share N_local / N_global of the mean over the GLOBAL ensemble
        dots = torch.randn(n_global, B, generator=gen)
        share = dots[lo:hi].mean().reshape(1) * ((hi - lo) / n_global)
        assert torch.allclose(parallel.all_reduce_sum_(share, site="dr3_dot"), dots.mean().reshape(1), atol=1e-6)
        out_q.put((rank, lo, hi))
    finally:
        parallel.disable()
        dist.destroy_process_group()


def test_sharded_exchange_world2_gloo():
    world, n_global = 2, 5
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, n_global, q)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    got = sorted(q.get(timeout=5) for _ in range(world))
    assert got == [(0, 0, 3), (1, 3, 5)]


def _member_worker(rank, world, port, e_global, out_q):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        lo, hi = parallel.enable_member_sharding(e_global)
        N, B, D = 2, 4, 3
        assert parallel.members_sharded() and parallel.members_global(hi - lo) == e_global and parallel.my_members() == (lo, hi)
        gen = torch.Generator().manual_seed(0)
        x_full = torch.randn(e_global, B, D, generator=gen)               # one batch per member
        x_all = parallel.all_gather_members(x_full[lo:hi].clone())
        assert torch.equal(x_all, x_full), "batches come back in global member order"
        # every rank's target critics (N per member) on every batch: q[net, batch, b]
        q_full = torch.randn(e_global * N, e_global, B, generator=gen)
        q_all = parallel.all_gather_members(q_full[lo * N:hi * N].clone())
        assert torch.equal(q_all, q_full), "values come back in global (member, net) order"
        tot = parallel.all_reduce_members_(torch.tensor([float(hi - lo)]))
        assert float(tot) == e_global
        out_q.put((rank, lo, hi))
    finally:
        parallel.disable()
        dist.destroy_process_group()


def test_member_sharding_exchange_world2_gloo():
    """SUNRISE members over ranks (SURVEY 8e, C3): uneven member blocks, both all-gathers restore the global order."""
    world, e_global = 2, 5
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_member_worker, args=(r, world, port, e_global, q)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    got = sorted(q.get(timeout=5) for _ in range(world))
    assert got == [(0, 0, 3), (1, 3, 5)]
    assert not parallel.members_sharded()


def test_one_partition_at_a_time(monkeypatch):
    """An ensemble is sharded one way at a time: enabling the other kind raises and leaves the first in place.  With
    sharding off the global sizes and member ids are the local ones."""
    monkeypatch.setenv("MASTER_ADDR", "127.0.0.1")
    monkeypatch.setenv("MASTER_PORT", str(_free_port()))
    dist.init_process_group("gloo", rank=0, world_size=1)
    try:
        assert not parallel.sharded()
        assert parallel.n_global(3) == 3 and parallel.members_global(4) == 4
        assert [parallel.member_id(i) for i in range(3)] == [0, 1, 2]
        for first, other, on in ((parallel.enable_critic_sharding, parallel.enable_member_sharding, parallel.critics_sharded),
                                 (parallel.enable_member_sharding, parallel.enable_critic_sharding, parallel.members_sharded)):
            first(5)
            with pytest.raises(NotImplementedError, match="cannot be combined"):
                other(5)
            assert on() and parallel.my_range() == (0, 5)
            parallel.disable()
        parallel.enable_critic_sharding(5)
        assert parallel.n_global(2) == 5 and parallel.members_global(2) == 2 and parallel.member_id(1) == 1
        parallel.disable()
        assert parallel.n_global(3) == 3 and not parallel.sharded()
    finally:
        parallel.disable()
        dist.destroy_process_group()

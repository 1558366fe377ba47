"""Batch sharding (parallel.enable_batch_sharding) on CPU: a world-2 gloo group.  The row partition (B not divisible by
the world as well), the augmented-row counts of aug_mix in global row numbers, mutual exclusion with critic and member
sharding, every refusal of the update entry points -- raised before anything is launched (the library is replaced by an
object that fails on any use) -- and the fallback all-reduce of a flat gradient (torch.distributed), which must leave
the same values on both ranks."""
import os
import socket
import traceback
import types

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

WORLD = 2


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


class _NoLaunch:
    def __getattr__(self, name):
        raise AssertionError(f"libssac_b200.{name} used before the refusal")


def _fake_agent(**kw):
    enc = torch.nn.Identity()
    a = dict(ensemble_size=1, num_critics=2, popart=[False], encoder=enc, deterministic=False, discrete=False)
    a.update(kw)
    return types.SimpleNamespace(**a)


def _critic_kw(agent, **kw):
    d = dict(buffer=None, agent=agent, target_agent=agent, critic_optimizer=None, encoder_optimizer=None, log_alphas=[None],
             batch_size=8, gamma=0.99, critic_clip=None, encoder_clip=None, target_critic_ensemble_n=2,
             weighted_bellman_temp=None, weight_type=None, pop=False, augmenter=None, encoder_lambda=0.0, random_process=None,
             noise_clip=None, aug_mix=0.0, discrete=False, per=False, update_priorities=False, dr3_coeff=0.0)
    d.update(kw)
    return d


def _case(rank):
    from super_sac_b200 import _lib, augmentations, learning, learning_utils as lu, parallel

    # row partition and augmented rows
    parallel.enable_batch_sharding()
    assert parallel.batches_sharded() and parallel.world_size() == WORLD
    for B in (2, 7, 10, 256, 513):
        ranges = [parallel.local_range(B, WORLD, r) for r in range(WORLD)]
        assert parallel.batch_range(B) == ranges[rank]
        assert ranges[0][0] == 0 and ranges[-1][1] == B and all(ranges[r][1] == ranges[r + 1][0] for r in range(WORLD - 1))
        sizes = [hi - lo for lo, hi in ranges]
        assert max(sizes) - min(sizes) <= 1
        for mix in (0.0, 0.3, 0.5, 0.75, 1.0):
            rows = [parallel.local_aug_rows(B, mix, lo, hi) for lo, hi in ranges]
            assert sum(rows) == int(B * mix), (B, mix, rows)
            for (lo, hi), n in zip(ranges, rows):   # the augmented rows are the batch's first int(B * mix) rows
                assert n == len([g for g in range(lo, hi) if g < int(B * mix)])
    assert parallel.batch_range(7) == ((0, 4) if rank == 0 else (4, 7))
    with pytest.raises(ValueError):
        parallel.batch_range(1)

    # mutual exclusion, both ways
    with pytest.raises(NotImplementedError):
        parallel.enable_critic_sharding(4)
    with pytest.raises(NotImplementedError):
        parallel.enable_member_sharding(4)
    parallel.disable()
    parallel.enable_critic_sharding(4)
    with pytest.raises(NotImplementedError):
        parallel.enable_batch_sharding()
    parallel.disable()
    parallel.enable_member_sharding(2)
    with pytest.raises(NotImplementedError):
        parallel.enable_batch_sharding()
    parallel.disable()
    assert parallel.batch_range(7) == (0, 7)   # nothing sharded: the whole batch

    # refusals before any launch
    parallel.enable_batch_sharding()
    real = _lib._lib
    _lib._lib = _NoLaunch()
    try:
        refused = [
            _critic_kw(_fake_agent(), per=True),
            _critic_kw(_fake_agent(), per=False, update_priorities=True),
            _critic_kw(_fake_agent(), weight_type="sunrise", weighted_bellman_temp=20.0),
            _critic_kw(_fake_agent(), dr3_coeff=0.01),
            _critic_kw(_fake_agent(), discrete=True),
            _critic_kw(_fake_agent(ensemble_size=2, popart=[False, False])),
            _critic_kw(_fake_agent(popart=[types.SimpleNamespace()])),   # a PopArt layer (truthy)
            _critic_kw(_fake_agent(encoder=torch.nn.Linear(8, 8))),      # a trainable encoder that is not the native one
        ]
        for kw in refused:
            with pytest.raises(NotImplementedError, match="batch sharding"):
                learning.critic_update(**kw)
        with pytest.raises(NotImplementedError, match="batch sharding"):
            learning.offline_actor_update(buffer=None, agent=_fake_agent(), actor_optimizer=None, encoder_optimizer=None,
                                          batch_size=8, actor_clip=None, update_encoder=False, encoder_clip=None,
                                          augmenter=None, actor_lambda=0.0, aug_mix=0.0)
        with pytest.raises(NotImplementedError, match="batch sharding"):
            learning.online_actor_update(buffer=None, agent=_fake_agent(ensemble_size=2), pop=False, actor_optimizer=None,
                                         log_alphas=[None, None], batch_size=8, clip=None, random_process=None,
                                         noise_clip=None, augmenter=None, aug_mix=0.0)
        with pytest.raises(NotImplementedError, match="batch sharding"):
            learning.online_actor_update(buffer=None, agent=_fake_agent(), pop=False, actor_optimizer=None,
                                         log_alphas=[None], batch_size=8, clip=None, random_process=None, noise_clip=None,
                                         augmenter=None, aug_mix=0.0, discrete=True)
        with pytest.raises(NotImplementedError, match="batch sharding"):
            learning.alpha_update(buffer=None, agent=_fake_agent(ensemble_size=2), optimizers=None, batch_size=8,
                                  log_alphas=None, augmenter=None, aug_mix=0.0, target_entropy=-1.0,
                                  premade_replay_dicts=None, discrete=False)
        with pytest.raises(NotImplementedError, match="batch sharding"):
            learning.alpha_update(buffer=None, agent=_fake_agent(), optimizers=None, batch_size=8, log_alphas=None,
                                  augmenter=None, aug_mix=0.0, target_entropy=-1.0, premade_replay_dicts=None,
                                  discrete=True)
        # updates that sample their own batch: the sampling is refused before the N(0,1) draws are launched
        identity = augmentations.AugmentationSequence([augmentations.IdentityAug(8)])
        with pytest.raises(NotImplementedError, match="batch sharding"):
            learning.online_actor_update(buffer=None, agent=_fake_agent(), pop=False, actor_optimizer=None,
                                         log_alphas=[None], batch_size=8, clip=None, random_process=None, noise_clip=None,
                                         augmenter=identity, aug_mix=0.0, per=True)
        for aug in (lambda o, o1: (o, o1), augmentations.AugmentationSequence([augmentations.DrqAug(8, noise=True)])):
            with pytest.raises(NotImplementedError, match="batch sharding"):
                learning.online_actor_update(buffer=None, agent=_fake_agent(), pop=False, actor_optimizer=None,
                                             log_alphas=[None], batch_size=8, clip=None, random_process=None,
                                             noise_clip=None, augmenter=aug, aug_mix=0.0)
            with pytest.raises(NotImplementedError, match="batch sharding"):
                learning.alpha_update(buffer=None, agent=_fake_agent(), optimizers=None, batch_size=8, log_alphas=None,
                                      augmenter=aug, aug_mix=0.0, target_entropy=-1.0, premade_replay_dicts=None,
                                      discrete=False)
            with pytest.raises(NotImplementedError, match="batch sharding"):
                learning.critic_update(**_critic_kw(_fake_agent(), augmenter=aug))
        # the sampler: prioritised draws, user augmenters and noisy DrQ cannot be split row for row
        with pytest.raises(NotImplementedError, match="batch sharding"):
            lu._batch_rows(8, augmentations.AugmentationSequence([augmentations.IdentityAug(8)]), per=True)
        with pytest.raises(NotImplementedError, match="batch sharding"):
            lu._batch_rows(8, lambda o, o1: (o, o1), per=False)
        with pytest.raises(NotImplementedError, match="batch sharding"):
            lu._batch_rows(8, augmentations.AugmentationSequence([augmentations.DrqAug(8, noise=True)]), per=False)
        with pytest.raises(ValueError, match="batch sharding"):   # shifts drawn for another batch size
            lu._batch_rows(8, augmentations.AugmentationSequence([augmentations.Drqv2Aug(16)]), per=False)
        assert lu._batch_rows(8, augmentations.AugmentationSequence([augmentations.Drqv2Aug(8)]), per=False) == \
            parallel.batch_range(8)
    finally:
        _lib._lib = real

    # fallback all-reduce: gloo, CPU tensors
    for n in (1, 3, 4097):
        g = torch.Generator().manual_seed(n)
        xs = [torch.randn(n, generator=g) for _ in range(WORLD)]
        t = xs[rank].clone()
        parallel.all_reduce_flat_(t, site="test")
        parts = [torch.empty_like(t) for _ in range(WORLD)]
        dist.all_gather(parts, t)
        assert all(torch.equal(p, parts[0]) for p in parts)
        assert torch.allclose(t, xs[0] + xs[1], rtol=1e-6, atol=1e-6)
    with pytest.raises(ValueError):
        parallel.all_reduce_flat_(torch.zeros(4, dtype=torch.float64), site="test")
    parallel.disable()


def _worker(rank, port, errq):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    try:
        dist.init_process_group("gloo", rank=rank, world_size=WORLD)
        try:
            _case(rank)
        finally:
            dist.destroy_process_group()
        errq.put((rank, None))
    except BaseException:  # noqa: BLE001
        errq.put((rank, traceback.format_exc()))


def test_batch_sharding_host_logic_gloo_world2():
    ctx = mp.get_context("spawn")
    errq = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, port, errq)) for r in range(WORLD)]
    for p in procs:
        p.start()
    results = [errq.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    errors = [f"rank {r}:\n{e}" for r, e in results if e is not None]
    assert not errors, "\n".join(errors)


@pytest.mark.parametrize("B,world", [(10, 2), (7, 2), (61, 4), (513, 8), (4, 4), (5, 4)])
def test_pooled_td_statistics_match_the_whole_batch(B, world):
    """The logged TD-target statistics of a batch-sharded update: every rank's mean / unbiased std / entropy bonus over
    its rows, pooled, equal the whole batch's (float64 reference), for uneven splits and parts of a single row."""
    import numpy as np

    from super_sac_b200 import learning_utils as lu, parallel

    rng = np.random.default_rng(B * 10 + world)
    y = rng.standard_normal(B) * 3.0 + 10.0
    e = rng.standard_normal(B)
    parts = [parallel.local_range(B, world, r) for r in range(world)]
    n = [hi - lo for lo, hi in parts]
    means = [float(y[lo:hi].mean()) for lo, hi in parts]
    stds = [float(y[lo:hi].std(ddof=1)) if hi - lo > 1 else float("nan") for lo, hi in parts]   # 0/0 for one row
    ents = [float(e[lo:hi].mean()) for lo, hi in parts]
    m, s, ent = lu.pooled_stats(n, means, stds, ents)
    assert m == pytest.approx(y.mean(), rel=1e-12)
    assert s == pytest.approx(y.std(ddof=1), rel=1e-10)
    assert ent == pytest.approx(e.mean(), rel=1e-10, abs=1e-12)

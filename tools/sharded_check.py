#!/usr/bin/env python
"""The ensemble-sharded update must equal the single-GPU update (one rank per GPU).  Used by bench.py --gpus N > 1
before any timing ("sharded_parity" in its JSON line) and, as a torchrun script, by tests/:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 \
        tools/sharded_check.py

Every rank (a) runs the full N-critic agent on its own GPU and (b) runs its shard of the same agent with the NCCL
exchange of super_sac_b200.parallel, on the same scripted draws, and compares post-update critics (its shard), actors,
log_alpha-independent TD targets and the logged loss at rtol 1e-4.  The torchrun script also runs ``logged_checks``:
every logged value on every rank, DR3 with the members sharded and the offline actor update with the members sharded
and a clip that engages.
"""
import copy
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "tools")):
    if _p not in sys.path:
        sys.path.insert(0, _p)
import math
from itertools import chain

import numpy as np
import torch
import torch.distributed as dist

import benchlib as bl
import super_sac_b200 as ssb
from super_sac_b200 import _arena, _rng, augmentations, learning, learning_utils as lu, nets, parallel

IdentityEncoder, _ = bl._encoders(ssb)


def optimizers(agent, cfg):
    critic_opt = torch.optim.Adam(chain(*(c.parameters() for c in agent.critics)), lr=cfg.get("critic_lr", 3e-4), betas=(0.9, 0.999))
    actor_opt = torch.optim.Adam(chain(*(a.parameters() for a in agent.actors)), lr=cfg.get("actor_lr", 3e-4), betas=(0.9, 0.999))
    enc_opt = torch.optim.Adam(agent.encoder.parameters(), lr=1e-4, betas=(0.9, 0.999))
    dev = agent._critic_arena.device
    log_alphas = []
    for _ in range(cfg["E"]):
        la = torch.Tensor([math.log(0.1)]).to(dev)
        la.requires_grad = True
        log_alphas.append(la)
    return critic_opt, actor_opt, enc_opt, log_alphas, None


def assert_close(a, b, rtol, atol, what=""):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    err, tol = np.abs(a - b), atol + rtol * np.abs(b)
    if not np.all(err <= tol):
        i = np.unravel_index(np.argmax(err - tol), err.shape)
        raise AssertionError(f"{what}: max violation at {i}: got {a[i]!r} want {b[i]!r} (|err|={err[i]:.3e}, tol={tol[i]:.3e})")


def build(N, S, A, H, device, seed):
    torch.manual_seed(seed)
    agent = ssb.Agent(act_space_size=A, encoder=IdentityEncoder(S), actor_network_cls=nets.mlps.ContinuousStochasticActor,
                      critic_network_cls=nets.mlps.ContinuousCritic, ensemble_size=1, num_critics=N, hidden_size=H,
                      auto_rescale_targets=False, log_std_low=-5.0, log_std_high=2.0)
    agent.to(device)
    return agent


def _keep_logged(logged, prefix, logs):
    """Collect into ``logged`` the logged values a sharded update reproduces (the gradient norms are each rank's own)."""
    if logged is not None:
        logged.update({prefix + k: v for k, v in logs.items() if not k.startswith("gradients/")})


def run(agent, target, buf, draws, B, M, cfg, pipelined=False, critic_clip=None, dr3_coeff=0.0, logged=None):
    """The scripted update sequence: len(draws) critic updates (+ Polyak) -- inside one lu.pipelined_updates() block when
    ``pipelined`` -- then one actor update on the last batch.  Returns the logged losses (all logged values: ``logged``)."""
    import contextlib

    critic_opt, actor_opt, enc_opt, log_alphas, _ = optimizers(agent, cfg)
    aug = augmentations.AugmentationSequence([augmentations.IdentityAug(B)])
    out = {}
    old = _rng.set_source(_rng.ScriptedSource())

    def critic_steps():
        rds = None
        for step, dr in enumerate(draws):
            src = _rng.ScriptedSource()
            _rng.set_source(src)
            src.push("indices", dr["idx"]).push("normal", dr["eps"]).push("subsets", dr["subset"])
            logs, rds = learning.critic_update(
                buffer=buf, agent=agent, target_agent=target, critic_optimizer=critic_opt, encoder_optimizer=enc_opt,
                log_alphas=log_alphas, batch_size=B, gamma=0.99, critic_clip=critic_clip, encoder_clip=None,
                target_critic_ensemble_n=M, weighted_bellman_temp=None, weight_type=None, pop=False, augmenter=aug,
                encoder_lambda=0.0, random_process=None, noise_clip=None, aug_mix=0.0, dr3_coeff=dr3_coeff)
            for ac, tc in zip(agent.critics, target.critics):
                lu.soft_update(tc, ac, 0.005)
            out[f"loss{step}"] = logs["losses/critic_overall_loss"]
            _keep_logged(logged, f"critic{step}/", logs)
            if dr3_coeff > 0:
                out[f"dr3_{step}"] = logs["dr3_dotproduct_0"]
        return rds

    try:
        with (lu.pipelined_updates() if pipelined else contextlib.nullcontext()):
            rds = critic_steps()
        src = _rng.ScriptedSource()
        _rng.set_source(src)
        src.push("normal", draws[-1]["eps2"])
        alogs = learning.online_actor_update(
            buffer=buf, agent=agent, pop=False, actor_optimizer=actor_opt, log_alphas=log_alphas, batch_size=B, clip=None,
            random_process=None, noise_clip=None, augmenter=aug, aug_mix=0.0, premade_replay_dicts=rds)
        out["actor_loss"] = alogs["losses/actor_pg_loss"]
        _keep_logged(logged, "actor/", alogs)
    finally:
        _rng.set_source(old)
    return out


def build_ensemble(E, N, S, A, H, device, seed):
    torch.manual_seed(seed)
    agent = ssb.Agent(act_space_size=A, encoder=IdentityEncoder(S), actor_network_cls=nets.mlps.ContinuousStochasticActor,
                      critic_network_cls=nets.mlps.ContinuousCritic, ensemble_size=E, num_critics=N, hidden_size=H,
                      auto_rescale_targets=False, log_std_low=-5.0, log_std_high=2.0)
    agent.to(device)
    return agent


def run_sunrise(agent, target, buf, draws, members, B, N, cfg, dr3_coeff=0.0, logged=None):
    """draws[step][member] for the GLOBAL member ids in ``members`` (this agent's members, in order)."""
    critic_opt, actor_opt, enc_opt, log_alphas, _ = optimizers(agent, dict(cfg, E=len(members)))
    aug = augmentations.AugmentationSequence([augmentations.IdentityAug(B)])
    out = {}
    old = _rng.set_source(_rng.ScriptedSource())
    try:
        for step, dr in enumerate(draws):
            src = _rng.ScriptedSource()
            _rng.set_source(src)
            for m in members:
                src.push("indices", dr[m]["idx"]).push("normal", dr[m]["eps"]).push("subsets", dr[m]["subset"])
            logs, rds = learning.critic_update(
                buffer=buf, agent=agent, target_agent=target, critic_optimizer=critic_opt, encoder_optimizer=enc_opt,
                log_alphas=log_alphas, batch_size=B, gamma=0.99, critic_clip=None, encoder_clip=None,
                target_critic_ensemble_n=N, weighted_bellman_temp=20.0, weight_type="sunrise", pop=False, augmenter=aug,
                encoder_lambda=0.0, random_process=None, noise_clip=None, aug_mix=0.0, dr3_coeff=dr3_coeff)
            for ac, tc in zip(agent.critics, target.critics):
                lu.soft_update(tc, ac, 0.005)
            out[f"loss{step}"] = logs["losses/critic_overall_loss"]
            _keep_logged(logged, f"critic{step}/", logs)
        src = _rng.ScriptedSource()
        _rng.set_source(src)
        for m in members:
            src.push("normal", draws[-1][m]["eps2"])
        alogs = learning.online_actor_update(
            buffer=buf, agent=agent, pop=False, actor_optimizer=actor_opt, log_alphas=log_alphas, batch_size=B, clip=None,
            random_process=None, noise_clip=None, augmenter=aug, aug_mix=0.0, premade_replay_dicts=rds)
        _keep_logged(logged, "actor/", alogs)
    finally:
        _rng.set_source(old)
    return out


def sunrise_check(rank, world, dev):
    """SUNRISE members sharded over the ranks (SURVEY 8e, C3) == the single-GPU ensemble, member by member."""
    E, N, S, A, H, B, nbuf = max(3, world), 2, 17, 6, 64, 256, 4096
    cfg = dict(critic_lr=3e-4, actor_lr=3e-4)
    rng = np.random.default_rng(1)   # identical on every rank
    s = rng.standard_normal((nbuf, S), dtype=np.float32); a = rng.uniform(-1, 1, (nbuf, A)).astype(np.float32)
    r = rng.standard_normal(nbuf, dtype=np.float32); s1 = rng.standard_normal((nbuf, S), dtype=np.float32)
    d = rng.uniform(size=nbuf) < 0.01
    draws = [[dict(idx=rng.integers(0, nbuf, B), eps=rng.standard_normal((B, A)).astype(np.float32),
                   subset=rng.permutation(N)[:N].astype(np.int32), eps2=rng.standard_normal((B, A)).astype(np.float32))
              for _ in range(E)] for _ in range(2)]

    def buffer():
        b = ssb.replay.ReplayBuffer(nbuf, device=dev)
        b.load_experience({"obs": s}, a, r, {"obs": s1}, d)
        return b

    names = ("W1", "b1", "W2", "b2", "W3", "b3")
    full = build_ensemble(E, N, S, A, H, dev, seed=11)
    full_t = copy.deepcopy(full)
    init_c = {n: full._critic_arena.p[n].clone() for n in names}
    init_a = {n: full._actor_arena.p[n].clone() for n in names}
    ref = run_sunrise(full, full_t, buffer(), draws, list(range(E)), B, N, cfg)

    lo, hi = parallel.enable_member_sharding(E)
    shard = build_ensemble(hi - lo, N, S, A, H, dev, seed=11)
    for n in names:
        shard._critic_arena.p[n].copy_(init_c[n][lo * N:hi * N])
        shard._actor_arena.p[n].copy_(init_a[n][lo:hi])
    shard_t = copy.deepcopy(shard)
    got = run_sunrise(shard, shard_t, buffer(), draws, list(range(lo, hi)), B, N, cfg)
    parallel.disable()
    for n in names:
        assert_close(shard._critic_arena.p[n].cpu().numpy(), full._critic_arena.p[n][lo * N:hi * N].cpu().numpy(), 1e-4, 1.5e-5,
                        f"sunrise critics {n}")
        assert_close(shard._actor_arena.p[n].cpu().numpy(), full._actor_arena.p[n][lo:hi].cpu().numpy(), 1e-4, 1.5e-5,
                        f"sunrise actors {n}")
    for k in ref:
        assert_close(got[k], ref[k], 2e-4, 1e-6, f"sunrise {k}")
    print(f"[rank {rank}] sharded members [{lo},{hi}) == single-GPU SUNRISE update; losses {got}", flush=True)


def run_checks(rank, world, dev):
    """Both partitionings of SURVEY 8e on an initialised process group: raises on the first mismatch."""
    sunrise_check(rank, world, dev)
    critics_check(rank, world, dev)


def critics_check(rank, world, dev):
    N, M, S, A, H, B, nbuf = 10, 2, 17, 6, 256, 256, 4096
    cfg = dict(E=1, critic_lr=3e-4, actor_lr=3e-4)
    rng = np.random.default_rng(0)   # identical on every rank
    s = rng.standard_normal((nbuf, S), dtype=np.float32); a = rng.uniform(-1, 1, (nbuf, A)).astype(np.float32)
    r = rng.standard_normal(nbuf, dtype=np.float32); s1 = rng.standard_normal((nbuf, S), dtype=np.float32)
    d = rng.uniform(size=nbuf) < 0.01
    draws = [dict(idx=rng.integers(0, nbuf, B), eps=rng.standard_normal((B, A)).astype(np.float32),
                  subset=rng.permutation(N)[:M].astype(np.int32), eps2=rng.standard_normal((B, A)).astype(np.float32))
             for _ in range(3)]

    def buffer():
        b = ssb.replay.ReplayBuffer(nbuf, device=dev)
        b.load_experience({"obs": s}, a, r, {"obs": s1}, d)
        return b

    # (a) single-GPU reference on this rank
    full = build(N, S, A, H, dev, seed=7)
    full_t = copy.deepcopy(full)
    init_c = {n: full._critic_arena.p[n].clone() for n in ("W1", "b1", "W2", "b2", "W3", "b3")}
    init_a = full._actor_arena.flat.clone()
    ref = run(full, full_t, buffer(), draws, B, M, cfg)

    # (b) this rank's shard with the NCCL exchange
    lo, hi = parallel.enable_critic_sharding(N)
    shard = build(hi - lo, S, A, H, dev, seed=7)
    for n in init_c:
        shard._critic_arena.p[n].copy_(init_c[n][lo:hi])
    shard._actor_arena.flat.copy_(init_a)
    shard_t = copy.deepcopy(shard)
    got = run(shard, shard_t, buffer(), draws, B, M, cfg)
    # the software-pipelined block (target side + exchange of update k+1 next to update k) must give the same bits
    if parallel.peer_exchange_ready():
        pshard = build(hi - lo, S, A, H, dev, seed=7)
        for n in init_c:
            pshard._critic_arena.p[n].copy_(init_c[n][lo:hi])
        pshard._actor_arena.flat.copy_(init_a)
        pshard_t = copy.deepcopy(pshard)
        pgot = run(pshard, pshard_t, buffer(), draws, B, M, cfg, pipelined=True)
        torch.cuda.synchronize()
        for n in init_c:
            assert torch.equal(pshard._critic_arena.p[n], shard._critic_arena.p[n]), f"pipelined sharded block: critics {n} differ"
            assert torch.equal(pshard_t._critic_arena.p[n], shard_t._critic_arena.p[n]), f"pipelined sharded block: targets {n} differ"
        assert torch.equal(pshard._actor_arena.flat, shard._actor_arena.flat), "pipelined sharded block: actor differs"
        print(f"[rank {rank}] pipelined sharded block == sequential sharded updates (bit-identical); losses {pgot}", flush=True)
    parallel.disable()

    # the same with global-norm clipping (active: the norm is far above 0.05) and the DR3 regulariser (SURVEY 8e (3)): the
    # clip coefficient needs sum ||g||^2 over EVERY rank's critics, DR3 the mean over the global ensemble
    full2 = build(N, S, A, H, dev, seed=7)
    full2_t = copy.deepcopy(full2)
    ref2 = run(full2, full2_t, buffer(), draws, B, M, cfg, critic_clip=0.05, dr3_coeff=0.01)
    parallel.enable_critic_sharding(N)
    shard2 = build(hi - lo, S, A, H, dev, seed=7)
    for n in init_c:
        shard2._critic_arena.p[n].copy_(init_c[n][lo:hi])
    shard2._actor_arena.flat.copy_(init_a)
    shard2_t = copy.deepcopy(shard2)
    got2 = run(shard2, shard2_t, buffer(), draws, B, M, cfg, critic_clip=0.05, dr3_coeff=0.01)
    parallel.disable()
    for n in init_c:
        assert_close(shard2._critic_arena.p[n].cpu().numpy(), full2._critic_arena.p[n][lo:hi].cpu().numpy(), 1e-4, 1.5e-5, f"clip+DR3 critics {n}")
    for k in ref2:
        assert_close(got2[k], ref2[k], 2e-4, 1e-6, "clip+DR3 " + k)
    print(f"[rank {rank}] sharded critics with global-norm clip + DR3 == single-GPU update; {got2}", flush=True)

    for n in init_c:
        assert_close(shard._critic_arena.p[n].cpu().numpy(), full._critic_arena.p[n][lo:hi].cpu().numpy(), 1e-4, 1.5e-5, f"critics {n}")
        assert_close(shard_t._critic_arena.p[n].cpu().numpy(), full_t._critic_arena.p[n][lo:hi].cpu().numpy(), 1e-4, 1.5e-5, f"targets {n}")
    assert_close(shard._actor_arena.flat.cpu().numpy(), full._actor_arena.flat.cpu().numpy(), 1e-4, 1.5e-5, "actor")
    for k in ref:
        assert_close(got[k], ref[k], 2e-4, 1e-6, k)
    # replicated state must be bit-identical across ranks (same all-reduced gradient everywhere)
    chk = shard._actor_arena.flat.double().sum().reshape(1)
    lst = [torch.zeros_like(chk) for _ in range(world)]
    dist.all_gather(lst, chk)
    assert all(torch.equal(x, lst[0]) for x in lst), "actor replicas diverged"
    print(f"[rank {rank}] sharded critics [{lo},{hi}) == single-GPU update; losses {got}", flush=True)


def _same_logs(got, ref, what, skip=lambda k: False):
    """Every value this rank logged, under the key the single-GPU update logs it with, equals that update's."""
    for k, v in got.items():
        if skip(k):
            continue
        assert k in ref, f"{what}: {k} is not a key of the single-GPU update's logs"
        assert_close(v, ref[k], 2e-4, 1e-6, f"{what} log {k}")


def _sunrise_data(E, N, B, A, nbuf, S, dev, seed):
    rng = np.random.default_rng(seed)   # identical on every rank
    s = rng.standard_normal((nbuf, S), dtype=np.float32); a = rng.uniform(-1, 1, (nbuf, A)).astype(np.float32)
    r = rng.standard_normal(nbuf, dtype=np.float32); s1 = rng.standard_normal((nbuf, S), dtype=np.float32)
    d = rng.uniform(size=nbuf) < 0.01
    draws = [[dict(idx=rng.integers(0, nbuf, B), eps=rng.standard_normal((B, A)).astype(np.float32),
                   subset=rng.permutation(N)[:N].astype(np.int32), eps2=rng.standard_normal((B, A)).astype(np.float32),
                   adv_eps=rng.standard_normal((4, B, A)).astype(np.float32))
              for _ in range(E)] for _ in range(2)]

    def buffer():
        b = ssb.replay.ReplayBuffer(nbuf, device=dev)
        b.load_experience({"obs": s}, a, r, {"obs": s1}, d)
        return b

    return draws, buffer


def run_offline(agent, buf, draws, members, B, clip):
    """One offline (filtered BC) actor update of the members ``members`` (global ids) on draws[0]; returns (logs, the
    squared clip norm)."""
    _, actor_opt, enc_opt, _, _ = optimizers(agent, dict(E=len(members)))
    aug = augmentations.AugmentationSequence([augmentations.IdentityAug(B)])
    src = _rng.ScriptedSource()
    old = _rng.set_source(src)
    for m in members:
        src.push("indices", draws[0][m]["idx"])
        for j in range(4):
            src.push("normal", draws[0][m]["adv_eps"][j])
    try:
        logs = learning.offline_actor_update(
            buffer=buf, agent=agent, actor_optimizer=actor_opt, encoder_optimizer=enc_opt, batch_size=B, actor_clip=clip,
            update_encoder=False, encoder_clip=None, augmenter=aug, actor_lambda=0.0, aug_mix=0.0, per=False, filter_=True)
        assert src.empty(), "not every scripted draw was consumed"
    finally:
        _rng.set_source(old)
    return logs, float(_arena.FlatAdam.attach(actor_opt, agent._actor_arena).gnorm_sq)


NAMES = ("W1", "b1", "W2", "b2", "W3", "b3")


def critics_logs_check(rank, world, dev):
    """Critics sharded: every value the critic and actor updates log equals the single-GPU update's."""
    N, M, S, A, H, B, nbuf = 10, 2, 17, 6, 256, 256, 4096
    rng = np.random.default_rng(0)
    s = rng.standard_normal((nbuf, S), dtype=np.float32); a = rng.uniform(-1, 1, (nbuf, A)).astype(np.float32)
    r = rng.standard_normal(nbuf, dtype=np.float32); s1 = rng.standard_normal((nbuf, S), dtype=np.float32)
    d = rng.uniform(size=nbuf) < 0.01
    draws = [dict(idx=rng.integers(0, nbuf, B), eps=rng.standard_normal((B, A)).astype(np.float32),
                  subset=rng.permutation(N)[:M].astype(np.int32), eps2=rng.standard_normal((B, A)).astype(np.float32))
             for _ in range(2)]

    def buffer():
        b = ssb.replay.ReplayBuffer(nbuf, device=dev)
        b.load_experience({"obs": s}, a, r, {"obs": s1}, d)
        return b

    cfg = dict(E=1, critic_lr=3e-4, actor_lr=3e-4)
    full = build(N, S, A, H, dev, seed=7)
    init_c = {n: full._critic_arena.p[n].clone() for n in NAMES}
    init_a = full._actor_arena.flat.clone()
    ref_logs, got_logs = {}, {}
    run(full, copy.deepcopy(full), buffer(), draws, B, M, cfg, logged=ref_logs)
    lo, hi = parallel.enable_critic_sharding(N)
    shard = build(hi - lo, S, A, H, dev, seed=7)
    for n in NAMES:
        shard._critic_arena.p[n].copy_(init_c[n][lo:hi])
    shard._actor_arena.flat.copy_(init_a)
    run(shard, copy.deepcopy(shard), buffer(), draws, B, M, cfg, logged=got_logs)
    parallel.disable()
    _same_logs(got_logs, ref_logs, "critics sharded")
    print(f"[rank {rank}] sharded critics [{lo},{hi}): {len(got_logs)} logged values == single-GPU update", flush=True)


def sunrise_dr3_check(rank, world, dev):
    """Members sharded, sunrise weights and DR3: parameters and every logged value equal the single-GPU update's."""
    E, N, S, A, H, B, nbuf = max(3, world), 2, 17, 6, 64, 256, 4096
    draws, buffer = _sunrise_data(E, N, B, A, nbuf, S, dev, seed=1)
    cfg = dict(critic_lr=3e-4, actor_lr=3e-4)
    full = build_ensemble(E, N, S, A, H, dev, seed=11)
    init_c = {n: full._critic_arena.p[n].clone() for n in NAMES}
    init_a = {n: full._actor_arena.p[n].clone() for n in NAMES}
    ref_logs, got_logs = {}, {}
    run_sunrise(full, copy.deepcopy(full), buffer(), draws, list(range(E)), B, N, cfg, dr3_coeff=0.01, logged=ref_logs)
    lo, hi = parallel.enable_member_sharding(E)
    shard = build_ensemble(hi - lo, N, S, A, H, dev, seed=11)
    for n in NAMES:
        shard._critic_arena.p[n].copy_(init_c[n][lo * N:hi * N])
        shard._actor_arena.p[n].copy_(init_a[n][lo:hi])
    run_sunrise(shard, copy.deepcopy(shard), buffer(), draws, list(range(lo, hi)), B, N, cfg, dr3_coeff=0.01,
                logged=got_logs)
    parallel.disable()
    for n in NAMES:
        assert_close(shard._critic_arena.p[n].cpu().numpy(), full._critic_arena.p[n][lo * N:hi * N].cpu().numpy(), 1e-4,
                     1.5e-5, f"sunrise + DR3 critics {n}")
        assert_close(shard._actor_arena.p[n].cpu().numpy(), full._actor_arena.p[n][lo:hi].cpu().numpy(), 1e-4, 1.5e-5,
                     f"sunrise + DR3 actors {n}")
    # (the Bellman-weight statistics are those of the rank's last member: the single-GPU ones on the last rank)
    _same_logs(got_logs, ref_logs, "members sharded + DR3", skip=lambda k: "bellman_weights/" in k and hi != E)
    print(f"[rank {rank}] sharded members [{lo},{hi}) with DR3 == single-GPU update ({len(got_logs)} logged values)",
          flush=True)


def offline_members_check(rank, world, dev):
    """Members sharded, the offline actor update (advantage filter) with a clip that engages (Adam absorbs most of a
    uniform gradient scale, the clip does not): actors and logged values equal the single-GPU update's."""
    E, N, S, A, H, B, nbuf, clip = max(3, world), 2, 17, 6, 64, 256, 4096, 1e-3
    draws, buffer = _sunrise_data(E, N, B, A, nbuf, S, dev, seed=2)
    full = build_ensemble(E, N, S, A, H, dev, seed=13)
    init_a = {n: full._actor_arena.p[n].clone() for n in NAMES}
    init_c = {n: full._critic_arena.p[n].clone() for n in NAMES}
    ref_logs, gsq = run_offline(full, buffer(), draws, list(range(E)), B, clip)
    assert gsq > 100 * clip * clip, f"the clip does not engage: |g|^2 = {gsq}"
    lo, hi = parallel.enable_member_sharding(E)
    shard = build_ensemble(hi - lo, N, S, A, H, dev, seed=13)
    for n in NAMES:
        shard._critic_arena.p[n].copy_(init_c[n][lo * N:hi * N])
        shard._actor_arena.p[n].copy_(init_a[n][lo:hi])
    got_logs, gsq_s = run_offline(shard, buffer(), draws, list(range(lo, hi)), B, clip)
    parallel.disable()
    assert_close(gsq_s, gsq, 1e-4, 0.0, "offline actor clip norm |g|^2")
    for n in NAMES:
        assert_close(shard._actor_arena.p[n].cpu().numpy(), full._actor_arena.p[n][lo:hi].cpu().numpy(), 1e-4, 1.5e-5,
                     f"offline actors {n}")
    _same_logs({k: v for k, v in got_logs.items() if not k.startswith("gradients/")}, ref_logs, "offline members sharded")
    print(f"[rank {rank}] sharded members [{lo},{hi}): clipped offline actor update == single-GPU update", flush=True)


def logged_checks(rank, world, dev):
    """What run_checks leaves out (bench.py's gate stays as it is): the logged values on every rank, DR3 with the members
    sharded and the offline actor update with the members sharded."""
    critics_logs_check(rank, world, dev)
    sunrise_dr3_check(rank, world, dev)
    offline_members_check(rank, world, dev)


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    run_checks(rank, world, dev)
    logged_checks(rank, world, dev)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()

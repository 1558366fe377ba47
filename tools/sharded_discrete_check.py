#!/usr/bin/env python
"""Sharded SAC-Discrete ensembles must equal the single-GPU discrete update (one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29531 \\
        tools/sharded_discrete_check.py

Every rank runs (a) the whole ensemble on its own GPU and (b) its shard of the same ensemble with the exchanges of
super_sac_b200.parallel, on the same scripted draws, and compares parameters, TD targets and logged scalars at rtol 1e-4:

- critics sharded, N = 3 and N = 10, DR3 + global-norm clipping + PopArt, with the priority refresh: critic, actor and
  temperature updates;
- critics sharded, E = 2 members: offline filtered BC on prioritised batches, with the priority refresh;
- members sharded, E = 3, sunrise weights: critic, actor and temperature updates.

Python's ``random`` (the host draw of the member that refreshes priorities) is seeded differently on each rank.  The
replicated state (actor, log_alpha, PopArt, the PER trees) must be bit-identical on every rank, and a sharded
``lu.pipelined_updates()`` block, eager and captured as one CUDA graph, must give the bits of the same updates run
sequentially.  Each passed check prints one ``[rank r] ...`` line.
"""
import contextlib
import copy
import math
import os
import random
import sys
from itertools import chain

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "tools")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np
import torch
import torch.distributed as dist

import benchlib as bl
import super_sac_b200 as ssb
from sharded_check import assert_close
from super_sac_b200 import _rng, augmentations, graphed, learning, learning_utils as lu, nets, parallel

IdentityEncoder, _ = bl._encoders(ssb)
NAMES = ("W1", "b1", "W2", "b2", "W3", "b3")
S, A, H, B, NBUF = 64, 18, 256, 256, 4096


def _data(seed):
    rng = np.random.default_rng(seed)   # identical on every rank
    return dict(s=rng.standard_normal((NBUF, S), dtype=np.float32), a=rng.integers(0, A, (NBUF, 1)).astype(np.float32),
                r=rng.standard_normal(NBUF, dtype=np.float32), s1=rng.standard_normal((NBUF, S), dtype=np.float32),
                d=(rng.uniform(size=NBUF) < 0.05).astype(np.float32), prio=rng.uniform(0.1, 2.0, NBUF))


def _buffer(data, dev):
    b = ssb.replay.ReplayBuffer(NBUF, device=dev)
    b.load_experience({"obs": data["s"]}, data["a"], data["r"], {"obs": data["s1"]}, data["d"])
    b.update_priorities(np.arange(NBUF), data["prio"])
    return b


def _agent(E, N, dev, popart, init=None, nets_=None, members=None):
    """A discrete agent; ``init`` (the whole ensemble's parameters) loaded at the rows ``nets_`` / ``members``."""
    agent = ssb.Agent(act_space_size=A, encoder=IdentityEncoder(S), actor_network_cls=nets.mlps.DiscreteActor,
                      critic_network_cls=nets.mlps.DiscreteCritic, discrete=True, ensemble_size=E, num_critics=N,
                      hidden_size=H, auto_rescale_targets=popart)
    agent.to(dev)
    if init is not None:
        with torch.no_grad():
            for n in NAMES:
                agent._critic_arena.p[n].copy_(init["c"][n][nets_])
                agent._actor_arena.p[n].copy_(init["a"][n][members])
    target = copy.deepcopy(agent)
    return agent, target


def _params(agent):
    return {"c": {n: agent._critic_arena.p[n].clone() for n in NAMES}, "a": {n: agent._actor_arena.p[n].clone() for n in NAMES}}


def _opts(agent, E, dev):
    c_opt = torch.optim.Adam(chain(*(c.parameters() for c in agent.critics)), lr=3e-4)
    a_opt = torch.optim.Adam(chain(*(a.parameters() for a in agent.actors)), lr=3e-4)
    e_opt = torch.optim.Adam(agent.encoder.parameters(), lr=1e-4)
    las = [torch.tensor([math.log(0.1)], device=dev, requires_grad=True) for _ in range(E)]
    return c_opt, a_opt, e_opt, las, [torch.optim.Adam([la], lr=1e-4, betas=(0.5, 0.999)) for la in las]


def _no_grads(logs):
    return {k: float(v) for k, v in logs.items() if not k.startswith("gradients/")}


def run_online(agent, target, buf, draws, members, E, hp, rseed=5):
    """len(draws) critic updates (+ Polyak), then one actor and one temperature update on the last batches.  ``draws``:
    per step, per GLOBAL member {idx, subset}; this agent's members are ``members``.  ``rseed`` seeds Python's ``random``
    (the host member draws).  Returns TD targets, weights, logs."""
    dev = agent._critic_arena.device
    c_opt, a_opt, e_opt, las, al_opts = _opts(agent, E, dev)
    aug = augmentations.AugmentationSequence([augmentations.IdentityAug(B)])
    out, rec = {}, {}
    o_td, o_bw = lu.compute_td_targets, lu.compute_backup_weights
    lu.compute_td_targets = lambda *a, **k: rec.setdefault("td", []).append(o_td(*a, **k)) or rec["td"][-1]
    lu.compute_backup_weights = lambda *a, **k: rec.setdefault("w", []).append(o_bw(*a, **k)) or rec["w"][-1]
    old = _rng.set_source(_rng.ScriptedSource())
    random.seed(rseed)
    try:
        for step, dr in enumerate(draws):
            src = _rng.ScriptedSource()
            _rng.set_source(src)
            for m in members:
                src.push("indices", dr[m]["idx"]).push("subsets", dr[m]["subset"])
            rec.clear()
            logs, rds = learning.critic_update(
                buffer=buf, agent=agent, target_agent=target, critic_optimizer=c_opt, encoder_optimizer=e_opt,
                log_alphas=las, batch_size=B, gamma=0.99, critic_clip=hp.get("clip"), encoder_clip=None,
                target_critic_ensemble_n=hp["M"], weighted_bellman_temp=hp.get("temp"), weight_type=hp.get("weights"),
                pop=hp.get("pop", False), augmenter=aug, encoder_lambda=0.0, random_process=None, noise_clip=None,
                aug_mix=0.0, discrete=True, per=False, update_priorities=hp.get("prio", False), dr3_coeff=hp.get("dr3", 0.0))
            assert src.empty(), "not every scripted draw was consumed"
            for ac, tc in zip(agent.critics, target.critics):
                lu.soft_update(tc, ac, 0.005)
            out[f"logs{step}"] = _no_grads(logs)
            for i, m in enumerate(members):
                out[f"td{step}_{m}"] = rec["td"][i][0].cpu().numpy()
                w = rec["w"][i]
                out[f"w{step}_{m}"] = w.cpu().numpy() if torch.is_tensor(w) else np.float32(w)
        out["actor_logs"] = _no_grads(learning.online_actor_update(
            buffer=buf, agent=agent, pop=hp.get("pop", False), actor_optimizer=a_opt, log_alphas=las, batch_size=B,
            clip=1.0, random_process=None, noise_clip=None, augmenter=aug, aug_mix=0.0, premade_replay_dicts=rds,
            per=False, discrete=True))
        out["alpha_logs"] = _no_grads(learning.alpha_update(
            buffer=buf, agent=agent, optimizers=al_opts, batch_size=B, log_alphas=las, augmenter=aug, aug_mix=0.0,
            target_entropy=-math.log(1.0 / A) * 0.98, premade_replay_dicts=rds, discrete=True))
        for i, m in enumerate(members):
            out[f"log_alpha_{m}"] = las[i].detach().cpu().numpy()
    finally:
        lu.compute_td_targets, lu.compute_backup_weights = o_td, o_bw
        _rng.set_source(old)
    return out


def _cmp_runs(got, ref, what, keep=lambda k: True):
    for k, v in ref.items():
        if k not in got:
            continue   # a member of another rank
        if isinstance(v, dict):
            for kk, vv in v.items():
                if keep(kk):
                    assert kk in got[k], f"{what}: {k} lacks {kk}"
                    assert_close(got[k][kk], vv, 2e-4, 1e-6, f"{what} {k}/{kk}")
        else:
            assert_close(got[k], v, 1e-4, 1e-5, f"{what} {k}")


def _same_on_all_ranks(t, what):
    t = t.detach().reshape(-1).contiguous().clone()
    lst = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(lst, t)
    assert all(torch.equal(x, lst[0]) for x in lst), f"{what}: replicas differ between ranks"


def _popart_state(agent):
    return torch.cat([torch.cat([p.mu, p.nu, p.w, p.b]).reshape(-1) for p in agent.popart if p] or [torch.zeros(1)])


def critics_check(rank, world, dev, N):
    """Critics sharded: N = 3 or 10 over the ranks, DR3 + clip + PopArt + priority refresh."""
    hp = dict(M=2, clip=0.5, dr3=0.01, pop=True, prio=True)
    data = _data(N)
    rng = np.random.default_rng(100 + N)
    draws = [[dict(idx=rng.integers(0, NBUF, B), subset=rng.permutation(N)[:2].astype(np.int32))] for _ in range(3)]
    torch.manual_seed(N)
    full, full_t = _agent(1, N, dev, popart=True)
    init = _params(full)
    buf_f = _buffer(data, dev)
    ref = run_online(full, full_t, buf_f, draws, [0], 1, hp)

    lo, hi = parallel.enable_critic_sharding(N)
    shard, shard_t = _agent(1, hi - lo, dev, popart=True, init=init, nets_=slice(lo, hi), members=slice(0, 1))
    buf_s = _buffer(data, dev)
    got = run_online(shard, shard_t, buf_s, draws, [0], 1, hp, rseed=5 + rank)   # the ranks' host draws differ
    parallel.disable()
    torch.cuda.synchronize()
    _cmp_runs(got, ref, f"critics N={N}")
    for n in NAMES:
        assert_close(shard._critic_arena.p[n].cpu().numpy(), full._critic_arena.p[n][lo:hi].cpu().numpy(), 1e-4, 1.5e-5,
                     f"critics N={N} {n}")
        assert_close(shard_t._critic_arena.p[n].cpu().numpy(), full_t._critic_arena.p[n][lo:hi].cpu().numpy(), 1e-4,
                     1.5e-5, f"critics N={N} target {n}")
    assert_close(shard._actor_arena.flat.cpu().numpy(), full._actor_arena.flat.cpu().numpy(), 1e-4, 1.5e-5, f"N={N} actor")
    assert_close(_popart_state(shard).cpu().numpy(), _popart_state(full).cpu().numpy(), 1e-4, 1e-6, f"N={N} popart")
    assert_close(buf_s._it_sum.cpu().numpy(), buf_f._it_sum.cpu().numpy(), 1e-4, 1e-9, f"N={N} PER sum tree")
    for t, what in ((shard._actor_arena.flat, "actor"), (got["log_alpha_0"], "log_alpha"), (_popart_state(shard), "popart"),
                    (buf_s._it_sum, "PER sum tree"), (buf_s._it_min, "PER min tree")):
        _same_on_all_ranks(torch.as_tensor(t, device=dev), f"critics N={N} {what}")
    print(f"[rank {rank}] sharded discrete critics N={N} [{lo},{hi}) == single-GPU update "
          f"(loss {got['logs2']['losses/critic_overall_loss']:.6f})", flush=True)


def offline_check(rank, world, dev):
    """Critics of E = 2 members sharded: filtered BC on prioritised batches, with the priority refresh."""
    E, N = 2, max(2, world)
    data = _data(7)
    rng = np.random.default_rng(7)
    us = [[rng.uniform(size=B) for _ in range(E)] for _ in range(2)]
    torch.manual_seed(7)
    full, _ = _agent(E, N, dev, popart=True)
    init = _params(full)

    def run(agent, buf, rseed):
        _, a_opt, e_opt, _, _ = _opts(agent, E, dev)
        aug = augmentations.AugmentationSequence([augmentations.IdentityAug(B)])
        old = _rng.set_source(_rng.ScriptedSource())
        random.seed(rseed)
        out = {}
        try:
            for step, u in enumerate(us):
                src = _rng.ScriptedSource()
                _rng.set_source(src)
                for m in range(E):
                    src.push("uniform01", u[m])
                out[f"logs{step}"] = _no_grads(learning.offline_actor_update(
                    buffer=buf, agent=agent, actor_optimizer=a_opt, encoder_optimizer=e_opt, batch_size=B, actor_clip=1.0,
                    update_encoder=False, encoder_clip=None, augmenter=aug, actor_lambda=0.0, aug_mix=0.0,
                    premade_replay_dicts=None, per=True, discrete=True, filter_=True))
                assert src.empty()
        finally:
            _rng.set_source(old)
        return out

    buf_f = _buffer(data, dev)
    ref = run(full, buf_f, 3)
    lo, hi = parallel.enable_critic_sharding(N)
    rows = torch.cat([torch.arange(i * N + lo, i * N + hi) for i in range(E)]).to(dev)
    shard, _ = _agent(E, hi - lo, dev, popart=True, init=init, nets_=rows, members=slice(0, E))
    buf_s = _buffer(data, dev)
    got = run(shard, buf_s, 3 + rank)   # rank 0's member draws (those of the reference) hold on every rank
    parallel.disable()
    torch.cuda.synchronize()
    _cmp_runs(got, ref, "offline")
    assert_close(shard._actor_arena.flat.cpu().numpy(), full._actor_arena.flat.cpu().numpy(), 1e-4, 1.5e-5, "offline actor")
    assert_close(buf_s._it_sum.cpu().numpy(), buf_f._it_sum.cpu().numpy(), 1e-4, 1e-9, "offline PER sum tree")
    for t, what in ((shard._actor_arena.flat, "actor"), (buf_s._it_sum, "PER sum tree"), (buf_s._it_min, "PER min tree")):
        _same_on_all_ranks(t, f"offline {what}")
    print(f"[rank {rank}] sharded discrete critics, offline filtered BC + priority refresh [{lo},{hi}) == single-GPU "
          f"update", flush=True)


def members_check(rank, world, dev):
    """Members sharded: E = max(3, world) over the ranks, sunrise weights."""
    E, N = max(3, world), 2
    hp = dict(M=N, weights="sunrise", temp=20.0)
    data = _data(3)
    rng = np.random.default_rng(3)
    draws = [[dict(idx=rng.integers(0, NBUF, B), subset=rng.permutation(N).astype(np.int32)) for _ in range(E)]
             for _ in range(2)]
    torch.manual_seed(3)
    full, full_t = _agent(E, N, dev, popart=False)
    init = _params(full)
    ref = run_online(full, full_t, _buffer(data, dev), draws, list(range(E)), E, hp)
    lo, hi = parallel.enable_member_sharding(E)
    shard, shard_t = _agent(hi - lo, N, dev, popart=False, init=init, nets_=slice(lo * N, hi * N), members=slice(lo, hi))
    got = run_online(shard, shard_t, _buffer(data, dev), draws, list(range(lo, hi)), hi - lo, hp)
    parallel.disable()
    torch.cuda.synchronize()
    last = hi == E

    def keep(k):   # per-member keys of this rank's members; the sunrise weights logged last are the last member's
        if k.startswith("bellman_weights/"):
            return last
        tail = k.rsplit("_", 1)[-1]
        return not tail.isdigit() or lo <= int(tail) < hi

    _cmp_runs(got, ref, "members", keep)
    for n in NAMES:
        assert_close(shard._critic_arena.p[n].cpu().numpy(), full._critic_arena.p[n][lo * N:hi * N].cpu().numpy(), 1e-4,
                     1.5e-5, f"members critics {n}")
        assert_close(shard._actor_arena.p[n].cpu().numpy(), full._actor_arena.p[n][lo:hi].cpu().numpy(), 1e-4, 1.5e-5,
                     f"members actors {n}")
    print(f"[rank {rank}] sharded discrete members [{lo},{hi}) of {E} == single-GPU SUNRISE update", flush=True)


def pipelined_check(rank, world, dev, N=10):
    """A sharded UTD block inside lu.pipelined_updates(), eager and captured as one graph, == the sequential schedule."""
    data = _data(11)

    def build():
        ssb.manual_seed(11)   # the same Philox stream on every rank and in every build
        torch.manual_seed(11)
        lo, hi = parallel.my_range()
        agent, target = _agent(1, hi - lo, dev, popart=False)
        with torch.no_grad():
            for n in NAMES:
                g = torch.Generator().manual_seed(NAMES.index(n))
                full = torch.randn((N,) + tuple(agent._critic_arena.p[n].shape[1:]), generator=g) * 0.05
                agent._critic_arena.p[n].copy_(full[lo:hi])
                target._critic_arena.p[n].copy_(full[lo:hi])
        buf = _buffer(data, dev)
        c_opt, a_opt, e_opt, las, al_opts = _opts(agent, 1, dev)
        aug = augmentations.AugmentationSequence([augmentations.IdentityAug(B)])
        kw = dict(buffer=buf, agent=agent, target_agent=target, critic_optimizer=c_opt, encoder_optimizer=e_opt,
                  log_alphas=las, batch_size=B, gamma=0.99, critic_clip=None, encoder_clip=None, target_critic_ensemble_n=2,
                  weighted_bellman_temp=None, weight_type=None, pop=False, augmenter=aug, encoder_lambda=0.0,
                  random_process=None, noise_clip=None, aug_mix=0.0, discrete=True, per=False, update_priorities=False,
                  dr3_coeff=0.0)

        def block(pipelined):
            with (lu.pipelined_updates() if pipelined else contextlib.nullcontext()):
                for k in range(8):
                    logs, rds = learning._critic_update_impl(**kw)
                    if k % 2 == 0:
                        for ac, tc in zip(agent.critics, target.critics):
                            lu.soft_update(tc, ac, 0.005)
                learning._online_actor_update_impl(
                    buffer=buf, agent=agent, pop=False, actor_optimizer=a_opt, log_alphas=las, batch_size=B, clip=None,
                    random_process=None, noise_clip=None, augmenter=aug, aug_mix=0.0, premade_replay_dicts=rds, per=False,
                    discrete=True)
                learning.alpha_update(buffer=buf, agent=agent, optimizers=al_opts, batch_size=B, log_alphas=las,
                                      augmenter=aug, aug_mix=0.0, target_entropy=-math.log(1.0 / A) * 0.98,
                                      premade_replay_dicts=rds, discrete=True)
            return logs

        return (agent, target, las), block

    def state(st):
        agent, target, las = st
        return [agent._critic_arena.flat.clone(), target._critic_arena.flat.clone(), agent._actor_arena.flat.clone(),
                las[0].detach().clone()]

    old = _rng.source()
    lo, hi = parallel.enable_critic_sharding(N)
    try:
        _rng.set_source(_rng.PhiloxSource(11))
        st0, block0 = build()
        for _ in range(5):
            block0(False)
        torch.cuda.synchronize()
        s0 = state(st0)
        kinds = []
        for captured in (False, True):
            st1, block1 = build()
            if captured:
                g = graphed.GraphedCall(lambda: block1(True), warmup=2)   # two eager pipelined blocks, then three replays
                for _ in range(3):
                    g.replay()
            else:
                for _ in range(5):
                    block1(True)
            torch.cuda.synchronize()
            assert lu.pipeline() is None
            for a, b, what in zip(state(st1), s0, ("critics", "targets", "actor", "log_alpha")):
                assert torch.equal(a, b), f"pipelined sharded block ({'graph' if captured else 'eager'}): {what} differ"
            kinds.append("graph" if captured else "eager")
        _same_on_all_ranks(s0[2], "pipelined block actor")
        piped = parallel.peer_exchange_ready()
    finally:
        parallel.disable()
        _rng.set_source(old)
    print(f"[rank {rank}] sharded discrete pipelined block ({', '.join(kinds)}) == sequential updates, bit-identical "
          f"[{lo},{hi}); exchange: {parallel.exchange_name()}; front stream used: {piped}", flush=True)


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    for N in sorted({max(3, world), 10}):   # (3 critics cannot be spread over more than 3 ranks)
        critics_check(rank, world, dev, N)
    offline_check(rank, world, dev)
    members_check(rank, world, dev)
    pipelined_check(rank, world, dev)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()

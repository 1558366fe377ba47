#!/usr/bin/env python
"""The batch-sharded update (parallel.enable_batch_sharding) must equal the single-GPU update.  One rank per GPU, under
torchrun (a world of one rank is allowed: then every comparison is bitwise):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29541 \
        tools/batch_sharded_check.py [--c4-baseline]

Every rank builds the same workload twice on its own GPU, each with its own Philox stream on the same seed: a plain one
(sharding switched off around its calls) and a batch-sharded one.  It checks

- ssac_peer_allreduce alone (parallel.all_reduce_flat_) at 1, 3, 4097 and 2^22 + 5 floats: bitwise the host's rank-order
  fp32 sum and the same on every rank, twice back to back and inside a captured CUDA graph;
- the batch: this rank's rows are bitwise rows [lo, hi) of the plain batch (classic ring, state and pixel observations);
- a sequence of critic + Polyak + actor + temperature updates at the sac / redq shapes and at the drqv2 pixel shape
  (B = 64; B = 61 as well, which no world of 2..8 ranks divides), where every other step the actor and temperature
  updates sample batches of their own instead of reusing the critic update's: parameters, target parameters, encoder parameters,
  optimiser moments and every logged value match the plain update (rtol 1e-4 over several ranks; over one rank the
  state bitwise and the logs, whose sums are accumulated with atomics, to rtol 1e-6), and
  the flat arenas are bitwise identical on every rank after every step;
- a captured step (graphed.GraphedCall) replays bit-identical to the eager sharded step;
- with --c4-baseline, one drqv2 update at the BASELINE batch of 512.
Each passed part prints "[rank r] batch-sharded <part>: ok".
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "tools")):
    if _p not in sys.path:
        sys.path.insert(0, _p)
import numpy as np
import torch
import torch.distributed as dist

import benchlib as bl
import super_sac_b200 as ssb
from super_sac_b200 import _rng, graphed, learning_utils as lu, parallel

RTOL, ATOL = 1e-4, 1e-6


def say(msg):
    print(f"[rank {dist.get_rank()}] batch-sharded {msg}", flush=True)


class Side:
    """One workload with its own Philox stream; ``sharded`` says whether batch sharding is on around its calls."""

    def __init__(self, name, dev, sharded, overrides):
        self.w = bl.Workload(ssb, name, dev, seed=7, buffer_size=overrides.pop("buffer", None), fill_on_device=True,
                             overrides=overrides)
        self.src = _rng.PhiloxSource(7)
        self.sharded = sharded

    def __enter__(self):
        _rng.set_source(self.src)
        if self.sharded:
            parallel.enable_batch_sharding()
        else:
            parallel.disable()
        return self.w

    def __exit__(self, *a):
        parallel.disable()

    def step(self, k, fetch=True, own_batches=False):
        """own_batches: the actor and temperature updates sample their own batches (premade_replay_dicts=None)."""
        with self as w:
            logs, rds = w.critic_update()
            w.polyak()
            alogs = w.actor_and_alpha(None if own_batches else rds)
            return {**dict(logs), **dict(alogs)} if fetch else None

    def state(self):
        w = self.w
        out = {"critics": w.agent._critic_arena.flat, "actor": w.agent._actor_arena.flat,
               "target_critics": w.target._critic_arena.flat, "log_alpha": w.log_alphas[0].detach()}
        for tag, m in (("encoder", w.agent.encoder), ("target_encoder", w.target.encoder)):
            for j, p in enumerate(m.parameters()):
                out[f"{tag}.{j}"] = p.detach()
        for tag, opt in (("critic_opt", w.critic_opt), ("actor_opt", w.actor_opt), ("enc_opt", w.enc_opt)):
            for j, st in enumerate(opt.state.values()):
                for key in ("exp_avg", "exp_avg_sq"):
                    if key in st:
                        out[f"{tag}.{j}.{key}"] = st[key]
        return {k: v.detach().reshape(-1).clone() for k, v in out.items()}


def check_close(what, got, want, exact):
    if exact:
        assert torch.equal(got, want), f"{what}: not bit-identical (max |diff| {(got - want).abs().max().item():.3e})"
    else:
        assert torch.allclose(got, want, rtol=RTOL, atol=ATOL), f"{what}: max |diff| {(got - want).abs().max().item():.3e}"


def check_logs(what, got, want, exact):
    assert set(got) == set(want), (what, sorted(set(got) ^ set(want)))
    for k in want:
        g, w_ = float(got[k]), float(want[k])
        # (on one rank the parameters are compared bitwise; logged batch sums are accumulated with atomics, whose order
        # differs from run to run even between two plain updates, so they get a float32 rounding margin)
        tol = 1e-6 if exact else RTOL
        ok = abs(g - w_) <= tol * abs(w_) + (1e-7 if exact else 1e-5)
        assert ok, f"{what}: log {k} = {g!r}, single GPU {w_!r}"


def same_on_every_rank(what, t):
    t = t.contiguous()
    parts = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(parts, t)
    for r, p in enumerate(parts):
        assert torch.equal(p, t), f"{what}: rank {r} differs"


def allreduce_part(dev):
    world, rank = dist.get_world_size(), dist.get_rank()
    parallel.enable_batch_sharding()
    try:
        for n in (1, 3, 4097, 2**22 + 5):
            xs = [np.random.default_rng(1000 * n + r).standard_normal(n).astype(np.float32) for r in range(world)]
            want = xs[0].copy()
            for r in range(1, world):
                want = want + xs[r]   # rank order, fp32
            want = torch.from_numpy(want).to(dev)
            for call in range(2):   # back to back on the same site
                t = torch.from_numpy(xs[rank] * (1 + call)).to(dev)
                parallel.all_reduce_flat_(t, site=f"check{n}")
                check_close(f"all-reduce n={n} call {call}", t, want * (1 + call), exact=True)
                same_on_every_rank(f"all-reduce n={n}", t)
            t = torch.empty(n, dtype=torch.float32, device=dev)
            x = torch.from_numpy(xs[rank]).to(dev)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                t.copy_(x)
                parallel.all_reduce_flat_(t, site=f"check{n}")
            for _ in range(2):
                t.zero_()
                g.replay()
                torch.cuda.synchronize()
                check_close(f"captured all-reduce n={n}", t, want, exact=True)
            dist.barrier()
    finally:
        parallel.disable()
    say(f"all-reduce ({parallel.exchange_name()}): ok")


def batch_part(dev, name, overrides):
    world = dist.get_world_size()
    plain, shard = Side(name, dev, False, dict(overrides)), Side(name, dev, True, dict(overrides))
    B = plain.w.cfg["B"]
    lo, hi = parallel.local_range(B, world, dist.get_rank())
    outs = []
    for side in (plain, shard):
        with side as w:
            draws = lu.draw_for_critic_member(w.buffer, w.agent, B, 2, w.noise, False)
            rd = lu.sample_move_and_augment(w.buffer, B, w.augmenter, w.kw["aug_mix"] if name != "drqv2" else 0.5,
                                            per=False, _idx=draws["idx"])
            o, a, r, o1, d = rd["primary_batch"]
            outs.append([*o.values(), a, r, *o1.values(), d] + ([draws["normal"]] if draws["normal"] is not None else []))
    for j, (full, part) in enumerate(zip(*outs)):
        check_close(f"{name} batch tensor {j}", part, full[lo:hi], exact=True)
    say(f"batch {name} B={B}: ok")


def update_part(dev, name, overrides, steps=4, captured=True):
    world = dist.get_world_size()
    exact = world == 1
    plain, shard = Side(name, dev, False, dict(overrides)), Side(name, dev, True, dict(overrides))
    B = plain.w.cfg["B"]
    for k in range(steps):
        own = k % 2 == 1   # every other step the actor and temperature updates sample their own batches
        want_logs, got_logs = plain.step(k, own_batches=own), shard.step(k, own_batches=own)
        torch.cuda.synchronize()
        want, got = plain.state(), shard.state()
        for key in want:
            check_close(f"{name} step {k} {key}", got[key], want[key], exact)
            same_on_every_rank(f"{name} step {k} {key}", got[key])
        check_logs(f"{name} step {k}", got_logs, want_logs, exact)
    say(f"updates {name} B={B}: ok")
    if not captured:
        return
    # a captured sharded step against the same eager sharded step (the same calls, its own workload and Philox stream)
    eager, cap = Side(name, dev, True, dict(overrides)), Side(name, dev, True, dict(overrides))
    with cap:
        g = graphed.GraphedCall(lambda: cap.step(0, fetch=False), warmup=2)
    for k in range(2):
        eager.step(0)
    for k in range(3):
        eager.step(0)
        with cap:
            g.replay()
        torch.cuda.synchronize()
        want, got = eager.state(), cap.state()
        for key in want:
            check_close(f"{name} captured step {k} {key}", got[key], want[key], exact=True)
    say(f"captured {name} B={B}: ok")


def main():
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    try:
        allreduce_part(dev)
        small = dict(buffer=20_000)
        pix = dict(buffer=4096, B=64)
        for name, ov in (("sac", small), ("redq", small), ("drqv2", pix)):
            batch_part(dev, name, ov)
        for name, ov in (("sac", small), ("redq", dict(small, B=61)), ("drqv2", pix), ("drqv2", dict(pix, B=61))):
            update_part(dev, name, ov, captured=ov.get("B") != 61)
        if "--c4-baseline" in sys.argv:
            update_part(dev, "drqv2", dict(buffer=8192), steps=1, captured=False)
        say("check: ok")
    finally:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Sharded SAC-Discrete ensembles timed on the device, one rank per GPU (torchrun):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node G tools/bench_discrete_sharded.py --steps 300 --warmup 30

Two workloads at Atari-like head sizes (64 features, H = 256, 18 actions, B = 256), each with the ensemble sharded over
the G ranks of the run and, on rank 0 alone, unsharded as the same-run baseline:

    critics    N = 10 critics (REDQ subset M = 2), one member: parallel.enable_critic_sharding(10)
    members    E = 4 members with 2 critics each and sunrise weights: parallel.enable_member_sharding(4)

For each it reports microseconds per critic update (critic_update + Polyak) and per full step (critic + Polyak + online
actor + temperature update), eager launches with logs read back every call, CUDA events around --steps calls after
--warmup calls.  Rank 0 prints one JSON line per workload with the card's name and power limit and the exchange in use.
"""
import argparse
import json
import math
import os
import subprocess
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
from super_sac_b200 import augmentations, learning, learning_utils as lu, nets, parallel

IdentityEncoder, _ = bl._encoders(ssb)
S, A, H, B, NBUF = 64, 18, 256, 256, 100_000


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or f"{torch.cuda.get_device_name()}, power limit unknown"


def setup(E, N, dev):
    ssb.manual_seed(1)   # the same Philox stream on every rank (critic sharding replicates the batch draws)
    torch.manual_seed(1)
    agent = ssb.Agent(act_space_size=A, encoder=IdentityEncoder(S), actor_network_cls=nets.mlps.DiscreteActor,
                      critic_network_cls=nets.mlps.DiscreteCritic, discrete=True, ensemble_size=E, num_critics=N,
                      hidden_size=H)
    agent.to(dev)
    import copy

    target = copy.deepcopy(agent)
    rng = np.random.default_rng(0)
    buf = ssb.replay.ReplayBuffer(NBUF, device=dev)
    buf.load_experience({"obs": rng.standard_normal((NBUF, S), dtype=np.float32)},
                        rng.integers(0, A, (NBUF, 1)).astype(np.float32), rng.standard_normal(NBUF, dtype=np.float32),
                        {"obs": rng.standard_normal((NBUF, S), dtype=np.float32)},
                        (rng.uniform(size=NBUF) < 0.01).astype(np.float32))
    c_opt = torch.optim.Adam(chain(*(c.parameters() for c in agent.critics)), lr=3e-4)
    a_opt = torch.optim.Adam(chain(*(a.parameters() for a in agent.actors)), lr=3e-4)
    e_opt = torch.optim.Adam(agent.encoder.parameters(), lr=1e-4)
    las = [torch.tensor([math.log(0.1)], device=dev, requires_grad=True) for _ in range(E)]
    al_opts = [torch.optim.Adam([la], lr=1e-4, betas=(0.5, 0.999)) for la in las]
    return agent, target, buf, c_opt, a_opt, e_opt, las, al_opts


def calls(E, N, M, weights, dev):
    agent, target, buf, c_opt, a_opt, e_opt, las, al_opts = setup(E, N, dev)
    aug = augmentations.AugmentationSequence([augmentations.IdentityAug(B)])
    state = {}

    def critic():
        logs, state["rds"] = learning.critic_update(
            buffer=buf, agent=agent, target_agent=target, critic_optimizer=c_opt, encoder_optimizer=e_opt, log_alphas=las,
            batch_size=B, gamma=0.99, critic_clip=None, encoder_clip=None, target_critic_ensemble_n=M,
            weighted_bellman_temp=20.0 if weights else None, weight_type="sunrise" if weights else None, pop=False,
            augmenter=aug, encoder_lambda=0.0, random_process=None, noise_clip=None, aug_mix=0.0, discrete=True)
        for ac, tc in zip(agent.critics, target.critics):
            lu.soft_update(tc, ac, 0.005)
        return logs

    def step():
        critic()
        learning.online_actor_update(buffer=buf, agent=agent, pop=False, actor_optimizer=a_opt, log_alphas=las,
                                     batch_size=B, clip=None, random_process=None, noise_clip=None, augmenter=aug,
                                     aug_mix=0.0, premade_replay_dicts=state["rds"], per=False, discrete=True)
        learning.alpha_update(buffer=buf, agent=agent, optimizers=al_opts, batch_size=B, log_alphas=las, augmenter=aug,
                              aug_mix=0.0, target_entropy=-math.log(1.0 / A) * 0.98, premade_replay_dicts=state["rds"],
                              discrete=True)

    return critic, step


def timed(fn, steps, warmup, sync_group):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if sync_group:
        dist.barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) * 1e3 / steps


def workload(name, rank, world, dev, args):
    if name == "critics":
        E, Ng, M, weights = 1, 10, 2, False
        lo, hi = parallel.enable_critic_sharding(Ng)
        E_loc, N_loc = 1, hi - lo
    else:
        E, Ng, M, weights = 4, 2, 2, True
        lo, hi = parallel.enable_member_sharding(E)
        E_loc, N_loc = hi - lo, Ng
    res = {}
    for what in ("critic", "step"):
        critic, step = calls(E_loc, N_loc, M, weights, dev)
        res[f"sharded_us_per_{what}"] = round(timed(critic if what == "critic" else step, args.steps, args.warmup, True), 2)
    exchange = parallel.exchange_name()
    parallel.disable()
    dist.barrier()
    if rank == 0:   # the same workload unsharded on one GPU, in the same run
        for what in ("critic", "step"):
            critic, step = calls(E, Ng, M, weights, dev)
            res[f"one_gpu_us_per_{what}"] = round(timed(critic if what == "critic" else step, args.steps, args.warmup,
                                                        False), 2)
    dist.barrier()
    shape = dict(N=Ng, M=M, E=1) if name == "critics" else dict(E=E, N=Ng, weights="sunrise")
    return dict(workload=name, gpus=world, **shape, S=S, H=H, A=A, B=B, steps=args.steps, warmup=args.warmup,
                card=card(), exchange=exchange, **res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=30)
    ap.add_argument("--workloads", default="critics,members")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file (rank 0)")
    args = ap.parse_args()
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", rank)))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    for name in args.workloads.split(","):
        if name == "members" and world > 4:
            continue   # 4 members over at most 4 ranks
        line = workload(name, rank, world, dev, args)
        if rank == 0:
            print(json.dumps(line), flush=True)
            if args.out:
                with open(args.out, "a") as f:
                    f.write(json.dumps(line) + "\n")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""SAC-Discrete step (SURVEY 8f N4) timed on the device: critic_update(discrete=True) + Polyak every second step +
online_actor_update + alpha_update, CUDA events around K steps.  Atari-like head sizes: 64 features, H = 256, 18 actions,
2 critics, B = 256.  One run, one shape, four execution models:

    eager      the drop-in calls, eager launches, logs read back every step
    auto       the same calls under graphed.enable_auto_graphs() (critic and actor updates replay graphs), logs read back
               every step
    utd        a block of --utd critic updates + Polyak every second one inside lu.pipelined_updates(), captured as ONE
               GraphedCall; time per update
    step_graph the full step (critic + Polyak/2 + actor + alpha) as one GraphedCall (two steps per capture, one with the
               Polyak step); time per step

plus kernel launches per eager step (a separate torch.profiler run) and the card's name and power limit.  With --ref the
UNMODIFIED reference (baseline/_ref) runs the eager step through PyTorch-CUDA on the same GPU, as a labelled comparison.

    python tools/bench_discrete.py --steps 300 --warmup 20 > bench_discrete.json
"""
import argparse
import copy
import json
import math
import os
import subprocess
import sys
from itertools import chain

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

S, A, H, N, M, B, NBUF = 64, 18, 256, 2, 2, 256, 100_000


def build(pkg, device, ours):
    class IdentityEncoder(pkg.nets.Encoder):
        def __init__(self):
            super().__init__()

        @property
        def embedding_dim(self):
            return S

        def forward(self, obs):
            return obs["obs"]

    torch.manual_seed(0)
    agent = pkg.Agent(act_space_size=A, encoder=IdentityEncoder(), actor_network_cls=pkg.nets.mlps.DiscreteActor,
                      critic_network_cls=pkg.nets.mlps.DiscreteCritic, discrete=True, ensemble_size=1, num_critics=N,
                      hidden_size=H, auto_rescale_targets=False)
    agent.to(device)
    target = copy.deepcopy(agent)
    target.to(device)
    rng = np.random.default_rng(0)
    buf = pkg.replay.ReplayBuffer(NBUF + 8, **(dict(device=device) if ours else {}))
    buf.load_experience({"obs": rng.standard_normal((NBUF, S)).astype(np.float32)},
                        rng.integers(0, A, size=(NBUF, 1)).astype(np.float32), rng.standard_normal(NBUF).astype(np.float32),
                        {"obs": rng.standard_normal((NBUF, S)).astype(np.float32)},
                        (rng.uniform(size=NBUF) < 0.05).astype(np.float32))
    critic_opt = torch.optim.Adam(chain(*(c.parameters() for c in agent.critics)), lr=3e-4)
    actor_opt = torch.optim.Adam(chain(*(a.parameters() for a in agent.actors)), lr=3e-4)
    enc_opt = torch.optim.Adam(agent.encoder.parameters(), lr=1e-4)
    la = torch.Tensor([math.log(0.1)]).to(device)
    la.requires_grad = True
    alpha_opt = torch.optim.Adam([la], lr=1e-4, betas=(0.5, 0.999))
    aug = pkg.augmentations.AugmentationSequence([pkg.augmentations.IdentityAug(B)])
    te = -math.log(1.0 / A) * 0.98
    L, lu = pkg.learning, pkg.learning_utils

    def critic(k):
        logs, rds = L.critic_update(
            buffer=buf, agent=agent, target_agent=target, critic_optimizer=critic_opt, encoder_optimizer=enc_opt,
            log_alphas=[la], batch_size=B, gamma=0.99, critic_clip=None, encoder_clip=None, target_critic_ensemble_n=M,
            weighted_bellman_temp=None, weight_type=None, pop=False, augmenter=aug, encoder_lambda=0.0, aug_mix=0.0,
            discrete=True, random_process=None, noise_clip=None, per=False, update_priorities=False, dr3_coeff=0.0)
        if k % 2 == 0:
            for ac, tc in zip(agent.critics, target.critics):
                lu.soft_update(tc, ac, 0.005)
        return logs, rds

    def step(k, read=True):
        logs, rds = critic(k)
        alogs = L.online_actor_update(
            buffer=buf, agent=agent, pop=False, actor_optimizer=actor_opt, log_alphas=[la], batch_size=B, clip=None,
            random_process=None, noise_clip=None, augmenter=aug, aug_mix=0.0, premade_replay_dicts=rds, per=False,
            discrete=True, use_baseline=False)
        L.alpha_update(buffer=buf, agent=agent, optimizers=[alpha_opt], batch_size=B, log_alphas=[la], augmenter=aug,
                       aug_mix=0.0, target_entropy=te, premade_replay_dicts=rds, discrete=True)
        if read:   # (not while a graph is being captured: the logs are read back after each replay)
            return float(logs["losses/critic_overall_loss"]), float(alogs["losses/actor_pg_loss"])
        return logs, alogs

    step.critic = critic
    return step


def timed(step, steps, warmup):
    for k in range(warmup):
        step(k)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(steps):
        out = step(k)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, out


def launches_per_step(step, steps=4):
    """Kernel launches of `steps` eager steps, from torch.profiler (CUDA activities), per step."""
    from torch.profiler import ProfilerActivity, profile

    for k in range(2):
        step(k)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for k in range(steps):
            step(k)
        torch.cuda.synchronize()
    kernels = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
               and not e.name.startswith(("Memcpy", "Memset", "[memory]"))]
    return len(kernels) / steps


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:   # noqa: BLE001 -- the card's name still comes from the runtime
        q = f"{torch.cuda.get_device_name(0)}, power limit unknown"
    return q


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--utd", type=int, default=8)
    ap.add_argument("--ref", action="store_true")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    import super_sac_b200 as ssb
    from super_sac_b200 import graphed, learning_utils as lu

    ms, out = timed(build(ssb, dev, True), args.steps, args.warmup)

    # (a) the same drop-in calls, replayed from graphs from the third call on
    graphed.enable_auto_graphs(True)
    try:
        ms_auto, _ = timed(build(ssb, dev, True), args.steps, args.warmup)
    finally:
        graphed.enable_auto_graphs(False)

    # (b) a UTD block of critic updates (+ Polyak every second) inside lu.pipelined_updates(), one graph
    step = build(ssb, dev, True)

    def utd_block():
        with lu.pipelined_updates():
            for k in range(args.utd):
                logs, _ = step.critic(k)
        return logs

    g_utd = graphed.GraphedCall(utd_block, warmup=2)
    ms_utd, _ = timed(lambda k: g_utd.replay(), max(1, args.steps // args.utd), 3)
    ms_utd /= args.utd
    utd_logs = g_utd.logs()

    # (c) the full step as one graph (two steps: with and without the Polyak step)
    step = build(ssb, dev, True)

    def two_steps():
        step(0, read=False)
        return step(1, read=False)

    g_step = graphed.GraphedCall(two_steps, warmup=2)
    ms_graph, _ = timed(lambda k: g_step.replay(), max(1, args.steps // 2), 3)
    ms_graph /= 2

    try:
        n_launch = launches_per_step(build(ssb, dev, True))
    except Exception as e:   # noqa: BLE001 -- the timings above stand without the count
        n_launch = f"not measured: {e!r}"
    line = {"metric": "sac_discrete_steps_per_sec", "unit": "steps/s", "value": 1e3 / ms, "ms_per_step": ms,
            "config": {"workload": f"SAC-Discrete step (critic + Polyak/2 + actor + alpha), S={S} H={H} A={A} N={N} B={B}",
                       "mode": "eager launches, logs read back every step"},
            "auto_graphs": {"ms_per_step": ms_auto, "value": 1e3 / ms_auto,
                            "mode": "drop-in calls under enable_auto_graphs(), logs read back every step"},
            "utd_block": {"us_per_update": 1e3 * ms_utd, "updates_per_block": args.utd,
                          "mode": "critic updates + Polyak/2 inside pipelined_updates(), one GraphedCall per block",
                          "last_loss": float(utd_logs["losses/critic_overall_loss"])},
            "step_graph": {"ms_per_step": ms_graph, "value": 1e3 / ms_graph,
                           "mode": "critic + Polyak/2 + actor + alpha as one GraphedCall"},
            "eager_kernel_launches_per_step": n_launch,
            "fused_forward": bool(ssb._lib.lib().get_fused_forward()),
            "card": card(),
            "steps": args.steps, "warmup": args.warmup, "dtype": "f32", "last_losses": out}
    if args.ref:
        from baseline import ref_import

        if ref_import.available():
            ref = ref_import.import_reference(device="cuda")
            rms, rout = timed(build(ref, "cuda", False), max(20, args.steps // 6), 5)
            line["reference_on_this_gpu_pytorch_cuda"] = {"ms_per_step": rms, "value": 1e3 / rms, "last_losses": rout}
    print(json.dumps(line))

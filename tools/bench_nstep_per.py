#!/usr/bin/env python
"""Prioritised replay over the frame-deduplicated n-step ring vs the classic prioritised ReplayBuffer, at the DrQv2 (C4)
shape: 3 stacked 3x84x84 uint8 frames, 6-dim actions, B = 512, 3-step returns.  Prints one JSON object:

* device events around ``sample_move_and_augment(per=True)`` (Drqv2Aug on every row, Philox draws) on both buffers, which
  hold the same n-step tuples (the classic one is fed the reference's deque tuples as they complete), and the uniform
  draw of the n-step ring for comparison;
* wall time per ``push`` of the n-step ring with ``prioritized`` on and off, in steady state (the ring is full, so every
  push evicts), the timed loop ending in a device synchronise;
* device bytes per transition of both layouts, computed from shapes;
* the card's name and power limit, read in the same run.

The sampled rings (20 000 transitions: 0.42 GB of frames for the n-step ring, 2.5 GB for the classic one) are far larger
than the 126 MB L2, so the gathers read HBM.

    python tools/bench_nstep_per.py > nstep_per.json
"""
import argparse
import json
import os
import subprocess
import sys
import time
from collections import deque

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

K, C, HW, A, B, N_STEP, GAMMA, EP_LEN = 3, 3, 84, 6, 512, 3, 0.99, 1000


class Stream:
    """Deterministic one-step pixel transitions: a cycle of 64 random frames, episodes of EP_LEN steps."""

    def __init__(self, seed=0):
        rng = np.random.default_rng(seed)
        self.pool = rng.integers(0, 256, (64, C, HW, HW), dtype=np.uint8)
        self.act = rng.uniform(-1, 1, (64, A)).astype(np.float32)
        self.rew = rng.standard_normal(64)
        self._stacks = {}

    def stack(self, t):
        key = t if t < K else K + t % 64
        if key not in self._stacks:
            self._stacks[key] = {"pixels": np.concatenate([self.pool[max(t - j, 0) % 64] for j in range(K - 1, -1, -1)], 0)}
        return self._stacks[key]

    def step(self, i):
        t = i % EP_LEN
        last = t == EP_LEN - 1
        return self.stack(t), self.act[i % 64], float(self.rew[i % 64]), self.stack(t + 1), False, last


def nstep_buffer(ssb, size, prioritized):
    return ssb.replay.NStepReplayBuffer(size, n_step=N_STEP, gamma=GAMMA, frame_stack=K, device="cuda", prioritized=prioritized)


def fill(nb, cb, stream, n):
    """n one-step transitions into the n-step ring; the reference's deque tuples into the classic buffer as they complete."""
    dq = deque([], maxlen=N_STEP)
    done = True
    for i in range(n):
        s, a, r, s1, term, over = stream.step(i)
        nb.push(s, a, r, s1, term, terminate_traj=over)
        if cb is None:
            continue
        if done:
            dq.clear()
        dq.append((s, a, r, s1, term))
        done = over
        if len(dq) == N_STEP:
            s0, a0, R, s_n, d = dq.popleft()
            for j, tr in enumerate(dq):
                R += (GAMMA ** (j + 1)) * tr[2]
                s_n, d = tr[3], tr[4]
            cb.push(s0, a0, R, s_n, d)


def time_sampling(lu, buf, augm, per, iters, warmup):
    for _ in range(warmup):
        lu.sample_move_and_augment(buffer=buf, batch_size=B, augmenter=augm, aug_mix=1.0, per=per)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        lu.sample_move_and_augment(buffer=buf, batch_size=B, augmenter=augm, aug_mix=1.0, per=per)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters


def time_pushes(ssb, stream, prioritized, size, n_fill, n_timed):
    nb = nstep_buffer(ssb, size, prioritized)
    fill(nb, None, stream, n_fill)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(n_fill, n_fill + n_timed):
        s, a, r, s1, term, over = stream.step(i)
        nb.push(s, a, r, s1, term, terminate_traj=over)
    torch.cuda.synchronize()
    assert nb._v_tail > 0
    return (time.perf_counter() - t0) * 1e6 / n_timed


def tree_bytes(size):
    cap2 = 1
    while cap2 < size:
        cap2 *= 2
    return 2 * 2 * cap2 * 8 / size   # float64 sum + min trees of 2 * cap2 nodes, per transition


def card():
    out = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        out["nvidia_smi"] = q
    except Exception as e:   # (reported, not fatal: the timings stand with the device name)
        out["nvidia_smi"] = f"unavailable: {e}"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=20_000)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--push-size", type=int, default=4096)
    ap.add_argument("--pushes", type=int, default=2000)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_nstep_per.py measures on the GPU; no CUDA device found")
    import super_sac_b200 as ssb
    from super_sac_b200 import augmentations, learning_utils as lu

    ssb.manual_seed(0)
    torch.manual_seed(0)
    stream = Stream()
    size = args.size
    nb = nstep_buffer(ssb, size, True)
    cb = ssb.replay.ReplayBuffer(size, device="cuda")
    fill(nb, cb, stream, size)
    assert nb._v_tail == 0 and len(nb) == len(cb)
    augm = augmentations.AugmentationSequence([augmentations.Drqv2Aug(B)], keys=["pixels"])
    res = dict(shape=dict(frame_stack=K, frame=[C, HW, HW], action_dim=A, batch=B, n_step=N_STEP, ring=size,
                          transitions=len(nb)),
               card=card())
    samp = {}
    for rep in range(2):   # alternate the arms: the spread between repetitions is part of the result
        samp.setdefault("nstep_per_us", []).append(time_sampling(lu, nb, augm, True, args.iters, args.warmup))
        samp.setdefault("classic_per_us", []).append(time_sampling(lu, cb, augm, True, args.iters, args.warmup))
        samp.setdefault("nstep_uniform_us", []).append(time_sampling(lu, nb, augm, False, args.iters, args.warmup))
    res["sample_move_and_augment_per_call"] = samp
    del nb, cb
    torch.cuda.empty_cache()
    pushes = {}
    for rep in range(2):
        for pr in (True, False):
            key = "prioritized_us" if pr else "uniform_us"
            pushes.setdefault(key, []).append(time_pushes(ssb, stream, pr, args.push_size, args.push_size + 500, args.pushes))
    res["push_wall_time_per_push"] = pushes
    frame = C * HW * HW
    nb_small = nstep_buffer(ssb, size, True)
    fill(nb_small, None, stream, 8)
    res["device_bytes_per_transition"] = dict(
        nstep_ring=nb_small.bytes_per_transition() + tree_bytes(size),
        nstep_ring_of_which_trees=tree_bytes(size),
        classic=2 * K * frame + 4 * A + 4 + 1 + tree_bytes(size))
    print(json.dumps(res))


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Time the batch-sharded update (parallel.enable_batch_sharding) against the plain single-GPU update, one rank per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node W --master-addr 127.0.0.1 --master-port 29561 \
        tools/bench_batch_sharded.py [--steps 50] [--out profiles/x.json]

For drqv2 (C4: pixels, B = 512) and redq (C2: B = 256): ms per update (critic + Polyak + actor, one CUDA graph replayed,
CUDA events), the sharded update over the W ranks next to the plain update on rank 0's GPU in the same run; and the
all-reduce alone (parallel.all_reduce_flat_) at 16.8 MB (the C4 critic and encoder gradients): time and bytes per second
per rank ((W - 1) / W of the buffer read and written over NVLink).  Rank 0 prints one JSON line with the card's name and
power limit, read in the same call."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "tools")):
    if _p not in sys.path:
        sys.path.insert(0, _p)
import torch
import torch.distributed as dist

import benchlib as bl
import super_sac_b200 as ssb
from super_sac_b200 import _rng, graphed, parallel


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def graph_ms(fn, steps, sync_group):
    g = graphed.GraphedCall(fn, warmup=3)
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    if sync_group:
        dist.barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        g.replay()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / steps


def update_ms(name, dev, sharded, steps, overrides):
    w = bl.Workload(ssb, name, dev, seed=3, buffer_size=overrides.get("buffer"), fill_on_device=True)
    src = _rng.PhiloxSource(3)
    _rng.set_source(src)

    def step():
        _, rds = w.critic_update()
        w.polyak()
        w.actor_and_alpha(rds)

    if sharded:
        parallel.enable_batch_sharding()
    try:
        return graph_ms(step, steps, sharded)
    finally:
        parallel.disable()


def allreduce_ms(dev, n, steps):
    parallel.enable_batch_sharding()
    try:
        t = torch.randn(n, device=dev)
        return graph_ms(lambda: parallel.all_reduce_flat_(t, site="bench"), steps, True)
    finally:
        parallel.disable()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev, world, rank = torch.device("cuda", local), dist.get_world_size(), dist.get_rank()
    res = dict(world=world, card=card(), steps=args.steps, configs={})
    for name, ov in (("drqv2", dict(buffer=20_000)), ("redq", dict(buffer=100_000))):
        plain = update_ms(name, dev, False, args.steps, ov) if rank == 0 else None
        dist.barrier()
        shard = update_ms(name, dev, True, args.steps, ov)
        res["configs"][name] = dict(B=bl.CONFIGS[name]["B"], plain_ms=plain, sharded_ms=shard,
                                    speedup=None if plain is None else plain / shard)
    n = 16_800_000 // 4
    ms = allreduce_ms(dev, n, args.steps)
    moved = 2 * 4 * n * (world - 1) / world   # read from and written to the peers, per rank
    res["allreduce"] = dict(bytes=4 * n, ms=ms, nvlink_bytes_per_s_per_rank=moved / (ms * 1e-3) if world > 1 else None)
    res["exchange"] = parallel.exchange_name()
    if rank == 0:
        line = json.dumps(res)
        print(line, flush=True)
        if args.out:
            with open(args.out, "w") as f:
                f.write(line + "\n")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()

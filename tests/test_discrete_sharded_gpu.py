"""Sharded SAC-Discrete ensembles on two GPUs (run with -m gpu): tools/sharded_discrete_check.py under torchrun with two
ranks must match the single-GPU discrete update -- critics sharded (N = 3 and 10, DR3 + clip + PopArt, priority refresh),
offline filtered BC, members sharded (E = 3, sunrise weights), and a sharded pipelined UTD block, eager and captured.
Skipped below two devices; the host logic is covered on CPU by tests/test_discrete_sharded_gloo.py."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu


def test_sharded_discrete_updates_equal_single_gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(root, "tools", "sharded_discrete_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    for r in (0, 1):
        for what in ("critics N=3", "critics N=10", "critics, offline", "members", "pipelined block"):
            assert f"[rank {r}] sharded discrete {what}" in res.stdout, (what, res.stdout[-3000:])

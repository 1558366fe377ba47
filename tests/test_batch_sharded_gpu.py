"""Batch sharding on the GPU (run with -m gpu).

- ssac_peer_allreduce on a world of one rank, called straight through the C ABI over plain device memory: the result is
  the input bit for bit (a sum of one contribution) at 1, 3, 4097 and 2^22 + 5 floats, from aligned and unaligned
  sources, back to back and inside a captured CUDA graph.
- tools/batch_sharded_check.py under torchrun with one rank: batch-sharded updates (critic + Polyak + actor +
  temperature at the sac / redq state shapes and the drqv2 pixel shape at B = 64) are bit-identical to plain updates,
  eager and captured.
- the same script with 2 ranks, and with 4 where the node has them (skipped below two devices): the sharded update
  matches the single-GPU one at rtol 1e-4 and the replicas stay bitwise identical.
The host logic is covered on CPU by tests/test_batch_sharded_gloo.py."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _allreduce_world1(src, dst, buf, sig, epoch, ticket, ptrs, sptrs):
    from super_sac_b200 import _lib

    n = src.numel()
    cap = (4 * n + 15) // 16 * 16
    _lib.lib().peer_allreduce(src.data_ptr(), dst.data_ptr(), n, buf.data_ptr(), cap, ptrs.data_ptr(), sig.data_ptr(),
                              sptrs.data_ptr(), 0, 1, epoch.data_ptr(), ticket.data_ptr(), _lib.stream_ptr())


@pytest.mark.parametrize("n", [1, 3, 4097, 2**22 + 5])
def test_peer_allreduce_world1_is_exact(n):
    import super_sac_b200  # noqa: F401

    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(n)
    cap = (4 * n + 15) // 16 * 16
    buf = torch.zeros(4 * cap, dtype=torch.uint8, device=dev)
    sig = torch.zeros(128, dtype=torch.int32, device=dev)
    epoch = torch.zeros(1, dtype=torch.int32, device=dev)
    ticket = torch.zeros(2, dtype=torch.int32, device=dev)
    tables = (torch.tensor([buf.data_ptr()], dtype=torch.int64, device=dev),
              torch.tensor([sig.data_ptr()], dtype=torch.int64, device=dev))
    store = torch.randn(n + 1, generator=g, device=dev)
    for call, src in enumerate((store[:n], store[1:], store[:n] * 3)):   # aligned, unaligned, back to back
        dst = torch.full((n + 1,), float("nan"), device=dev)[1:] if call == 1 else torch.empty(n, device=dev)
        _allreduce_world1(src, dst, buf, sig, epoch, ticket, *tables)
        torch.cuda.synchronize()
        assert torch.equal(dst, src), f"call {call}"
    assert int(epoch.item()) == 3 and ticket.tolist() == [0, 0]
    # in place, captured, replayed twice
    x = torch.randn(n, generator=g, device=dev)
    t = torch.empty(n, device=dev)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        t.copy_(x)
        _allreduce_world1(t, t, buf, sig, epoch, ticket, *tables)
    for _ in range(2):
        t.zero_()
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(t, x)
    assert int(epoch.item()) == 5


def _torchrun(nproc, port, *extra):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc), "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tools", "batch_sharded_check.py"), *extra]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=1500)
    assert res.returncode == 0, res.stdout[-4000:] + res.stderr[-4000:]
    for r in range(nproc):
        assert f"[rank {r}] batch-sharded check: ok" in res.stdout, res.stdout[-4000:]
    return res.stdout


def test_batch_sharded_world1_bit_identical():
    out = _torchrun(1, 29547)
    for what in ("updates sac", "updates redq", "updates drqv2 B=64", "captured sac", "captured drqv2 B=64"):
        assert f"[rank 0] batch-sharded {what}" in out, what


@pytest.mark.parametrize("world", [2, 4])
def test_batch_sharded_equals_single_gpu(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    _torchrun(world, 29548 + world, *(["--c4-baseline"] if world == 2 else []))

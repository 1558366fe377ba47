#!/usr/bin/env python
"""Timing of the row-local forward (impl 3 of ssac_mlp_forward) against the tensor-core forward (one JSON line each)."""
import json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch
import benchlib as bl
import super_sac_b200 as ssb
from super_sac_b200 import _lib

dev = torch.device("cuda", 0)
W = bl.Workload(ssb, "redq", dev, buffer_size=10000)
target = W.target
S, A, B = 17, 6, 256
X1 = torch.randn(B, S + A, device=dev)
L = _lib.lib()
for G in (1, 2, 3, 10):
    q = torch.empty(G, B, 1, device=dev)
    ca = target._critic_arena
    for impl in (3, 2):
        def f():
            W1, b1, W2, b2, W3, b3 = ca.ptrs(0)
            L.mlp_forward(W1, b1, W2, b2, W3, b3, None, G, ca.D, ca.H, 1, X1.data_ptr(), S + A, 0, B, None if impl == 3 else h1.data_ptr(),
                          None if impl == 3 else h2.data_ptr(), 0, q.data_ptr(), impl, _lib.stream_ptr())
        h1 = torch.empty(G, B, 256, device=dev); h2 = torch.empty_like(h1)
        ms = bl.graph_time(f, per=10, iters=20)
        print(json.dumps({"what": f"critic forward G={G} B=256", "impl": impl, "us": ms * 1e3}), flush=True)

"""SAC-Discrete under the single-kernel forward and CUDA graphs (run with -m gpu on a B200).

1. The single-kernel forward at the discrete shapes (first-layer width 33..64 = two k-chunks, 17..32 outputs) against a
   float64 forward and against the layered path: plain outputs, a net_index subset, kept h1 / h2, operands at the end of
   their allocation.
2. The BASELINE-size discrete update sequence against the oracle with the single-kernel forward on and off.
3. ``graphed.enable_auto_graphs()``: discrete critic / actor updates replayed from graphs give the eager run's bits;
   PER and priority updates stay eager.
4. A UTD block of discrete critic updates inside ``lu.pipelined_updates()`` (eager and captured) gives the sequential
   schedule's bits.
"""
import contextlib
import copy
import math
import os
import subprocess
import sys
from itertools import chain

import numpy as np
import pytest
import torch

if __name__ == "__main__":   # the allocation-tail check below runs this file as a script
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import golden_util as gu

pytestmark = pytest.mark.gpu


def _forward64(W1, b1, W2, b2, W3, b3, x):
    h1 = torch.relu(x @ W1.T + b1)
    h2 = torch.relu(h1 @ W2.T + b2)
    return h1, h2, h2 @ W3.T + b3


def _arena(G, D, H, O, seed):
    from super_sac_b200 import _arena

    ar = _arena.MLPArena(G, D, H, O, "cuda")
    gen = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n, fan_in in (("W1", D), ("b1", D), ("W2", H), ("b2", H), ("W3", H), ("b3", H)):
            ar.p[n].copy_((torch.rand(ar.p[n].shape, generator=gen) * 2 - 1) / math.sqrt(fan_in))
    return ar


def _run(ar, G, x, ldx, B, fused, keep, net_index=None):
    import super_sac_b200 as ssb
    from super_sac_b200 import _ops

    ssb.set_fused_forward(fused)
    try:
        h1 = torch.full((G, B, ar.H), float("nan"), device="cuda")
        h2 = torch.full_like(h1, float("nan"))
        y = torch.full((G, B, ar.O), float("nan"), device="cuda")
        _ops.mlp_forward(ar, 0, G, x, B, h1, h2, y, ldx=ldx, net_index=net_index, keep_hidden=keep)
        torch.cuda.synchronize()
    finally:
        ssb.set_fused_forward(True)
    return h1, h2, y


# (D, O, H, B, G, ldx - D): first-layer widths 33 / 50 / 64, 17 / 18 / 32 outputs, H 64 / 256, B 1 / 100 / 256 / 1024, the
# 16-byte-aligned vector loads (ldx = D, D % 4 == 0) and the scalar ones (the packed s|a rows of a discrete batch: ldx = D + 1)
FWD_CASES = [
    (33, 17, 64, 1, 1, 0), (50, 18, 256, 100, 3, 1), (64, 18, 256, 256, 2, 1), (64, 32, 256, 1024, 10, 0),
    (64, 32, 64, 256, 10, 0), (33, 32, 256, 1024, 4, 1), (50, 17, 64, 1024, 2, 0), (64, 18, 256, 1, 10, 0),
    (33, 18, 256, 100, 10, 1), (64, 17, 256, 256, 1, 0),
]


@pytest.mark.parametrize("D,O,H,B,G,pad", FWD_CASES, ids=[f"D{c[0]}-O{c[1]}-H{c[2]}-B{c[3]}-G{c[4]}" for c in FWD_CASES])
def test_wide_fused_forward_matches_float64_and_layered(D, O, H, B, G, pad):
    ar = _arena(G, D, H, O, seed=D * 1000 + O * 10 + G)
    ldx = D + pad
    gen = torch.Generator().manual_seed(B + D)
    xs = torch.randn(B, ldx, generator=gen)
    x = xs.cuda()
    h1f, _, yf = _run(ar, G, x, ldx, B, fused=True, keep=False)
    # keep_hidden = 0 leaves h1 untouched on the single-kernel path only: proof that this shape takes it
    assert torch.isnan(h1f).all(), "the single-kernel forward was not taken"
    _, _, yl = _run(ar, G, x, ldx, B, fused=False, keep=False)
    x64 = xs[:, :D].double()
    for g in range(G):
        want = _forward64(*(ar.p[n][g].double().cpu() for n in ("W1", "b1", "W2", "b2", "W3", "b3")), x64)[2]
        scale = float(want.abs().max())
        gu.assert_close(yf[g].cpu().numpy(), want.numpy(), 1e-4, 1e-5 * scale, f"fused y[{g}] vs float64")
        gu.assert_close(yl[g].cpu().numpy(), yf[g].cpu().numpy(), 1e-4, 1e-5 * scale, f"layered y[{g}] vs fused")


@pytest.mark.parametrize("D,O,H,B", [(64, 18, 256, 256), (40, 32, 128, 300)])
def test_wide_fused_forward_net_subset_and_kept_activations(D, O, H, B):
    """net_index (the REDQ-style target subset) and keep_hidden (h1 / h2 for the backward) at the discrete shapes.  h1 /
    h2 come from two correct fp32 forwards: a pre-activation within rounding of zero may land on either side of the ReLU
    (DESIGN 4), so they are compared with an absolute tolerance scaled to the activations."""
    G, M = 6, 3
    ar = _arena(G, D, H, O, seed=7 + D)
    gen = torch.Generator().manual_seed(3)
    xs = torch.randn(B, D, generator=gen)
    x = xs.cuda()
    sub = [4, 1, 5]
    ni = torch.tensor(sub, dtype=torch.int32, device="cuda")
    _, _, ys = _run(ar, M, x, D, B, fused=True, keep=False, net_index=ni)
    for j, g in enumerate(sub):
        want = _forward64(*(ar.p[n][g].double().cpu() for n in ("W1", "b1", "W2", "b2", "W3", "b3")), xs.double())[2]
        gu.assert_close(ys[j].cpu().numpy(), want.numpy(), 1e-4, 1e-5 * float(want.abs().max()), f"subset y[{j}]")
    for net_index, GG in ((None, G), (ni, M)):
        h1f, h2f, yf = _run(ar, GG, x, D, B, fused=True, keep=True, net_index=net_index)
        h1l, h2l, yl = _run(ar, GG, x, D, B, fused=False, keep=True, net_index=net_index)
        for name, a, b in (("h1", h1f, h1l), ("h2", h2f, h2l), ("y", yf, yl)):
            assert not torch.isnan(a).any(), f"{name} not fully written"
            gu.assert_close(a.cpu().numpy(), b.cpu().numpy(), 1e-4, 1e-5 * float(b.abs().max()), f"kept {name}")


@pytest.mark.parametrize("which", ["arena_tail", "h_tail"])
def test_wide_fused_forward_operands_at_allocation_tail(which):
    """Weights / kept activations that end at the last byte of their cudaMalloc block (as
    test_cuda_kernels.test_tma_operands_at_allocation_tail, at the discrete shape): this file run as a script, in a
    process where every tensor is its own allocation."""
    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ, PYTORCH_NO_CUDA_MEMORY_CACHING="1")
    out = subprocess.run([sys.executable, os.path.abspath(__file__), which], env=env, capture_output=True, text=True,
                         timeout=300, cwd=here)
    assert out.returncode == 0 and f"ok {which}" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]


def _tail_check(which):
    from super_sac_b200 import _ops

    G, D, H, O, B = 2, 64, 256, 18, 200
    ar = _arena(G, D, H, O, seed=1)
    n = ar.numel
    big = torch.zeros(8 << 20, dtype=torch.uint8, device="cuda")
    x = torch.randn(B, D, device="cuda")
    h1 = torch.empty(G, B, H, device="cuda")
    h2 = torch.empty_like(h1)
    y = torch.empty(G, B, O, device="cuda")
    ni = torch.tensor([1, 0], dtype=torch.int32, device="cuda")
    _ops.mlp_forward(ar, 0, G, x, B, h1, h2, y, ldx=D, net_index=ni, keep_hidden=True)
    torch.cuda.synchronize()
    want = y.clone()
    if which == "arena_tail":
        flat = big.view(torch.float32)[-n:]
        flat.copy_(ar.flat)
        ar.flat = flat
        ar._make_views()
    else:
        hb = big.view(torch.float32)[-2 * G * B * H:]
        h1, h2 = hb[: G * B * H].view(G, B, H), hb[G * B * H:].view(G, B, H)
    for keep in (False, True):
        y.zero_()
        _ops.mlp_forward(ar, 0, G, x, B, h1, h2, y, ldx=D, net_index=ni, keep_hidden=keep)
        torch.cuda.synchronize()
        assert torch.allclose(y, want, rtol=1e-5, atol=1e-6), (which, keep, float((y - want).abs().max()))
    print("ok", which)


@pytest.mark.parametrize("fused", [True, False], ids=["fused", "layered"])
def test_discrete_baseline_size_update_with_and_without_fused_forward(fused):
    """The 3-update SAC-Discrete sequence at H = 256 / B = 256 / A = 18 / 64 features against the oracle, with every
    actor and critic forward through the single-kernel path (fused) or the layered one."""
    import super_sac_b200 as ssb
    import test_discrete_parity as tdp

    ssb.set_fused_forward(fused)
    try:
        tdp.test_discrete_update_baseline_size_matches_oracle()
    finally:
        ssb.set_fused_forward(True)


# ------------------------------------------------------------------------------------------------ auto graphs
class _PixelEnc:
    def __new__(cls):
        from super_sac_b200 import nets
        from super_sac_b200.nets import cnns

        class Enc(nets.Encoder):
            def __init__(self):
                super().__init__()
                self.net = cnns.BigPixelEncoder((3, 20, 20), 12)

            @property
            def embedding_dim(self):
                return 12

            def forward(self, obs_dict):
                return self.net(obs_dict["pixels"])

        return Enc()


def _discrete_setup(case, seed=3):
    """Agent, target, buffer, optimisers and update arguments of one configuration, identically seeded."""
    import cuda_util as cu
    import super_sac_b200 as ssb
    from super_sac_b200 import augmentations, nets

    ssb.manual_seed(seed)
    torch.manual_seed(seed)
    A, N, H, B, S = 18, 2, 64, 64, 24
    E = 2 if case == "sunrise" else 1
    pixels = case == "pixels"
    if pixels:
        A, N, H, B = 4, 2, 32, 16
    enc = _PixelEnc() if pixels else cu.IdentityEncoder(S)
    agent = ssb.Agent(act_space_size=A, encoder=enc, actor_network_cls=nets.mlps.DiscreteActor,
                      critic_network_cls=nets.mlps.DiscreteCritic, discrete=True, ensemble_size=E, num_critics=N,
                      hidden_size=H, auto_rescale_targets=(case == "popart"))
    agent.to("cuda")
    target = copy.deepcopy(agent)
    target.to("cuda")
    rng = np.random.default_rng(seed)
    n = 512
    if pixels:
        obs = lambda: {"pixels": rng.integers(0, 256, (n, 3, 20, 20), dtype=np.uint8)}   # noqa: E731
    else:
        obs = lambda: {"obs": rng.standard_normal((n, S)).astype(np.float32)}   # noqa: E731
    buf = ssb.replay.ReplayBuffer(n + 8, device="cuda")
    buf.load_experience(obs(), rng.integers(0, A, size=(n, 1)).astype(np.float32), rng.standard_normal(n).astype(np.float32),
                        obs(), (rng.uniform(size=n) < 0.1).astype(np.float32))
    c_opt = torch.optim.Adam(chain(*(c.parameters() for c in agent.critics)), lr=3e-4)
    a_opt = torch.optim.Adam(chain(*(a.parameters() for a in agent.actors)), lr=3e-4)
    e_opt = torch.optim.Adam(agent.encoder.parameters(), lr=1e-3)
    las = []
    for _ in range(E):
        la = torch.tensor([math.log(0.1)], device="cuda", requires_grad=True)
        las.append(la)
    al_opts = [torch.optim.Adam([la], lr=1e-4, betas=(0.5, 0.999)) for la in las]
    aug = augmentations.AugmentationSequence([augmentations.Drqv2Aug(B) if pixels else augmentations.IdentityAug(B)])
    kw = dict(buffer=buf, agent=agent, target_agent=target, critic_optimizer=c_opt, encoder_optimizer=e_opt, log_alphas=las,
              batch_size=B, gamma=0.99, critic_clip=None, encoder_clip=None, target_critic_ensemble_n=N,
              weighted_bellman_temp=None, weight_type=None, pop=False, augmenter=aug, encoder_lambda=0.0,
              random_process=None, noise_clip=None, aug_mix=1.0 if pixels else 0.0, discrete=True, per=False,
              update_priorities=False, dr3_coeff=0.0)
    if case == "popart":
        kw["pop"] = True
    if case == "dr3_clip":
        kw.update(dr3_coeff=0.1, critic_clip=0.5)
    if case == "sunrise":
        kw.update(weight_type="sunrise", weighted_bellman_temp=20.0)
    if case == "pixels":
        kw.update(encoder_clip=5.0)
    if case == "per":
        kw.update(per=True, update_priorities=True)
    te = -math.log(1.0 / A) * 0.98
    return dict(agent=agent, target=target, buf=buf, c_opt=c_opt, a_opt=a_opt, e_opt=e_opt, las=las, al_opts=al_opts,
                aug=aug, kw=kw, te=te, E=E, B=B)


def _discrete_steps(st, steps):
    """critic + Polyak every second step + actor + temperature, through the drop-in entry points."""
    from super_sac_b200 import learning, learning_utils as lu

    kw, agent, target = st["kw"], st["agent"], st["target"]
    all_logs = []
    for k in range(steps):
        logs, rds = learning.critic_update(**kw)
        if k % 2 == 0:
            for ac, tc in zip(agent.critics, target.critics):
                lu.soft_update(tc, ac, 0.005)
        alogs = learning.online_actor_update(
            buffer=st["buf"], agent=agent, pop=kw["pop"], actor_optimizer=st["a_opt"], log_alphas=st["las"],
            batch_size=st["B"], clip=None, random_process=None, noise_clip=None, augmenter=st["aug"], aug_mix=kw["aug_mix"],
            premade_replay_dicts=rds, per=False, discrete=True, use_baseline=False)
        llogs = learning.alpha_update(buffer=st["buf"], agent=agent, optimizers=st["al_opts"], batch_size=st["B"],
                                      log_alphas=st["las"], augmenter=st["aug"], aug_mix=kw["aug_mix"],
                                      target_entropy=st["te"], premade_replay_dicts=rds, discrete=True)
        all_logs.append((dict(logs), dict(alogs), dict(llogs)))
    torch.cuda.synchronize()
    return all_logs


def _state(st):
    agent, target = st["agent"], st["target"]
    out = {"critics": agent._critic_arena.flat, "actors": agent._actor_arena.flat, "target": target._critic_arena.flat}
    for name, opt in (("c", st["c_opt"]), ("a", st["a_opt"])):
        fa = opt._ssac_flat_adam
        out[f"{name}_m"], out[f"{name}_v"], out[f"{name}_step"] = fa.m, fa.v, fa.ctl[:1]
    for i, la in enumerate(st["las"]):
        out[f"log_alpha{i}"] = la.detach()
    for i, p in enumerate(agent.popart):
        if p:
            out[f"popart{i}"] = torch.cat([p.mu, p.nu, p.w, p.b])
    if any(q.requires_grad for q in agent.encoder.parameters()):
        for j, q in enumerate(agent.encoder.parameters()):
            out[f"enc{j}"] = q.detach()
        for j, q in enumerate(target.encoder.parameters()):
            out[f"tenc{j}"] = q.detach()
    return {k: v.detach().clone().cpu() for k, v in out.items()}


@pytest.mark.parametrize("case", ["popart", "dr3_clip", "sunrise", "pixels"])
def test_discrete_auto_graphs_equal_eager(case):
    """Two identically seeded runs of K = 7 steps, eager and under enable_auto_graphs() (calls 3..K of the critic and
    actor updates replay captured graphs): parameters, target parameters, Adam moments and steps and log_alpha identical,
    the same log keys.  The logged scalars are block sums in atomic order (entropy bonus, gradient norms), which differs
    in the last bit between two eager runs as well: they, and the parameters of the clipped case (the clip factor divides
    by such a sum; the actor reads those critics), are compared within fp32 rounding."""
    import random

    from super_sac_b200 import graphed

    K = 7
    runs = []
    for auto in (False, True):
        random.seed(0)
        st = _discrete_setup(case)
        graphed.enable_auto_graphs(auto)
        try:
            logs = _discrete_steps(st, K)
            captured = sorted(k[0] for k, e in graphed._auto["cache"].items() if any(sl.graph is not None for sl in e.slots))
        finally:
            graphed.enable_auto_graphs(False)
        assert captured == (["actor", "critic"] if auto else []), captured
        assert st["c_opt"]._ssac_flat_adam.steps == K and st["a_opt"]._ssac_flat_adam.steps == K
        assert st["buf"].total_sample_calls == K * st["E"]
        if case == "pixels":
            assert float(st["e_opt"].state[st["agent"].encoder.net.conv2.weight]["step"]) == K
        runs.append((_state(st), logs))
    (s0, l0), (s1, l1) = runs
    assert s0.keys() == s1.keys()
    for k in s0:
        if case == "dr3_clip":   # post-Adam parameters: an atol tied to the learning rate, as the parity tests use
            gu.assert_close(s1[k].numpy(), s0[k].numpy(), 1e-4, 3e-4 * 0.01, f"{case}: {k}")
        else:
            assert torch.equal(s0[k], s1[k]), f"{case}: {k} differs"
    _same_logs(l0, l1, skip_random=st["E"] > 1)


def _same_logs(l0, l1, skip_random=False):
    for t, (a, b) in enumerate(zip(l0, l1)):
        for part_a, part_b in zip(a, b):
            assert part_a.keys() == part_b.keys()
            for key in part_a:
                if skip_random and t >= 2 and "random" in key:
                    continue   # the logged member of an ensemble is a host-side random.choice, frozen at capture
                gu.assert_close(float(part_b[key]), float(part_a[key]), 1e-5, 1e-7, f"step {t} log {key}")


def test_discrete_per_and_priority_updates_stay_eager():
    """per=True / update_priorities=True: nothing is captured, and the results are the eager ones."""
    import random

    from super_sac_b200 import graphed

    runs = []
    for auto in (False, True):
        random.seed(0)
        st = _discrete_setup("per")
        graphed.enable_auto_graphs(auto)
        try:
            logs = _discrete_steps(st, 5)
            captured = [k[0] for k, e in graphed._auto["cache"].items() if any(sl.graph is not None for sl in e.slots)]
        finally:
            graphed.enable_auto_graphs(False)
        assert captured == []
        runs.append((_state(st), logs, st["buf"]._it_sum.detach().clone().cpu()))
    (s0, l0, t0), (s1, l1, t1) = runs
    for k in s0:
        assert torch.equal(s0[k], s1[k]), k
    assert torch.equal(t0, t1)
    _same_logs(l0, l1)


# ------------------------------------------------------------------------------------------------ pipelined UTD block
@pytest.mark.parametrize("captured", [False, True], ids=["eager", "graph"])
def test_discrete_pipelined_update_block_equals_sequential(captured):
    """lu.pipelined_updates() with discrete critic updates: 8 updates, Polyak every second, then an actor and a temperature
    update, as the UTD loop runs them.  The target side of update k+1 runs on the front stream next to update k's backward
    and Adam; the result must be the sequential schedule's, bit for bit."""
    from super_sac_b200 import graphed, learning, learning_utils as lu

    def build():
        st = _discrete_setup("plain", seed=9)
        st["kw"].update(batch_size=256)
        st["B"] = 256
        from super_sac_b200 import augmentations

        st["aug"] = st["kw"]["augmenter"] = augmentations.AugmentationSequence([augmentations.IdentityAug(256)])
        agent, target, kw = st["agent"], st["target"], st["kw"]

        def block(pipelined):
            ctx = lu.pipelined_updates() if pipelined else contextlib.nullcontext()
            with ctx:
                for k in range(8):
                    logs, rds = learning._critic_update_impl(**kw)
                    if k % 2 == 0:
                        for ac, tc in zip(agent.critics, target.critics):
                            lu.soft_update(tc, ac, 0.005)
                learning._online_actor_update_impl(
                    buffer=st["buf"], agent=agent, pop=False, actor_optimizer=st["a_opt"], log_alphas=st["las"],
                    batch_size=256, clip=None, random_process=None, noise_clip=None, augmenter=st["aug"], aug_mix=0.0,
                    premade_replay_dicts=rds, per=False, discrete=True)
                learning.alpha_update(buffer=st["buf"], agent=agent, optimizers=st["al_opts"], batch_size=256,
                                      log_alphas=st["las"], augmenter=st["aug"], aug_mix=0.0, target_entropy=st["te"],
                                      premade_replay_dicts=rds, discrete=True)
            return logs

        return st, block

    st0, block0 = build()
    for _ in range(5):
        l0 = block0(False)
    l0 = dict(l0.fetch(keep=True)) if hasattr(l0, "fetch") else dict(l0)
    st1, block1 = build()
    if captured:
        g = graphed.GraphedCall(lambda: block1(True), warmup=2)   # two eager pipelined blocks, then three replays
        for _ in range(3):
            g.replay()
        l1 = g.logs()
    else:
        for _ in range(5):
            l1 = block1(True)
        l1 = dict(l1.fetch(keep=True)) if hasattr(l1, "fetch") else dict(l1)
    torch.cuda.synchronize()
    assert lu.pipeline() is None
    s0, s1 = _state(st0), _state(st1)
    for k in ("critics", "actors", "target", "log_alpha0"):
        assert torch.equal(s0[k], s1[k]), k
    assert l0.keys() == l1.keys()
    for k in l0:
        gu.assert_close(float(l1[k]), float(l0[k]), 1e-5, 1e-7, f"log {k}")


if __name__ == "__main__":
    _tail_check(sys.argv[1])

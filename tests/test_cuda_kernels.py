"""Kernel-level GPU parity against the CPU oracle (run with -m gpu on a B200), through the C ABI.

Bit-exact: Polyak, replay gather, pixel gather+augment, segment-tree indices.  fp32 tolerance rtol 1e-4 (north_star)
for everything that sums in a different order than the oracle.
"""
import ctypes
import math

import numpy as np
import pytest
import torch

import golden_util as gu
from oracle import aug_oracle as ao
from oracle import replay_oracle as ro
from oracle import update_oracle as uo

pytestmark = pytest.mark.gpu
DEV = "cuda"


def L():
    from super_sac_b200 import _lib

    return _lib.lib()


def S():
    from super_sac_b200 import _lib

    return _lib.stream_ptr()


def dev(x, dtype=None):
    t = torch.as_tensor(np.asarray(x))
    if dtype is not None:
        t = t.to(dtype)
    return t.to(DEV).contiguous()


# ------------------------------------------------------------------------------------------------ Polyak / Adam
@pytest.mark.parametrize("n,off", [(1, 0), (7, 0), (721930, 0), (4097, 1), (2_000_003, 3)])
@pytest.mark.parametrize("tau", [0.005, 0.01, 1.0])
def test_polyak_bit_exact(n, off, tau):
    g = torch.Generator().manual_seed(n)
    t0, s0 = torch.randn(n + off, generator=g), torch.randn(n + off, generator=g)
    want = t0[off:] * (1.0 - tau) + s0[off:] * tau  # the reference's three fp32 ops (learning_utils.py:162)
    t, s = t0.to(DEV), s0.to(DEV)
    L().polyak(t.data_ptr() + 4 * off, s.data_ptr() + 4 * off, n, tau, S())
    assert torch.equal(t[off:].cpu(), want)
    assert torch.equal(t[:off].cpu(), t0[:off])


def test_polyak_multi_bit_exact():
    from super_sac_b200 import learning_utils as lu

    torch.manual_seed(0)
    src = torch.nn.Sequential(torch.nn.Conv2d(3, 8, 3), torch.nn.Linear(10, 33), torch.nn.LayerNorm(7)).to(DEV)
    tgt = torch.nn.Sequential(torch.nn.Conv2d(3, 8, 3), torch.nn.Linear(10, 33), torch.nn.LayerNorm(7)).to(DEV)
    want = [t.detach().cpu() * (1.0 - 0.01) + s.detach().cpu() * 0.01 for t, s in zip(tgt.parameters(), src.parameters())]
    lu.soft_update(tgt, src, 0.01)
    for t, w in zip(tgt.parameters(), want):
        assert torch.equal(t.detach().cpu(), w)
    lu.hard_update(tgt, src)
    for t, s in zip(tgt.parameters(), src.parameters()):
        assert torch.equal(t, s)


@pytest.mark.parametrize("wd,clip", [(0.0, None), (1e-3, None), (0.0, 0.5), (1e-3, 40.0)])
def test_adam_matches_oracle(wd, clip):
    n = 72193
    g = torch.Generator().manual_seed(3)
    p0 = torch.randn(n, generator=g)
    opt = uo.Adam([p0.clone()], lr=3e-4, weight_decay=wd)
    p, m, v = p0.to(DEV), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    ctl = torch.zeros(2, dtype=torch.int32, device=DEV)
    gn = torch.zeros(1, device=DEV)
    for step in range(5):
        grad = torch.randn(n, generator=g) * (10.0 ** (step - 3))
        gd = grad.to(DEV)
        ref_g = grad.clone()
        if clip:
            uo.clip_grad_norm([ref_g], clip)
            L().sumsq(gd.data_ptr(), n, gn.data_ptr(), 0, S())
        opt.step([ref_g])
        L().adam_step(p.data_ptr(), gd.data_ptr(), m.data_ptr(), v.data_ptr(), n, ctl.data_ptr(), 3e-4, 0.9, 0.999, 1e-8, wd,
                      gn.data_ptr() if clip else None, clip or 0.0, 1, S())
        if clip:
            gu.assert_close(gd.cpu().numpy(), ref_g.numpy(), 1e-5, 1e-12, f"clipped grad step {step}")
        gu.assert_close(p.cpu().numpy(), opt.params[0].numpy(), 1e-6, 3e-4 * 1e-3, f"adam params step {step}")
    assert int(ctl[0]) == 5 and int(ctl[1]) == 0
    gu.assert_close(m.cpu().numpy(), opt.m[0].numpy(), 1e-5, 1e-6 * float(opt.m[0].abs().max()), "exp_avg")
    gu.assert_close(v.cpu().numpy(), opt.v[0].numpy(), 1e-5, 1e-6 * float(opt.v[0].abs().max()), "exp_avg_sq")


def test_adam_polyak_fused_equals_separate():
    n = 50001
    g = torch.Generator().manual_seed(5)
    p0, t0, gr = torch.randn(n, generator=g), torch.randn(n, generator=g), torch.randn(n, generator=g)
    outs = []
    for fused in (False, True):
        p, t, gd = p0.to(DEV), t0.to(DEV), gr.to(DEV)
        m, v = torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
        ctl = torch.zeros(2, dtype=torch.int32, device=DEV)
        if fused:
            L().adam_polyak_step(p.data_ptr(), gd.data_ptr(), m.data_ptr(), v.data_ptr(), t.data_ptr(), n, ctl.data_ptr(),
                                 3e-4, 0.9, 0.999, 1e-8, 0.0, None, 0.0, 0, 0.005, S())
        else:
            L().adam_step(p.data_ptr(), gd.data_ptr(), m.data_ptr(), v.data_ptr(), n, ctl.data_ptr(), 3e-4, 0.9, 0.999, 1e-8,
                          0.0, None, 0.0, 0, S())
            L().polyak(t.data_ptr(), p.data_ptr(), n, 0.005, S())
        outs.append((p.cpu(), t.cpu()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


# ------------------------------------------------------------------------------------------------ replay
def test_gather_rows_bit_exact():
    from super_sac_b200 import _ops

    rng = np.random.default_rng(0)
    cap, B = 1000, 256
    s = rng.standard_normal((cap, 17)).astype(np.float32)
    a = rng.uniform(-1, 1, (cap, 6)).astype(np.float32)
    d = (rng.uniform(size=(cap, 1)) < 0.3).astype(np.uint8)
    px = rng.integers(0, 256, (cap, 3, 8, 8), dtype=np.uint8)
    idx = rng.integers(0, cap, B)
    X = torch.zeros((B, 23), device=DEV)
    dd = torch.zeros((B, 1), device=DEV)
    pxo = torch.zeros((B, 3, 8, 8), dtype=torch.uint8, device=DEV)
    pxf = torch.zeros((B, 3, 8, 8), device=DEV)
    ts, ta, td, tp = dev(s), dev(a), dev(d), dev(px)
    _ops.gather_rows([ts, ta, td, tp, tp], [X, X[:, 17:], dd, pxo, pxf], [17, 6, 1, 192, 192], [23, 23, 1, 192, 192],
                     [0, 0, 1, 2, 1], dev(idx), B)
    assert np.array_equal(X.cpu().numpy(), np.concatenate([s[idx], a[idx]], 1))
    assert np.array_equal(dd.cpu().numpy(), d[idx].astype(np.float32))
    assert np.array_equal(pxo.cpu().numpy(), px[idx])
    assert np.array_equal(pxf.cpu().numpy(), px[idx].astype(np.float32))


def test_replay_buffer_matches_golden_ops():
    """Ring writes (single, batched, wrap-around), uniform gather and the PER trees against the reference's own
    outputs (tests/golden/replay_per.npz)."""
    import super_sac_b200 as ssb
    from super_sac_b200 import _rng

    fx = gu.load("replay_per")
    buf = ssb.replay.ReplayBuffer(50, alpha=0.6, beta=0.7, device=DEV)
    for k in range(int(fx["n_ops"])):
        op = gu.sub(fx, f"op{k}")
        if str(op["kind"]) == "push1":
            buf.push({"obs": op["s"]}, op["a"], float(op["r"]), {"obs": op["s1"]}, bool(op["d"]))
        else:
            buf.push({"obs": op["s"]}, op["a"], op["r"], {"obs": op["s1"]}, op["d"], priorities=op["priorities"])
    ap = gu.sub(fx, "after_push")
    st = buf._storage
    assert np.array_equal(st.s_stack["obs"].cpu().numpy(), ap["s"]) and np.array_equal(st.s1_stack["obs"].cpu().numpy(), ap["s1"])
    assert np.array_equal(st.action_stack.cpu().numpy(), ap["a"]) and np.array_equal(st.reward_stack.cpu().numpy(), ap["r"])
    assert np.array_equal(st.done_stack.cpu().numpy(), ap["d"])
    assert st._next_idx == int(ap["next_idx"]) and len(buf) == int(ap["filled"])
    assert np.array_equal(buf._it_sum.cpu().numpy(), ap["sum_tree"]) and np.array_equal(buf._it_min.cpu().numpy(), ap["min_tree"])
    old = _rng.set_source(_rng.ScriptedSource())
    try:
        u = gu.sub(fx, "uniform")
        _rng.source().push("indices", u["idx"])
        (s, a, r, s1, d), idx = buf.sample_uniform(8)
        for got, want in ((s["obs"], u["s"]), (a, u["a"]), (r, u["r"]), (s1["obs"], u["s1"]), (d, u["d"])):
            assert np.array_equal(got.cpu().numpy(), want)
        assert np.array_equal(idx, u["ridx"])
        for t in range(4):
            p = gu.sub(fx, f"per{t}")
            _rng.source().push("uniform01", p["u"])
            (s, a, r, s1, d), w, idxes = buf.sample(16)
            assert np.array_equal(idxes, p["idxes"])  # float64 descent: bit-exact
            gu.assert_close(w.cpu().numpy(), p["weights"], 1e-14, 0.0, "IS weights")
            assert np.array_equal(s["obs"].cpu().numpy(), p["s"]) and np.array_equal(a.cpu().numpy(), p["a"])
            buf.update_priorities(idxes, p["new_priorities"])
            assert np.array_equal(buf._it_sum.cpu().numpy(), p["sum_tree"])
            assert np.array_equal(buf._it_min.cpu().numpy(), p["min_tree"])
            assert buf._max_priority == float(p["max_priority"])
    finally:
        _rng.set_source(old)


def test_per_tree_large_matches_oracle():
    """2^21-leaf trees (BASELINE config 5 size): bulk load + 1024-sample rounds against the numpy restatement."""
    import super_sac_b200 as ssb

    rng = np.random.default_rng(1)
    n, cap = 2_000_000, 1 << 21
    orc = ro.ReplayOracle(cap)
    pr = rng.uniform(0.01, 4.0, n)
    orc.it_sum.set(np.arange(n), pr**0.6)
    orc.it_min.set(np.arange(n), pr**0.6)
    sum_t = torch.zeros(2 * cap, dtype=torch.float64, device=DEV)
    min_t = torch.full((2 * cap,), float("inf"), dtype=torch.float64, device=DEV)
    all_idx, all_val = dev(np.arange(n)), dev(pr**0.6)  # keep the device tensors alive across the async launch
    L().tree_set(sum_t.data_ptr(), min_t.data_ptr(), cap, all_idx.data_ptr(), all_val.data_ptr(), n, S())
    assert np.array_equal(sum_t.cpu().numpy(), orc.it_sum.value) and np.array_equal(min_t.cpu().numpy(), orc.it_min.value)
    for rnd in range(3):
        u = rng.uniform(size=1024)
        total = orc.it_sum.reduce(0, n - 1)
        want = orc.it_sum.find_prefixsum_idx(u * total)
        idx = torch.empty(1024, dtype=torch.int64, device=DEV)
        w = torch.empty(1024, dtype=torch.float64, device=DEV)
        ud = dev(u)
        L().tree_sample(sum_t.data_ptr(), min_t.data_ptr(), cap, n, ud.data_ptr(), 1024, 1.0, idx.data_ptr(), w.data_ptr(), S())
        assert np.array_equal(idx.cpu().numpy(), want)
        newp = rng.uniform(1e-3, 5.0, 1024) ** 0.6
        orc.it_sum.set(want, newp)
        orc.it_min.set(want, newp)
        npd = dev(newp)
        L().tree_set(sum_t.data_ptr(), min_t.data_ptr(), cap, idx.data_ptr(), npd.data_ptr(), 1024, S())
        assert np.array_equal(sum_t.cpu().numpy(), orc.it_sum.value) and np.array_equal(min_t.cpu().numpy(), orc.it_min.value)


def test_tree_set_last_write_wins_on_duplicates():
    """numpy fancy assignment semantics (replay.py:263-277): with repeated leaves the LAST value sticks."""
    rng = np.random.default_rng(3)
    cap = 1 << 12
    for n_leaves, n in ((7, 1024), (200, 1000), (4096, 1024), (1, 33)):
        orc = ro.SegmentTree(cap, np.add, 0.0)
        orc_min = ro.SegmentTree(cap, np.minimum, float("inf"))
        sum_t = torch.zeros(2 * cap, dtype=torch.float64, device=DEV)
        min_t = torch.full((2 * cap,), float("inf"), dtype=torch.float64, device=DEV)
        idx = rng.integers(0, n_leaves, n)
        val = rng.uniform(0.1, 3.0, n)
        orc.set(idx, val)
        orc_min.set(idx, val)
        idx_d, val_d = dev(idx), dev(val)
        L().tree_set(sum_t.data_ptr(), min_t.data_ptr(), cap, idx_d.data_ptr(), val_d.data_ptr(), n, S())
        assert np.array_equal(sum_t.cpu().numpy(), orc.value), (n_leaves, n)
        assert np.array_equal(min_t.cpu().numpy(), orc_min.value), (n_leaves, n)


# ------------------------------------------------------------------------------------------------ pixels
def _aug_call(src, idx, shift, B, C, H, W, pad, mode, aug_rows, noise=None):
    out = torch.empty((B, C, H, W), device=DEV)
    L().gather_aug_u8(src.data_ptr(), out.data_ptr(), idx.data_ptr(), None if shift is None else shift.data_ptr(),
                      None if noise is None else noise.data_ptr(), B, C, H, W, pad, mode, aug_rows, S())
    return out.cpu().numpy()


def test_pixel_gather_aug_matches_golden_reference():
    fx = gu.load("aug_pixels")
    b = gu.sub(fx, "buffer")
    s, s1 = dev(b["s"]), dev(b["s1"])
    _, C, H, W = b["s"].shape
    g = gu.sub(fx, "drqv1")
    B = len(g["idx"])
    idx = dev(g["idx"])
    sh = dev(np.stack([g["w1"], g["h1"]], 1), torch.int32)
    assert np.array_equal(_aug_call(s, idx, sh, B, C, H, W, 4, 2, B), g["o"])     # DrqNoNoiseAug: exact in the reference
    assert np.array_equal(_aug_call(s1, idx, sh, B, C, H, W, 4, 2, B), g["o1"])
    g = gu.sub(fx, "drqv1_noise")
    assert np.array_equal(_aug_call(s, idx, sh, B, C, H, W, 4, 2, B // 2, dev(g["n0"])), g["o"])
    assert np.array_equal(_aug_call(s1, idx, sh, B, C, H, W, 4, 2, B // 2, dev(g["n1"])), g["o1"])
    g = gu.sub(fx, "drqv2")
    sh2 = dev(g["shift"].reshape(B, 2), torch.int32)
    got = _aug_call(s, idx, sh2, B, C, H, W, 4, 1, int(B * 0.75))
    assert np.array_equal(got, ao.mix(b["s"][g["idx"]].astype(np.float32), ao.drq_v2_crop(b["s"][g["idx"]], g["shift"]), 0.75))
    assert np.abs(got - g["o"]).max() <= 4e-3  # vs the reference's bilinear grid_sample (SURVEY F9)
    assert np.array_equal(_aug_call(s, idx, None, B, C, H, W, 4, 0, 0), g["oo"])


def test_rad_crop_matches_golden_reference():
    """RadAug (augmentations.py:129-162) fused into the gather (pad_mode 3) against the reference's own output
    (tests/golden/aug_rad.npz): bit-exact on the 9-channel frame stack; on the 3-channel image cv2's small-channel
    path rounds differently, so there the kernel is bit-exact with the oracle and within 1e-3 (0..255 scale) of cv2."""
    fx = gu.load("aug_rad")
    for tag in ("stack9", "rgb3"):
        g = gu.sub(fx, tag)
        idx, crop, mixv = g["idx"], int(g["crop"]), float(g["mix"])
        B = len(idx)
        _, C, H, W = g["s"].shape
        sh = dev(np.stack([g["w"], g["h"]], 1), torch.int32)
        for key, src in (("o", g["s"]), ("o1", g["s1"])):
            got = _aug_call(dev(src), dev(idx), sh, B, C, H, W, crop, 3, int(B * mixv))
            want = ao.mix(src[idx].astype(np.float32), ao.rad_crop(src[idx], g["h"], g["w"], crop), mixv)
            assert np.array_equal(got, want), f"{tag}/{key}: kernel vs oracle"
            if C > 4:
                assert np.array_equal(got, g[key]), f"{tag}/{key}: kernel vs reference (cv2 generic-channel path)"
            else:
                assert np.abs(got - g[key]).max() <= 1e-3


def test_rad_crop_full_size_and_drop_in():
    """BASELINE config 4 shape (B=512, 9x84x84) through sample_move_and_augment with RadAug(512, crop=16): sampled rows
    against the oracle, un-augmented rows are a pure cast, and the window of a constant image is that constant."""
    import super_sac_b200 as ssb
    from super_sac_b200 import _rng, augmentations, learning_utils as lu

    rng = np.random.default_rng(8)
    cap, B, C, H, W, crop = 1024, 512, 9, 84, 84, 16
    s = rng.integers(0, 256, (cap, C, H, W), dtype=np.uint8)
    s[7] = 131                                     # a constant frame: bilinear interpolation must return it unchanged
    buf = ssb.replay.ReplayBuffer(cap, device=DEV)
    buf.load_experience({"pixels": s}, np.zeros((cap, 2), np.float32), np.zeros(cap, np.float32), {"pixels": s[::-1].copy()},
                        np.zeros(cap, bool))
    idx = rng.integers(0, cap, B)
    idx[3] = 7
    shift = rng.integers(0, crop, (B, 2))
    src = _rng.ScriptedSource()
    old = _rng.set_source(src)
    try:
        src.push("indices", idx).push("shifts", shift.astype(np.int32))
        rd = lu.sample_move_and_augment(buf, B, augmentations.AugmentationSequence([augmentations.RadAug(B, crop=crop)]), 0.75, per=False)
        assert src.empty()
    finally:
        _rng.set_source(old)
    o = rd["primary_batch"][0]["pixels"].cpu().numpy()
    o1 = rd["primary_batch"][3]["pixels"].cpu().numpy()
    k = int(B * 0.75)
    rows = np.array([0, 1, 3, 200, k - 1])
    assert np.array_equal(o[rows], ao.rad_crop(s[idx[rows]], shift[rows, 1], shift[rows, 0], crop))
    assert np.array_equal(o1[rows], ao.rad_crop(s[::-1][idx[rows]], shift[rows, 1], shift[rows, 0], crop))
    assert np.array_equal(o[k:], s[idx[k:]].astype(np.float32))
    assert np.all(o[3] == 131.0)
    assert o.min() >= 0.0 and o.max() <= 255.0


@pytest.mark.parametrize("mode", [1, 2])
def test_pixel_gather_aug_full_size(mode):
    """BASELINE config 4 shape: B=512 of 9x84x84 uint8 frames.  Oracle on a sample of rows + exact properties."""
    rng = np.random.default_rng(2)
    cap, B, C, H, W = 2048, 512, 9, 84, 84
    src = torch.randint(0, 256, (cap, C, H, W), dtype=torch.uint8, device=DEV)
    idx = rng.integers(0, cap, B)
    hi = 9 if mode == 1 else 8
    shift = rng.integers(0, hi, (B, 2))
    aug_rows = 384
    got = _aug_call(src, dev(idx), dev(shift, torch.int32), B, C, H, W, 4, mode, aug_rows)
    rows = np.concatenate([np.arange(0, 8), np.arange(380, 392), np.arange(504, 512)])
    sub = src[dev(idx[rows])].cpu().numpy()
    if mode == 1:
        want = ao.drq_v2_crop(sub, shift[rows])
    else:
        want = ao.drq_v1_crop(sub, shift[rows, 0], shift[rows, 1])
    plain = sub.astype(np.float32)
    for j, rrow in enumerate(rows):
        assert np.array_equal(got[rrow], want[j] if rrow < aug_rows else plain[j])
    # properties over the whole batch: values are uint8-valued; a centre shift (= pad) is the identity
    assert np.array_equal(got, np.round(got)) and got.min() >= 0 and got.max() <= 255
    ident = _aug_call(src, dev(idx), dev(np.full((B, 2), 4), torch.int32), B, C, H, W, 4, mode, B)
    assert np.array_equal(ident, src[dev(idx)].float().cpu().numpy())


# ------------------------------------------------------------------------------------------------ MLP
def _arena_from(stack):
    from super_sac_b200._arena import MLPArena

    ar = MLPArena(stack.G, stack.D, stack.H, stack.O, DEV)
    for n in uo.PARAM_NAMES:
        ar.p[n].copy_(getattr(stack, n).to(DEV))
    return ar


@pytest.fixture
def tma(request):
    """impl 2 has two operand-staging paths (TMA and registers) and, for 2 x 256-class nets, a single-kernel forward
    next to the layered one; run all of them.  param: 1 = TMA + fused forward, 0 = registers, 2 = TMA, layered."""
    mode = int(getattr(request, "param", 1))
    L().set_tma_enabled(int(mode != 0))
    L().set_fused_forward(int(mode == 1))
    yield
    L().set_tma_enabled(1)
    L().set_fused_forward(1)


IMPLS = [pytest.param(1, 1, id="ffma"), pytest.param(2, 1, id="tcgen05-tma"), pytest.param(2, 0, id="tcgen05-regs"),
         pytest.param(2, 2, id="tcgen05-layered")]


@pytest.mark.parametrize("impl,tma", IMPLS, indirect=["tma"])
@pytest.mark.parametrize("G,D,H,O,B", [(10, 23, 256, 1, 256), (3, 5, 33, 3, 17), (2, 67, 1024, 1, 512), (1, 17, 256, 12, 256),
                                       (2, 40, 200, 40, 130), (3, 24, 64, 48, 300)])
def test_mlp_forward_backward_matches_oracle(G, D, H, O, B, impl, tma):
    from super_sac_b200 import _ops

    gen = torch.Generator().manual_seed(G * 1000 + H)
    st = uo.MLPStack(G, D, H, O).random_init(gen)
    ar = _arena_from(st)
    x = torch.randn(B, D, generator=gen)
    dy = torch.randn(G, B, O, generator=gen) / B
    extra = torch.randn(G, B, H, generator=gen)
    xd = x.to(DEV)
    h1 = torch.empty((G, B, H), device=DEV)
    h2 = torch.empty_like(h1)
    y = torch.empty((G, B, O), device=DEV)
    _ops.mlp_forward(ar, 0, G, xd, B, h1, h2, y, impl=impl)
    grads = st.zeros_like()
    dx_want = torch.zeros(G, B, D)
    h1_ref, h2_ref = torch.empty(G, B, H), torch.empty(G, B, H)
    for g in range(G):
        yw, h1w, h2w = uo.mlp_forward(st, g, x)
        scale = float(h2w.abs().max())
        gu.assert_close(y[g].cpu().numpy(), yw.numpy(), 1e-4, 2e-5 * max(1.0, float(yw.abs().max())), f"y[{g}]")
        gu.assert_close(h2[g].cpu().numpy(), h2w.numpy(), 1e-4, 2e-5 * scale, f"h2[{g}]")
        gu.assert_close(h1[g].cpu().numpy(), h1w.numpy(), 1e-4, 2e-5 * float(h1w.abs().max()), f"h1[{g}]")
        h1_ref[g], h2_ref[g] = h1w, h2w
        dx_want[g] = uo.mlp_backward(st, g, x, h1w, h2w, dy[g], grads, dh2_extra=0.25 * extra[g], need_dx=True)
    # the backward is checked on the oracle's activations: a pre-activation within rounding of zero may land on
    # either side of the ReLU in two correct fp32 forwards, which flips a whole gradient row (not a kernel property)
    h1.copy_(h1_ref.to(DEV))
    h2.copy_(h2_ref.to(DEV))
    dx = torch.empty((G, B, D), device=DEV)
    _ops.mlp_backward(ar, 0, G, xd, B, h1, h2, dy.to(DEV), dh2_extra=extra.to(DEV), extra_scale=0.25, want_dw=True,
                      accumulate=False, dx=dx, lddx=D, impl=impl)
    scale = {n: float(getattr(grads, n).abs().max()) for n in uo.PARAM_NAMES}
    for n in uo.PARAM_NAMES:
        gu.assert_close(ar.g[n].cpu().numpy(), getattr(grads, n).numpy(), 1e-4, 1e-5 * scale[n], f"grad {n}")
    gu.assert_close(dx.cpu().numpy(), dx_want.numpy(), 1e-4, 1e-5 * float(dx_want.abs().max()), "dx")
    # accumulate = True adds a second identical pass
    _ops.mlp_backward(ar, 0, G, xd, B, h1, h2, dy.to(DEV), dh2_extra=extra.to(DEV), extra_scale=0.25, want_dw=True,
                      accumulate=True, impl=impl)
    for n in uo.PARAM_NAMES:
        gu.assert_close(ar.g[n].cpu().numpy(), 2 * getattr(grads, n).numpy(), 1e-4, 2e-5 * scale[n], f"accumulated grad {n}")
    # input-gradient-only pass with dy = None is the DR3 second pass
    dx2 = torch.empty((G, B, D), device=DEV)
    _ops.mlp_backward(ar, 0, G, xd, B, h1, h2, None, dh2_extra=extra.to(DEV), extra_scale=1.0, want_dw=False, dx=dx2, lddx=D,
                      impl=impl)
    for g in range(G):
        want = uo.mlp_backward(st, g, x, h1_ref[g], h2_ref[g], torch.zeros(B, O), st.zeros_like(), dh2_extra=extra[g], need_dx=True,
                               need_dw=False)
        gu.assert_close(dx2[g].cpu().numpy(), want.numpy(), 1e-4, 1e-5 * float(want.abs().max()), f"dx-only[{g}]")


@pytest.mark.parametrize("impl,tma", IMPLS, indirect=["tma"])
def test_mlp_subset_and_per_group_inputs(impl, tma):
    from super_sac_b200 import _ops

    gen = torch.Generator().manual_seed(9)
    G, D, H, O, B = 6, 24, 64, 1, 40
    st = uo.MLPStack(G, D, H, O).random_init(gen)
    ar = _arena_from(st)
    # REDQ subset: groups {4, 1} of member starting at net 1, inputs embedded in a wider matrix (ldx > D)
    xw = torch.randn(B, D + 8, generator=gen)
    sub = torch.tensor([4, 1], dtype=torch.int32)
    h1 = torch.empty((2, B, H), device=DEV); h2 = torch.empty_like(h1); y = torch.empty((2, B, O), device=DEV)
    _ops.mlp_forward(ar, 1, 2, xw.to(DEV), B, h1, h2, y, ldx=D + 8, net_index=sub.to(DEV), impl=impl)
    for j, k in enumerate(sub.tolist()):
        gu.assert_close(y[j].cpu().numpy(), uo.mlp_forward(st, 1 + k, xw[:, :D].contiguous())[0].numpy(), 1e-4, 1e-5, f"subset {k}")
    # per-group inputs (x_gs != 0)
    xg = torch.randn(G, B, D, generator=gen)
    h1 = torch.empty((G, B, H), device=DEV); h2 = torch.empty_like(h1); y = torch.empty((G, B, O), device=DEV)
    _ops.mlp_forward(ar, 0, G, xg.to(DEV), B, h1, h2, y, x_gs=B * D, impl=impl)
    for g in range(G):
        gu.assert_close(y[g].cpu().numpy(), uo.mlp_forward(st, g, xg[g])[0].numpy(), 1e-4, 1e-5, f"per-group {g}")


@pytest.mark.parametrize("G,D,H,O,B", [(10, 23, 256, 1, 256), (1, 17, 256, 12, 256), (3, 32, 256, 16, 200), (2, 4, 128, 2, 129),
                                       (4, 9, 96, 1, 64), (2, 23, 32, 6, 1000), (3, 17, 48, 12, 300), (1, 8, 240, 3, 128)])
def test_fused_forward_matches_oracle_and_layered(G, D, H, O, B):
    """The single-kernel forward against the oracle and against the layered launches: ragged batch tiles, narrow and
    full hidden widths, kept and discarded activations."""
    from super_sac_b200 import _ops

    gen = torch.Generator().manual_seed(G * 77 + H + B)
    st = uo.MLPStack(G, D, H, O).random_init(gen)
    ar = _arena_from(st)
    x = torch.randn(B, D, generator=gen).to(DEV)
    out = {}
    for mode in ("fused", "fused-nokeep", "layered"):
        L().set_fused_forward(int(mode != "layered"))
        h1 = torch.full((G, B, H), float("nan"), device=DEV)
        h2 = torch.full((G, B, H), float("nan"), device=DEV)
        y = torch.full((G, B, O), float("nan"), device=DEV)
        _ops.mlp_forward(ar, 0, G, x, B, h1, h2, y, impl=2, keep_hidden=(mode != "fused-nokeep"))
        torch.cuda.synchronize()
        out[mode] = (y.cpu(), h1.cpu(), h2.cpu())
    L().set_fused_forward(1)
    assert torch.isnan(out["fused-nokeep"][1]).all(), "keep_hidden=0 must not spend bandwidth on h1 (fused path not taken?)"
    assert torch.equal(out["fused"][0], out["fused-nokeep"][0])
    for g in range(G):
        yw, h1w, h2w = uo.mlp_forward(st, g, x.cpu())
        for mode in ("fused", "layered"):
            y, h1, h2 = out[mode]
            gu.assert_close(y[g].numpy(), yw.numpy(), 1e-4, 2e-5 * max(1.0, float(yw.abs().max())), f"{mode} y[{g}]")
            gu.assert_close(h1[g].numpy(), h1w.numpy(), 1e-4, 2e-5 * float(h1w.abs().max()), f"{mode} h1[{g}]")
            gu.assert_close(h2[g].numpy(), h2w.numpy(), 1e-4, 2e-5 * float(h2w.abs().max()), f"{mode} h2[{g}]")


@pytest.mark.parametrize("u_async", [False, True], ids=["u-in-order", "u-on-second-stream"])
@pytest.mark.parametrize("G,D,H,B", [(10, 23, 256, 256), (2, 4, 64, 200), (3, 32, 128, 300)])
def test_split_critic_backward_matches_oracle(G, D, H, B, u_async):
    """ssac_mlp_backward_pre / _post (TD-independent chain first, seed applied afterwards) against the oracle's backward
    and against the one-call ssac_mlp_backward."""
    from super_sac_b200 import _ops

    gen = torch.Generator().manual_seed(G * 31 + H + B)
    st = uo.MLPStack(G, D, H, 1).random_init(gen)
    ar = _arena_from(st)
    x = torch.randn(B, D, generator=gen)
    dq = torch.randn(G, B, 1, generator=gen) / B
    grads = st.zeros_like()
    h1_ref, h2_ref = torch.empty(G, B, H), torch.empty(G, B, H)
    for g in range(G):
        _, h1w, h2w = uo.mlp_forward(st, g, x)
        h1_ref[g], h2_ref[g] = h1w, h2w
        uo.mlp_backward(st, g, x, h1w, h2w, dq[g], grads, need_dx=False)
    xd, h1, h2, dqd = x.to(DEV), h1_ref.to(DEV), h2_ref.to(DEV), dq.to(DEV)
    ws = torch.empty(L().mlp_backward_ws(G, B, H), dtype=torch.float32, device=DEV)
    W1, _, W2, _, W3, _ = ar.ptrs(0)
    gW1, gb1, gW2, gb2, gW3, gb3 = ar.ptrs(0, grad=True)
    ar.grad.fill_(float("nan"))
    L().mlp_backward_pre(W2, W3, G, H, B, h1.data_ptr(), h2.data_ptr(), ws.data_ptr(), int(u_async), 2, None)
    L().mlp_backward_post(W3, G, D, H, xd.data_ptr(), D, 0, B, h1.data_ptr(), h2.data_ptr(), dqd.data_ptr(), ws.data_ptr(), gW1, gb1,
                          gW2, gb2, gW3, gb3, 2, None)
    torch.cuda.synchronize()
    split = {n: ar.g[n].cpu().clone() for n in uo.PARAM_NAMES}
    for n in uo.PARAM_NAMES:
        want = getattr(grads, n)
        gu.assert_close(split[n].numpy(), want.numpy(), 1e-4, 1e-5 * float(want.abs().max()), f"split grad {n}")
    _ops.mlp_backward(ar, 0, G, xd, B, h1, h2, dqd, want_dw=True, accumulate=False, impl=2)
    torch.cuda.synchronize()
    for n in ("W2", "b2"):               # identical operands and summation order: bit-identical
        assert torch.equal(ar.g[n].cpu(), split[n]), f"split vs one-call {n}"
    for n in ("W1", "b1", "W3", "b3"):   # dq applied after instead of before the W2 product / another (fixed) summation order
        gu.assert_close(ar.g[n].cpu().numpy(), split[n].numpy(), 1e-4, 2e-6 * float(split[n].abs().max()), f"split vs one-call {n}")


@pytest.mark.parametrize("G,S,A,H,B", [(10, 17, 6, 256, 256), (2, 3, 1, 64, 100), (3, 11, 12, 128, 130)])
def test_action_gradient_through_critics(G, S, A, H, B):
    """ssac_mlp_backward_dact == input-gradient pass of ssac_mlp_backward summed over the nets (and the oracle)."""
    from super_sac_b200 import _ops

    gen = torch.Generator().manual_seed(G * 13 + H + A)
    D = S + A
    st = uo.MLPStack(G, D, H, 1).random_init(gen)
    ar = _arena_from(st)
    x = torch.randn(B, D, generator=gen)
    # arg-min routing: one net per row carries the seed
    dq = torch.zeros(G, B, 1)
    dq[torch.randint(0, G, (B,), generator=gen), torch.arange(B), 0] = -torch.rand(B, generator=gen) / B
    h1_ref, h2_ref = torch.empty(G, B, H), torch.empty(G, B, H)
    want = torch.zeros(B, A)
    for g in range(G):
        _, h1w, h2w = uo.mlp_forward(st, g, x)
        h1_ref[g], h2_ref[g] = h1w, h2w
        dx = uo.mlp_backward(st, g, x, h1w, h2w, dq[g], st.zeros_like(), need_dx=True, need_dw=False)
        want += dx[:, S:]
    xd, h1, h2, dqd = x.to(DEV), h1_ref.to(DEV), h2_ref.to(DEV), dq.to(DEV)
    ws = torch.empty(L().mlp_backward_ws(G, B, H), dtype=torch.float32, device=DEV)
    da = torch.full((B, A), float("nan"), device=DEV)
    W1, _, W2, _, W3, _ = ar.ptrs(0)
    for impl in (1, 2):
        L().mlp_backward_dact(W1, W2, W3, G, D, H, S, A, B, h1.data_ptr(), h2.data_ptr(), dqd.data_ptr(), da.data_ptr(),
                              ws.data_ptr(), impl, None)
        torch.cuda.synchronize()
        gu.assert_close(da.cpu().numpy(), want.numpy(), 1e-4, 1e-5 * float(want.abs().max()), f"da impl {impl}")
    dxg = torch.empty((G, B, D), device=DEV)
    _ops.mlp_backward(ar, 0, G, xd, B, h1, h2, dqd, want_dw=False, dx=dxg, lddx=D, impl=2)
    gu.assert_close(da.cpu().numpy(), dxg.sum(0)[:, S:].cpu().numpy(), 1e-4, 1e-5 * float(want.abs().max()), "da vs dx path")


def test_3xtf32_accuracy_against_float64():
    """The operand split assumes that kind::tf32 TRUNCATES an fp32 operand to its top 19 bits (lo = x - trunc(x) is then
    exactly what the tensor core dropped).  If the hardware rounded instead, elements whose dropped bits exceed half an
    ulp would be off by 2^-11 relative and the error below would be ~100x larger than the fp32-FFMA path's."""
    from super_sac_b200 import _ops

    gen = torch.Generator().manual_seed(21)
    G, D, H, O, B = 4, 23, 256, 1, 256
    st = uo.MLPStack(G, D, H, O).random_init(gen)
    ar = _arena_from(st)
    x = torch.randn(B, D, generator=gen)
    xd = x.to(DEV)
    ref = []
    for g in range(G):   # float64 forward
        W1, b1, W2, b2 = (getattr(st, n)[g].double() for n in ("W1", "b1", "W2", "b2"))
        h1 = torch.relu(x.double() @ W1.T + b1)
        ref.append(torch.relu(h1 @ W2.T + b2))
    ref = torch.stack(ref)
    errs = {}
    for name, impl, fused in (("ffma", 1, 0), ("tcgen05-layered", 2, 0), ("tcgen05-fused", 2, 1)):
        L().set_fused_forward(fused)
        h1 = torch.empty((G, B, H), device=DEV); h2 = torch.empty_like(h1); y = torch.empty((G, B, O), device=DEV)
        _ops.mlp_forward(ar, 0, G, xd, B, h1, h2, y, impl=impl, keep_hidden=True)
        errs[name] = float((h2.double().cpu() - ref).abs().max() / ref.abs().max())
    L().set_fused_forward(1)
    assert errs["ffma"] < 2e-6, errs
    assert errs["tcgen05-layered"] < 1e-5 and errs["tcgen05-fused"] < 1e-5, errs   # rounding hardware would give ~2e-4


# ------------------------------------------------------------------------------------------------ heads / TD / weights
def test_policy_heads_match_oracle():
    gen = torch.Generator().manual_seed(4)
    B, A, lo, hi = 300, 6, -5.0, 2.0
    out = torch.randn(B, 2 * A, generator=gen) * 1.5
    eps = torch.randn(B, A, generator=gen)
    a_w, logp_w, cache = uo.tanh_normal_sample(out, eps, lo, hi)
    od, ed = out.to(DEV), eps.to(DEV)
    X = torch.zeros((B, 17 + A), device=DEV)
    logp = torch.empty(B, device=DEV)
    L().tanh_normal_forward(od.data_ptr(), ed.data_ptr(), B, A, lo, hi, X[:, 17:].data_ptr(), 17 + A, logp.data_ptr(), S())
    gu.assert_close(X[:, 17:].cpu().numpy(), a_w.numpy(), 1e-5, 1e-6, "a")
    gu.assert_close(logp.cpu().numpy(), logp_w[:, 0].numpy(), 1e-4, 1e-4, "logp")
    assert float(X[:, :17].abs().max()) == 0.0
    da = torch.randn(B, A, generator=gen)
    la = torch.tensor([math.log(0.2)])
    dout_w = uo.tanh_normal_sample_backward(cache, da, torch.full((B, 1), 0.2 / B))
    dout = torch.empty((B, 2 * A), device=DEV)
    dad, lad = da.to(DEV), la.to(DEV)
    L().tanh_normal_backward(od.data_ptr(), ed.data_ptr(), B, A, lo, hi, dad.data_ptr(), A, 1.0 / B, lad.data_ptr(),
                             dout.data_ptr(), S())
    gu.assert_close(dout.cpu().numpy(), dout_w.numpy(), 1e-4, 1e-6, "dout")
    # dataset actions (cache miss), incl. |a| > 0.99
    act = (torch.rand(B, A, generator=gen) * 2 - 1) * 1.05
    lp_w, c2 = uo.tanh_normal_logprob_data(out, act.clamp(-1, 1), lo, hi)
    dl = torch.randn(B, 1, generator=gen)
    dw = uo.tanh_normal_logprob_data_backward(c2, dl)
    lp = torch.empty(B, device=DEV)
    dout2 = torch.empty((B, 2 * A), device=DEV)
    actd, dld = act.clamp(-1, 1).to(DEV), dl[:, 0].contiguous().to(DEV)
    L().tanh_normal_logprob(od.data_ptr(), actd.data_ptr(), A, B, A, lo, hi, lp.data_ptr(), dld.data_ptr(), dout2.data_ptr(), S())
    gu.assert_close(lp.cpu().numpy(), lp_w[:, 0].numpy(), 1e-4, 1e-3, "logp(data)")
    gu.assert_close(dout2.cpu().numpy(), dw.numpy(), 2e-4, 1e-3 * float(dw.abs().max()) * 1e-2, "dout(data)")
    # deterministic head + TD3 noise
    o2 = torch.randn(B, A, generator=gen)
    nz = torch.randn(B, A, generator=gen)
    want = uo.gaussian_noise_clamp(torch.tanh(o2), nz, 0.7, 0.3, -1.0, 1.0)
    a2 = torch.empty((B, A), device=DEV); th = torch.empty((B, A), device=DEV)
    o2d, nzd = o2.to(DEV), nz.to(DEV)
    L().det_head_forward(o2d.data_ptr(), None, nzd.data_ptr(), B, A, 0.7, 0.3, a2.data_ptr(), A, th.data_ptr(), S())
    gu.assert_close(a2.cpu().numpy(), want.numpy(), 1e-6, 1e-6, "td3 action")


@pytest.mark.parametrize("use_popart,pop,warm", [(False, False, False), (True, True, False), (True, True, True)])
def test_td_target_matches_oracle(use_popart, pop, warm):
    gen = torch.Generator().manual_seed(6)
    M, B = 2, 256
    q = torch.randn(M, B, generator=gen) * 3
    logp = torch.randn(B, 1, generator=gen)
    r = torch.randn(B, 1, generator=gen)
    d = (torch.rand(B, 1, generator=gen) < 0.1).float()
    la = torch.tensor([math.log(0.1)])
    pa = None
    if use_popart:
        pa = uo.PopArt()
        if warm:
            pa.t, pa.mu, pa.nu, pa.w, pa.b = 1500, torch.tensor([0.3]), torch.tensor([1.7]), torch.tensor([0.9]), torch.tensor([0.1])
    val = q.min(0).values.unsqueeze(1) - la.exp() * logp
    if pa is not None and pop:
        val = pa.forward(val, normalized=False)
    y_w = r + 0.99 * (1.0 - d) * val
    st = ctl = None
    if pa is not None:
        st = torch.cat([pa.mu, pa.nu, pa.w, pa.b]).to(DEV)
        ctl = torch.tensor([pa.t, 0], dtype=torch.int32, device=DEV)
        pa.update_stats(y_w)
        y_w = pa.normalize_values(y_w)
    y = torch.empty(B, device=DEV); logs = torch.zeros(3, device=DEV)
    qd, lpd, lad, rd, dd = q.to(DEV), logp.to(DEV), la.to(DEV), r.to(DEV), d.to(DEV)
    L().td_target(qd.data_ptr(), M, B, lpd.data_ptr(), lad.data_ptr(), rd.data_ptr(),
                  dd.data_ptr(), 0.99, None if st is None else st.data_ptr(), None if ctl is None else ctl.data_ptr(),
                  int(pop), 1e-4, 1000, y.data_ptr(), logs.data_ptr(), S())
    gu.assert_close(y.cpu().numpy(), y_w[:, 0].numpy(), 1e-4, 1e-5, "td target")
    gu.assert_close(logs.cpu().numpy(), [y_w.mean().item(), y_w.std().item(), (la.exp() * logp).mean().item()], 1e-4, 1e-5, "logs")
    if pa is not None:
        gu.assert_close(st.cpu().numpy(), torch.cat([pa.mu, pa.nu, pa.w, pa.b]).numpy(), 1e-5, 1e-7, "popart state")
        assert ctl.cpu().tolist() == [pa.t, int(pa.stable)]


@pytest.mark.parametrize("kind", [0, 1])
def test_backup_weights_match_oracle(kind):
    gen = torch.Generator().manual_seed(8)
    E, N, B, T = 5, 2, 256, 20.0
    q = torch.randn(E, N, B, generator=gen)
    std = q.min(1).values.std(0)
    want = torch.sigmoid(-std * T) + 0.5 if kind == 0 else B * torch.softmax(-std * T, dim=0)
    w = torch.empty(B, device=DEV); logs = torch.zeros(4, device=DEV)
    qd = q.to(DEV)
    L().backup_weights(qd.data_ptr(), E, N, B, T, kind, w.data_ptr(), logs.data_ptr(), S())
    gu.assert_close(w.cpu().numpy(), want.numpy(), 1e-4, 1e-6, "weights")
    gu.assert_close(logs.cpu().numpy(), [want.mean().item(), want.max().item(), want.min().item(), want.std().item()], 1e-4, 1e-6, "logs")


def test_rng_fill_statistics_and_replay_advance():
    from super_sac_b200 import _rng

    src = _rng.PhiloxSource(123)
    idx = torch.empty(1 << 16, dtype=torch.int64, device=DEV)
    nrm = torch.empty(1 << 18, device=DEV)
    sub = torch.empty(4096 * 2, dtype=torch.int32, device=DEV)
    sh = torch.empty(1 << 14, dtype=torch.int32, device=DEV)
    src.fill(DEV, idx=idx, n_filled=1000, normal=nrm, subset=sub, N=10, M=2, shift=sh, shift_range=9)
    i1 = idx.clone()
    assert int(idx.min()) >= 0 and int(idx.max()) < 1000
    cnt = torch.bincount(idx, minlength=1000).float()
    assert abs(float(cnt.mean()) - 65.536) < 1e-3 and float(cnt.std()) < 12
    assert abs(float(nrm.mean())) < 0.01 and abs(float(nrm.std()) - 1.0) < 0.01
    assert abs(float((nrm**4).mean()) - 3.0) < 0.1
    s2 = sub.view(-1, 2)
    assert int(s2.min()) >= 0 and int(s2.max()) < 10 and bool((s2[:, 0] != s2[:, 1]).all())
    pair = torch.bincount(s2[:, 0] * 10 + s2[:, 1], minlength=100).float()
    assert float(pair[pair > 0].min()) > 15  # 90 ordered pairs, ~45 each
    assert int(sh.min()) == 0 and int(sh.max()) == 8
    src.fill(DEV, idx=idx, n_filled=1000)
    assert not torch.equal(idx, i1)  # the offset advanced on the device
    src2 = _rng.PhiloxSource(123)
    j = torch.empty(1 << 16, dtype=torch.int64, device=DEV)
    src2.fill(DEV, idx=j, n_filled=1000)
    assert torch.equal(j, i1)  # same seed, same first draw


@pytest.mark.parametrize("method", ["mean", "max"])
def test_advantage_estimator_mean_and_max(method):
    """agent.adv_estimator(o, a, i) (adv_estimator.py:58-79): A = Q(s,a) - V(s) with V the mean or the max over n = 4
    policy samples, min over the critics, PopArt affine -- against the oracle on the same N(0,1) draws."""
    import twin_util as tw
    from super_sac_b200 import _rng

    E, N, S_, A, H, B = 2, 2, 17, 6, 256, 200
    agent, _, o_agent, _ = tw.make_twins(E, N, S_, A, H, popart=True, seed=9)
    agent.adv_estimator.cont_method = method
    for i, p in enumerate(agent.popart):
        p.w, p.b = 1.5 + i, -0.25
        o_agent.popart[i].w, o_agent.popart[i].b = torch.tensor([1.5 + i]), torch.tensor([-0.25])
    rng = np.random.default_rng(9)
    s = rng.standard_normal((B, S_)).astype(np.float32)
    a = rng.uniform(-1, 1, (B, A)).astype(np.float32)
    eps = [rng.standard_normal((B, A)).astype(np.float32) for _ in range(4)]
    src = _rng.ScriptedSource()
    old = _rng.set_source(src)
    try:
        for e in eps:
            src.push("normal", e)
        got = agent.adv_estimator({"obs": dev(s)}, dev(a), 1)
        assert src.empty()
    finally:
        _rng.set_source(old)
    want = uo.advantage(o_agent, 1, {"obs": torch.as_tensor(s)}, torch.as_tensor(a), [torch.as_tensor(e) for e in eps], method=method)
    gu.assert_close(got.cpu().numpy(), want.numpy(), 1e-4, 2e-5, f"advantage ({method})")


# ------------------------------------------------------------------------------------------------ row-local CUDA-core forwards
def _rand_stack(G, D, H, O, seed):
    return uo.MLPStack(G, D, H, O).random_init(torch.Generator().manual_seed(seed))


@pytest.mark.parametrize("G,D,H,O,B", [(2, 23, 256, 1, 256), (3, 9, 48, 5, 37), (1, 56, 128, 16, 8), (10, 23, 256, 1, 5),
                                        (1, 17, 256, 12, 256), (2, 64, 40, 3, 19)])
def test_rows_forward_matches_oracle(G, D, H, O, B):
    """ssac_mlp_forward impl 3 (ssac_mlp_rows.cu: clusters of 4 CTAs, 8 rows each, exact fp32 on the CUDA cores)."""
    st = _rand_stack(G, D, H, O, seed=G * 1000 + H)
    x = torch.randn(B, D + 3, generator=torch.Generator().manual_seed(B))   # wider rows than D: exercises ldx
    y = torch.empty(G, B, O, device=DEV)
    xd = x.to(DEV)
    p = {n: getattr(st, n).to(DEV).contiguous() for n in uo.PARAM_NAMES}
    L().mlp_forward(p["W1"].data_ptr(), p["b1"].data_ptr(), p["W2"].data_ptr(), p["b2"].data_ptr(), p["W3"].data_ptr(),
                    p["b3"].data_ptr(), None, G, D, H, O, xd.data_ptr(), D + 3, 0, B, None, None, 0, y.data_ptr(), 3, S())
    want = torch.stack([uo.mlp_forward(st, g, x[:, :D])[0] for g in range(G)], 0)
    gu.assert_close(y.cpu().numpy(), want.numpy(), 1e-5, 2e-6, "rows forward")


@pytest.mark.parametrize("envs", [1, 5])
def test_acting_path_kernels_match_oracle(envs):
    """SURVEY 8f N1: Agent.forward / sample_action (agent.py:204-327) through the kernels at B = num_envs, incl. SUNRISE's
    UCB choice (every actor proposes, every member's critics score every proposal) -- against the oracle on the same draws."""
    import twin_util as tw
    from super_sac_b200 import _rng

    E, N, S_, A, H = 3, 2, 17, 6, 256
    agent, _, o_agent, _ = tw.make_twins(E, N, S_, A, H, seed=21)
    rng = np.random.default_rng(envs)
    s = rng.standard_normal((envs, S_)).astype(np.float32)
    obs = {"obs": s[0] if envs == 1 else s}
    st = torch.as_tensor(s)
    # greedy action: mean over the actors of tanh(mu)
    want = torch.stack([torch.tanh(uo.mlp_forward(o_agent.actors, i, st)[0][:, :A]) for i in range(E)], 0).mean(0).numpy()
    got = agent.forward(obs, num_envs=envs)
    gu.assert_close(got, want[0] if envs == 1 else want, 1e-5, 2e-6, "Agent.forward")
    # UCB exploration
    agent.ucb_bonus = 2.5
    eps = [rng.standard_normal((envs, A)).astype(np.float32) for _ in range(E)]
    src = _rng.ScriptedSource()
    old = _rng.set_source(src)
    try:
        for e in eps:
            src.push("normal", e)
        got = agent.sample_action(obs, num_envs=envs)
        assert src.empty()
    finally:
        _rng.set_source(old)
        agent.ucb_bonus = 0.0
    cands = torch.stack([uo.actor_sample(o_agent, i, st, torch.as_tensor(eps[i]))[0] for i in range(E)], 0)       # [E, envs, A]
    q = torch.stack([torch.stack([o_agent.critic_min(c, st, cands[e]) for e in range(E)], 0) for c in range(E)], 0)  # [Ec, E, envs, 1]
    ucb = (q.mean(0) + 2.5 * q.std(0)).squeeze(-1)
    best = ucb.argmax(0)
    srt = ucb.sort(0, descending=True).values
    assert float((srt[0] - srt[1]).min()) > 1e-4, "test data: UCB scores too close to call"
    want = cands[best, torch.arange(envs)].numpy()
    gu.assert_close(got, want[0] if envs == 1 else want, 1e-5, 2e-6, "UCB sample_action")


@pytest.mark.parametrize("which", ["arena_tail", "h_tail"])
def test_tma_operands_at_allocation_tail(which):
    """TMA operands that end exactly at the end of their cudaMalloc block (regression: the box hanging over the tensor's
    end faulted on B200 although those rows are out of bounds for the tensor map) -- tests/tail_alloc_check.py."""
    import os
    import subprocess
    import sys

    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ, PYTORCH_NO_CUDA_MEMORY_CACHING="1")
    out = subprocess.run([sys.executable, os.path.join(here, "tail_alloc_check.py"), which], env=env, capture_output=True,
                         text=True, timeout=300)
    assert out.returncode == 0 and f"ok {which}" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]

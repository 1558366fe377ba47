"""The update's output-layer epilogues and small kernels, called one by one through the C ABI, against float64.

Each fused entry point is checked twice: its raw output layer (q, out) against a float64 forward with the MLP tolerance of
test_cuda_kernels.py, and every epilogue output against the float64 epilogue evaluated on the kernel's OWN raw output,
with a per-element bound built from fp32 rounding of the operands (a few ulp of their magnitudes).  That bound is tight
enough to catch a wrong constant, a dropped factor or a missing term, which a blanket rtol would let through.

The float64 reference (``ref_*`` below) restates nets/distributions.py:9-15,64-114, learning_utils.py:48-59,298-354 and
learning.py:90-112,222-263,400-408 of the reference; test_float64_reference_matches_oracle pins it to the fp32 oracle on
the CPU.  Every output is NaN-prefilled, neighbouring columns / the element past the end carry a marker value, and the
accumulators start from non-zero values, so that a missed element, a stray write and `=` versus `+=` all show.
"""
import math

import pytest
import torch
import torch.nn.functional as F

import golden_util as gu
from oracle import update_oracle as uo

gpu = pytest.mark.gpu
DEV = "cuda"
U = 2.0 ** -24          # unit roundoff of fp32
MARK = -1234.5          # value of the elements an entry point must not write
LOG2 = math.log(2.0)
LOG_SQRT_2PI = 0.5 * math.log(2.0 * math.pi)


def L():
    from super_sac_b200 import _lib

    return _lib.lib()


def S():
    from super_sac_b200 import _lib

    return _lib.stream_ptr()


def ptr(t):
    return None if t is None else t.data_ptr()


def f64(t):
    return torch.as_tensor(t).detach().cpu().double()


def assert_within(got, want, tol, what):
    """|got - want| <= tol element-wise (a NaN anywhere fails)."""
    got, want = f64(got), f64(want)
    tol = torch.broadcast_to(f64(tol), want.shape)
    assert got.shape == want.shape, f"{what}: shape {tuple(got.shape)} vs {tuple(want.shape)}"
    err = (got - want).abs()
    ok = err <= tol
    if not bool(ok.all()):
        i = int(torch.argmax(torch.where(ok, torch.zeros_like(err), torch.nan_to_num(err - tol, nan=math.inf))))
        g, w, e, t = got.flatten()[i].item(), want.flatten()[i].item(), err.flatten()[i].item(), tol.flatten()[i].item()
        raise AssertionError(f"{what}: {int((~ok).sum())} of {ok.numel()} elements off; worst at flat index {i}: "
                             f"got {g!r} want {w!r} (|err| {e:.3e}, bound {t:.3e})")


def ulp(t):
    """Spacing of the fp32 numbers at |t| (normal range)."""
    t = f64(t).abs().clamp_min(2.0 ** -126)
    return torch.exp2(torch.floor(torch.log2(t)) - 23)


def sum_bound(terms, term_err=0.0):
    """Error bound of an fp32 sum of `terms` in any order: the terms' own errors plus (n - 1) u sum|term|."""
    terms = f64(terms).flatten()
    return float(f64(term_err).sum()) + max(terms.numel() - 1, 1) * U * float(terms.abs().sum())


def assert_mlp_close(got, want, what):
    """The MLP tolerance of test_cuda_kernels.py (rtol 1e-4, atol scaled by the output magnitude)."""
    want = f64(want)
    gu.assert_close(f64(got).numpy(), want.numpy(), 1e-4, 2e-5 * max(1.0, float(want.abs().max())), what)


def profiled_kernels(fn):
    """Names of the CUDA kernels `fn` launched (torch.profiler, CUDA activity)."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = {e.name for e in prof.events()}
    assert any("kernel" in n for n in names), f"the profiler recorded no kernel: {sorted(names)}"
    return names


def assert_ran(names, kernel, absent=()):
    assert any(kernel in n for n in names), f"{kernel} did not run; kernels: {sorted(names)}"
    for k in absent:
        assert not any(k in n for n in names), f"{k} ran; kernels: {sorted(names)}"


# ------------------------------------------------------------------------------------------------ float64 reference
def ref_mlp(st, g, x):
    """One net of an MLPStack in float64: (h1, h2, out)."""
    W1, b1, W2, b2, W3, b3 = (getattr(st, n)[g].double() for n in uo.PARAM_NAMES)
    h1 = torch.relu(f64(x) @ W1.T + b1)
    h2 = torch.relu(h1 @ W2.T + b2)
    return h1, h2, h2 @ W3.T + b3


def ref_tanh_normal(out, eps, lo, hi):
    """nets/distributions.py:9-15,64-104: a = tanh(mu + eps std), logp = sum_j Normal.log_prob(x_j) - log|d tanh(x_j)|,
    std = exp(lo + (hi - lo) (tanh(raw) + 1) / 2).  Returns a [B,A], logp [B] and an error bound for each of them when
    the same arithmetic runs in fp32 on fp32 operands (tanhf / expf 2 ulp, logf / log1pf 1 ulp, CUDA C guide)."""
    out, eps = f64(out), f64(eps)
    A = out.shape[-1] // 2
    mu, raw = out[:, :A], out[:, A:]
    log_std = lo + 0.5 * (hi - lo) * (torch.tanh(raw) + 1.0)
    sd = log_std.exp()
    x = mu + eps * sd
    a = torch.tanh(x)
    sp = F.softplus(-2.0 * x)
    ladj = 2.0 * (LOG2 - x - sp)
    q = (x - mu) ** 2 / (2.0 * sd * sd)
    term = (0.0 - ladj) + (-q - log_std - LOG_SQRT_2PI)
    logp = term.sum(-1)
    e_ls = 6 * U * (abs(lo) + abs(hi))                      # log_std
    e_sd = e_ls + 3 * U                                     # relative, std
    e_x = eps.abs() * sd * (e_sd + 2 * U) + 2 * U * (mu.abs() + x.abs())
    e_a = (1.0 - a * a) * e_x + 3 * U
    e_ladj = 2 * e_x + 4 * U * (LOG2 + x.abs() + sp.abs() + 1.0)
    dxm = (x - mu).abs()
    e_q = dxm * (e_x + U * dxm) / (sd * sd) + q * (2 * e_sd + 4 * U)
    e_term = e_ladj + e_q + e_sd + 2 * U * log_std.abs() + 3 * U * (ladj.abs() + q + log_std.abs() + 1.0)
    e_logp = e_term.sum(-1) + A * U * term.abs().sum(-1)
    return a, logp, 2 * e_a, 2 * e_logp


def ref_det_head(out, eps, noise, sigma, clip):
    """Deterministic head (nets/distributions.py:107-114 rsample jitter 1e-4 eps) + TD3 noise (learning_utils.py:48-59):
    a = clamp(tanh(out) [+ 1e-4 eps] + clamp(sigma noise, +-clip), -1 + 1e-6, 1 - 1e-6); clip <= 0: no noise clip;
    no noise: no clamp either.  Returns tanh(out), a and the bound on a."""
    th = torch.tanh(f64(out))
    v = th.clone()
    if eps is not None:
        v = v + 1e-4 * f64(eps)
    nz = torch.zeros_like(th)
    if noise is not None:
        nz = sigma * f64(noise)
        if clip > 0:
            nz = nz.clamp(-clip, clip)
        v = (v + nz).clamp(-1.0 + 1e-6, 1.0 - 1e-6)
    return th, v, 8 * U * (1.0 + nz.abs())


def ref_critic_epilogue(q, y, w, imp, popart, pop, E, n_total):
    """learning.py:90-98,112 on q [N,B]: q' = popw q + popb if pop; td = y - q'; dq = -2 w imp td popw / (B E n_total);
    loss[0] gains sum w imp td^2 / (B E n_total), loss[1] = mean_b td of the last net.  Returns (dq, loss0, loss1) and
    their fp32 error bounds."""
    q, y = f64(q), f64(y)
    N, B = q.shape
    nt = n_total if n_total > 0 else N
    inv = 1.0 / (B * E * nt)
    on = popart is not None and pop
    pw, pb = (float(popart[2]), float(popart[3])) if on else (1.0, 0.0)
    qq = pw * q + pb
    td = y - qq
    ww = (f64(w) if w is not None else torch.ones(B, dtype=torch.float64)) * (f64(imp) if imp is not None else 1.0)
    dq = -2.0 * ww * td * pw * inv
    lt = ww * td * td * inv
    e_td = U * ((pw * q).abs() + qq.abs()) + U * td.abs()
    e_dq = (2.0 * ww * pw * inv) * e_td + 6 * U * dq.abs()
    e_lt = 2.0 * ww * inv * td.abs() * e_td + 5 * U * lt
    return dq, float(lt.sum()), float(td[-1].mean()), e_dq, sum_bound(lt, e_lt), sum_bound(td[-1], e_td[-1]) / B + U * abs(float(td[-1].mean()))


def ref_td_target(qt, logp, alpha, r, d, gamma):
    """learning_utils.py:319-353 without PopArt: y = r + gamma (1 - d) (min_m qt - alpha logp)."""
    v = f64(qt).min(0).values - (alpha * f64(logp) if logp is not None else 0.0)
    return f64(r) + gamma * (1.0 - f64(d)) * v


def ref_adam_scalar(p, g, m, v, t, lr, b1, b2, eps):
    """torch.optim.Adam (_single_tensor_adam, no weight decay) on one scalar, in float64."""
    m = m + (1.0 - b1) * (g - m)
    v = b2 * v + (1.0 - b2) * g * g
    denom = math.sqrt(v) / math.sqrt(1.0 - b2**t) + eps
    return p - (lr / (1.0 - b1**t)) * (m / denom), m, v


def test_float64_reference_matches_oracle():
    """The float64 restatements above against the fp32 oracle on random inputs (CPU)."""
    gen = torch.Generator().manual_seed(11)
    B, A, lo, hi = 64, 5, -5.0, 2.0
    out = torch.randn(B, 2 * A, generator=gen) * 2
    eps = torch.randn(B, A, generator=gen)
    a, logp, _, _ = ref_tanh_normal(out, eps, lo, hi)
    a_o, logp_o, _ = uo.tanh_normal_sample(out, eps, lo, hi)
    gu.assert_close(a.numpy(), a_o.numpy(), 1e-5, 1e-6, "tanh-Normal a")
    gu.assert_close(logp.numpy(), logp_o[:, 0].numpy(), 1e-4, 1e-4, "tanh-Normal logp")
    o2, nz, jit = torch.randn(B, A, generator=gen), torch.randn(B, A, generator=gen), torch.randn(B, A, generator=gen)
    for clip in (0.3, 0.0):
        _, v, _ = ref_det_head(o2, jit, nz, 0.7, clip)
        want = uo.gaussian_noise_clamp(torch.tanh(o2) + 1e-4 * jit, nz, 0.7, clip if clip > 0 else None, -1.0, 1.0)
        gu.assert_close(v.numpy(), want.numpy(), 0.0, 1e-6, f"det head clip {clip}")
    th, v, _ = ref_det_head(o2, None, None, 0.7, 0.3)
    assert torch.equal(th, v)
    # critic loss seed against the oracle's PopArt forward and learning.py's loss / dq
    N, E = 3, 2
    q = torch.randn(N, B, generator=gen)
    y = torch.randn(B, generator=gen)
    w, imp = torch.rand(B, generator=gen) + 0.5, torch.rand(B, generator=gen) + 0.2
    pa = uo.PopArt()
    pa.w, pa.b = torch.tensor([1.7]), torch.tensor([-0.3])
    dq, l0, l1, *_ = ref_critic_epilogue(q, y, w, imp, torch.tensor([0.0, 1.0, 1.7, -0.3]), 1, E, 2 * N)
    td = y - pa.forward(q)
    gu.assert_close(dq.numpy(), (-2.0 / (B * E * 2 * N) * w * imp * td * pa.w).numpy(), 1e-6, 1e-9, "critic dq")
    gu.assert_close(l0, float((w * imp * td * td).mean(1).sum()) / (E * 2 * N), 1e-6, 1e-9, "critic loss")
    gu.assert_close(l1, float(td[-1].mean()), 1e-6, 1e-7, "critic mean td")
    # TD target and the arg-min routing against torch's fp32 min
    M = 4
    qt = torch.randn(M, B, generator=gen)
    qt[2, :7] = qt[0, :7]                                  # ties
    lp, r, d = torch.randn(B, generator=gen), torch.randn(B, generator=gen), (torch.rand(B, generator=gen) < 0.2).float()
    vals, arg = torch.stack(list(qt), 0).min(0)
    gu.assert_close(ref_td_target(qt, lp, 0.2, r, d, 0.99).numpy(), (r + 0.99 * (1 - d) * (vals - 0.2 * lp)).numpy(), 1e-6,
                    1e-6, "td target")
    assert torch.equal(ref_arg_min(qt), arg)
    # Adam on a scalar
    p = torch.tensor([math.log(0.1)])
    opt = uo.Adam([p], lr=1e-2, betas=(0.5, 0.999))
    pr, m, v = float(p), 0.0, 0.0
    for t in range(1, 6):
        g = torch.tensor([0.3 * (-1) ** t + 0.1])
        pr, m, v = ref_adam_scalar(pr, float(g), m, v, t, 1e-2, 0.5, 0.999, 1e-8)
        opt.step([g])
    gu.assert_close(pr, float(opt.params[0]), 1e-6, 1e-7, "adam")
    gu.assert_close([m, v], [float(opt.m[0]), float(opt.v[0])], 1e-6, 1e-7, "adam state")   # |g| ~ 0.3: fp32 rounding


def ref_arg_min(q):
    """The reference's gradient routing: the net torch.stack(..).min(0) picks on the CPU (first of equal minima)."""
    return torch.stack(list(torch.as_tensor(q).float().cpu()), 0).min(0).indices


# ------------------------------------------------------------------------------------------------ paths
PATHS = ("ffma", "tc-fused", "tc-layered", "tc-regs")


@pytest.fixture(params=PATHS)
def path(request):
    """ffma: impl 1; tc-fused: impl 2 with the single-kernel forward and TMA; tc-layered: ssac_set_fused_forward(0);
    tc-regs: ssac_set_tma_enabled(0).  Switches are restored whatever happens."""
    lib = L()
    try:
        lib.set_fused_forward(int(request.param != "tc-layered"))
        lib.set_tma_enabled(int(request.param != "tc-regs"))
        yield request.param
    finally:
        lib.set_fused_forward(1)
        lib.set_tma_enabled(1)


def impl_of(path):
    return 1 if path == "ffma" else 2


def output_kernel(path, D, H, O):
    """The kernel that must compute the output layer and its epilogue (launch_mlp3_fused's range)."""
    fused = path == "tc-fused" and 32 <= H <= 256 and H % 16 == 0 and D <= 64 and O <= 32
    return "mlp3_forward_kernel" if fused else "head_forward_kernel"


def params_dev(st):
    return {n: getattr(st, n).to(DEV).contiguous() for n in uo.PARAM_NAMES}


def wptrs(P):
    return [P[n].data_ptr() for n in uo.PARAM_NAMES]


def nan_with_tail(n, tail=1):
    """n NaN elements followed by `tail` marker elements."""
    t = torch.full((n + tail,), float("nan"), device=DEV)
    t[n:] = MARK
    return t


def assert_tail(t, n, what):
    assert bool((t[n:].cpu() == MARK).all()), f"{what}: written past its end"


# ------------------------------------------------------------------------------------------------ A / B: critic forward + loss
CRITIC_SHAPES = [(2, 23, 256, 256), (10, 23, 256, 1000), (10, 23, 256, 5), (2, 4, 64, 129), (3, 40, 48, 300), (1, 9, 32, 1),
                 (2, 67, 1024, 1024)]
CRITIC_OPTS = ["plain", "weighted-popart", "popart-off", "sharded"]


def critic_call(P, N, D, H, x, ldx, B, h1, h2, q, y, w, imp, pa, pop, E, nt, dq, loss, phase, impl, qt=None, M=0, logp=None,
                la=None, r=None, d=None, gamma=0.99, y_out=None, td_logs=None, raw=False):
    fn = L().critic_forward_loss.raw if raw else L().critic_forward_loss
    return fn(*wptrs(P), N, D, H, ptr(x), ldx, B, ptr(h1), ptr(h2), ptr(q), ptr(y), ptr(w), ptr(imp), ptr(pa), pop, E, nt,
              ptr(dq), ptr(loss), phase, ptr(qt), M, ptr(logp), ptr(la), ptr(r), ptr(d), gamma, ptr(y_out), ptr(td_logs),
              impl, S())


def check_critic_epilogue(q, dq, loss, loss_init, y, w, imp, pa, pop, E, nt, what, loss1_init=None):
    """dq and loss of one call against the float64 epilogue on that call's own q [N,B].  loss1_init None: loss[1] is
    stored, not accumulated."""
    dq_r, l0, l1, e_dq, e_l0, e_l1 = ref_critic_epilogue(q, y, w, imp, pa, pop, E, nt)
    assert_within(dq, dq_r, e_dq, f"{what}: dq")
    lo = f64(loss)
    assert_within(lo[0], loss_init[0] + l0, e_l0 + U * abs(float(lo[0])), f"{what}: loss[0] (+=)")
    base1 = loss_init[1] if loss1_init is None else loss1_init
    assert_within(lo[1], base1 + l1, e_l1 + U * abs(float(lo[1])), f"{what}: loss[1]")


@gpu
@pytest.mark.parametrize("opt", CRITIC_OPTS)
@pytest.mark.parametrize("N,D,H,B", CRITIC_SHAPES)
def test_critic_forward_loss(N, D, H, B, opt, path):
    impl = impl_of(path)
    gen = torch.Generator().manual_seed(N * 7919 + D * 131 + H * 17 + B + CRITIC_OPTS.index(opt))
    st = uo.MLPStack(N, D, H, 1).random_init(gen)
    P = params_dev(st)
    ldx = D + 3                                             # x is a column block of a wider matrix
    X = torch.randn(B, ldx, generator=gen)
    y = torch.randn(B, generator=gen) * 1.5 + 0.3
    w = imp = pa = None
    pop, E, nt = 0, 1, 0
    if opt == "weighted-popart":
        w, imp = torch.rand(B, generator=gen) * 1.5 + 0.25, torch.rand(B, generator=gen) * 0.8 + 0.2
        pa, pop = torch.tensor([0.2, 1.3, 1.7, -0.3]), 1
    elif opt == "popart-off":
        pa = torch.tensor([0.2, 1.3, 1.7, -0.3])
    elif opt == "sharded":
        E, nt = 3, 2 * N
    Xd, yd = X.to(DEV), y.to(DEV)
    wd, impd, pad = (None if t is None else t.to(DEV) for t in (w, imp, pa))
    ref = [ref_mlp(st, g, X[:, :D]) for g in range(N)]
    q_ref = torch.stack([r[2][:, 0] for r in ref])
    init = (0.375, -0.625)

    def run(phase, h1, h2, q, dq, loss):
        critic_call(P, N, D, H, Xd, ldx, B, h1, h2, q, yd, wd, impd, pad, pop, E, nt, dq, loss, phase, impl)

    # phase 0: the whole forward and the loss seed in one call
    h1, h2 = torch.full((N, B, H), float("nan"), device=DEV), torch.full((N, B, H), float("nan"), device=DEV)
    q, dq = nan_with_tail(N * B), nan_with_tail(N * B)
    loss = torch.tensor(init, device=DEV)
    names = profiled_kernels(lambda: run(0, h1, h2, q, dq, loss))
    want = output_kernel(path, D, H, 1)
    assert_ran(names, want, absent=("head_forward_kernel",) if want == "mlp3_forward_kernel" else ("mlp3_forward_kernel",))
    assert_tail(q, N * B, "q")
    assert_tail(dq, N * B, "dq")
    qk = q[: N * B].view(N, B).cpu()
    assert_mlp_close(qk, q_ref, "q")
    for g in range(N):
        assert_mlp_close(h1[g].cpu(), ref[g][0], f"h1[{g}]")
        assert_mlp_close(h2[g].cpu(), ref[g][1], f"h2[{g}]")
    dqk = dq[: N * B].view(N, B).cpu()
    check_critic_epilogue(qk, dqk, loss.cpu(), init, y, w, imp, pa, pop, E, nt, "phase 0")

    # ssac_critic_loss_seed on the q the forward produced: same operations in the same order -> the same dq bits
    dq2 = nan_with_tail(N * B)
    loss2 = torch.tensor(init, device=DEV)
    L().critic_loss_seed(q.data_ptr(), N, B, yd.data_ptr(), ptr(wd), ptr(impd), ptr(pad), pop, E, nt, dq2.data_ptr(),
                         loss2.data_ptr(), S())
    assert_tail(dq2, N * B, "critic_loss_seed dq")
    assert torch.equal(dq2[: N * B].view(N, B).cpu(), dqk), "critic_loss_seed dq != fused epilogue dq"
    check_critic_epilogue(qk, dqk, loss2.cpu(), init, y, w, imp, pa, pop, E, nt, "critic_loss_seed", loss1_init=0.0)

    # phase 1 (hidden layers) then phase 2 (output layer + loss) == phase 0
    h1b, h2b = torch.full((N, B, H), float("nan"), device=DEV), torch.full((N, B, H), float("nan"), device=DEV)
    q3, dq3 = nan_with_tail(N * B), nan_with_tail(N * B)
    loss3 = torch.tensor(init, device=DEV)
    names = profiled_kernels(lambda: (run(1, h1b, h2b, None, None, None), run(2, h1b, h2b, q3, dq3, loss3)))
    assert_ran(names, "head_forward_kernel")
    if want == "mlp3_forward_kernel":
        assert_ran(names, "mlp3_forward_kernel")
    for g in range(N):
        assert_mlp_close(h2b[g].cpu(), ref[g][1], f"phase 1 h2[{g}]")
    q3k = q3[: N * B].view(N, B).cpu()
    assert_mlp_close(q3k, q_ref, "phase 2 q")
    gu.assert_close(q3k.numpy(), qk.numpy(), 1e-4, 2e-5 * max(1.0, float(qk.abs().max())), "phase 1+2 q vs phase 0 q")
    check_critic_epilogue(q3k, dq3[: N * B].view(N, B).cpu(), loss3.cpu(), init, y, w, imp, pa, pop, E, nt, "phase 1+2")
    assert_tail(q3, N * B, "phase 2 q")
    assert_tail(dq3, N * B, "phase 2 dq")


TD_CASES = [  # N, D, H, B, M, with logp, reward mean
    (2, 23, 256, 256, 1, True, 0.0), (2, 23, 256, 256, 2, True, 0.0), (2, 23, 256, 256, 5, False, 0.0),
    (10, 23, 256, 1000, 2, False, 0.0), (10, 23, 256, 1000, 5, True, 0.0), (3, 9, 48, 2, 1, False, 0.0),
    (3, 9, 48, 2, 2, True, 0.0), (2, 23, 256, 256, 2, True, 1000.0), (2, 23, 256, 300, 5, False, 1000.0),
]


@gpu
@pytest.mark.parametrize("N,D,H,B,M,with_logp,r_mean", TD_CASES)
def test_critic_inplace_td_target(N, D, H, B, M, with_logp, r_mean):
    """Phase 2 with qt_dev: the TD target evaluated inside the loss kernel."""
    gen = torch.Generator().manual_seed(N * 101 + B * 7 + M * 3 + int(with_logp) + int(r_mean))
    st = uo.MLPStack(N, D, H, 1).random_init(gen)
    P = params_dev(st)
    X = torch.randn(B, D, generator=gen)
    h2 = torch.stack([ref_mlp(st, g, X)[1] for g in range(N)]).float()
    spread = 0.01 if r_mean else 1.0
    qt = torch.randn(M, B, generator=gen) * 2 * spread
    qt[M - 1, : B // 4] = qt[0, : B // 4]                   # ties between target nets
    logp = torch.randn(B, generator=gen) * spread if with_logp else None
    la = torch.tensor([math.log(0.2)])
    r = r_mean + torch.randn(B, generator=gen) * (0.01 if r_mean else 1.0)
    d = (torch.rand(B, generator=gen) < 0.1).float()
    d[0] = 0.0
    gamma = 0.99
    Xd, h2d, qtd, lad, rd, dd = (t.to(DEV) for t in (X, h2, qt, la, r, d))
    lpd = None if logp is None else logp.to(DEV)
    h1d = torch.zeros((N, B, H), device=DEV)
    y_out = nan_with_tail(B)
    q, dq = nan_with_tail(N * B), nan_with_tail(N * B)
    loss = torch.tensor([0.375, -0.625], device=DEV)
    logs_init = (0.25, 0.5, -0.75, 99.0)
    td_logs = torch.tensor(logs_init, device=DEV)
    critic_call(P, N, D, H, Xd, D, B, h1d, h2d, q, None, None, None, None, 0, 1, 0, dq, loss, 2, 2, qt=qtd, M=M, logp=lpd,
                la=lad, r=rd, d=dd, gamma=gamma, y_out=y_out, td_logs=td_logs)
    # the same inputs through ssac_td_target
    y_td, logs_td = torch.full((B,), float("nan"), device=DEV), torch.zeros(3, device=DEV)
    L().td_target(qtd.data_ptr(), M, B, ptr(lpd), lad.data_ptr(), rd.data_ptr(), dd.data_ptr(), gamma, None, None, 0, 0.0, 0,
                  y_td.data_ptr(), logs_td.data_ptr(), S())
    # phase 2 reading that y
    yk = y_out[:B].clone()
    q2, dq2 = nan_with_tail(N * B), nan_with_tail(N * B)
    loss2 = torch.tensor([0.375, -0.625], device=DEV)
    critic_call(P, N, D, H, Xd, D, B, h1d, h2d, q2, yk, None, None, None, 0, 1, 0, dq2, loss2, 2, 2)
    torch.cuda.synchronize()
    assert_tail(y_out, B, "y_out")
    yk = yk.cpu()
    assert torch.equal(yk, y_td.cpu()), "in-place TD target != ssac_td_target"
    alpha = math.exp(float(la))
    y_ref = ref_td_target(qt, logp, alpha if with_logp else 0.0, r, d, gamma)
    ent = alpha * f64(logp) if with_logp else torch.zeros(B, dtype=torch.float64)
    assert_within(yk, y_ref, 4 * U * (f64(r).abs() + f64(qt).abs().max(0).values + 4 * ent.abs() + yk.abs().double()), "y")
    assert torch.equal(q.cpu(), q2.cpu()) and torch.equal(dq.cpu(), dq2.cpu()), "qt in place vs y read back: dq differs"
    qk = q[: N * B].view(N, B).cpu()
    assert_mlp_close(qk, torch.stack([f64(h2[g]) @ f64(st.W3[g, 0]) + float(st.b3[g, 0]) for g in range(N)]), "q")
    check_critic_epilogue(qk, dq[: N * B].view(N, B).cpu(), loss.cpu(), (0.375, -0.625), yk, None, None, None, 0, 1, 0,
                          "in-place target")
    check_critic_epilogue(qk, dq2[: N * B].view(N, B).cpu(), loss2.cpu(), (0.375, -0.625), yk, None, None, None, 0, 1, 0,
                          "y read back")   # same terms, atomicAdds in another order
    # logged statistics: td_logs[0..2] += {sum (y - c), sum (y - c)^2, sum alpha logp}, td_logs[3] = c = y[0]
    tl = f64(td_logs.cpu())
    c = float(yk[0])
    assert float(tl[3]) == c, "td_logs[3] != y[0]"
    dev_ = f64(yk) - c
    s1, s2, se = float(dev_.sum()), float((dev_ * dev_).sum()), float(ent.sum())
    e1 = sum_bound(dev_) + U * abs(float(tl[0]))
    e2 = sum_bound(dev_ * dev_, 2 * U * dev_ * dev_) + U * abs(float(tl[1]))
    e3 = sum_bound(ent, 4 * U * ent.abs()) + U * abs(float(tl[2]))
    assert_within(tl[0] - logs_init[0], s1, e1, "td_logs[0] (+= sum y - c)")
    assert_within(tl[1] - logs_init[1], s2, e2, "td_logs[1] (+= sum (y - c)^2)")
    assert_within(tl[2] - logs_init[2], se, e3, "td_logs[2] (+= sum alpha logp)")
    # the statistics the update logs from them (learning_utils.py, _fuse_into_loss) against ssac_td_target's two-pass logs
    t1, t2, t3 = float(tl[0]) - logs_init[0], float(tl[1]) - logs_init[1], float(tl[2]) - logs_init[2]
    mean_f = c + t1 / B
    std_f = max((t2 - t1 * t1 / B) / (B - 1), 0.0) ** 0.5
    ent_f = t3 / B
    mean64, std64 = float(f64(yk).mean()), float(f64(yk).std())
    e_std_f = ((e2 + (2 * abs(t1) * e1 + e1 * e1) / B) / (B - 1)) / max(2 * std64, 1e-30) + 1e-12
    assert_within(mean_f, mean64, e1 / B + 1e-12, "mean formed from td_logs")
    assert_within(std_f, std64, 2 * e_std_f, "std formed from td_logs")
    assert_within(ent_f, se / B, e3 / B, "entropy bonus formed from td_logs")
    lg = f64(logs_td.cpu())
    e_m = 16 * U * float(f64(yk).abs().mean())             # ssac_td_target: one fp32 tree sum over the block
    assert_within(lg[0], mean64, e_m, "ssac_td_target mean")
    assert_within(lg[1], std64, e_m * e_m / max(std64, 1e-30) + 16 * U * std64 + 1e-12, "ssac_td_target std")
    assert_within(lg[2], se / B, e3 / B + 16 * U * float(ent.abs().mean()), "ssac_td_target entropy bonus")
    assert_within(mean_f, lg[0], e1 / B + e_m, "formed mean vs ssac_td_target")
    assert_within(std_f, lg[1], 2 * e_std_f + e_m * e_m / max(std64, 1e-30) + 16 * U * std64 + 1e-12,
                  "formed std vs ssac_td_target")


# ------------------------------------------------------------------------------------------------ C: actor forward + head
ACTOR_CASES = [  # A, deterministic, D, H, B, keep_hidden, variant
    (1, False, 17, 256, 256, 0, "plain"),
    (3, False, 11, 64, 37, 1, "saturate"),
    (6, False, 17, 256, 600, 0, "saturate"),
    (8, False, 24, 128, 1, 1, "saturate"),
    (12, False, 40, 256, 256, 0, "saturate"),
    (16, False, 17, 256, 600, 0, "saturate"),
    (6, False, 17, 1024, 600, 0, "saturate"),
    (1, True, 17, 256, 37, 0, "eps+noise-clip"),
    (6, True, 17, 256, 256, 1, "plain"),
    (6, True, 17, 256, 600, 0, "eps"),
    (13, True, 9, 128, 600, 0, "eps+noise-noclip"),
    (16, True, 17, 256, 1, 0, "noise-clip"),
    (6, True, 23, 1024, 600, 0, "eps+noise-noclip"),
]
LO, HI, SIGMA, CLIP = -5.0, 2.0, 0.7, 0.3


def actor_inputs(A, det, D, H, B, variant, seed):
    gen = torch.Generator().manual_seed(seed)
    O = A if det else 2 * A
    st = uo.MLPStack(1, D, H, O).random_init(gen)
    if variant == "saturate":   # |mu + eps std| well past 50 (mu_1 = -mu_0): tanh saturates, softplus(-2x) takes its threshold branch
        st.W3[0, 0] *= 150.0
        st.W3[0, 1], st.b3[0, 1] = -st.W3[0, 0], -st.b3[0, 0]
    X = torch.randn(B, D + 2, generator=gen)
    eps = torch.randn(B, A, generator=gen) if (not det or "eps" in variant) else None
    noise = torch.randn(B, A, generator=gen) * 2 if "noise" in variant else None
    clip = CLIP if "noise-clip" in variant else 0.0
    return st, X, eps, noise, clip


def check_head(det, out, eps, noise, clip, a, logp, tanh_out, what):
    """The epilogue outputs of one call against the float64 head evaluated on that call's own raw output."""
    if det:
        th, v, e_v = ref_det_head(out, eps, noise, SIGMA, clip)
        assert_within(a, v, e_v, f"{what}: a")
        if tanh_out is not None:
            assert_within(tanh_out, th, 2.5 * ulp(th), f"{what}: tanh(out)")   # tanhf: 2 ulp
    else:
        av, lp, e_a, e_lp = ref_tanh_normal(out, eps, LO, HI)
        assert_within(a, av, e_a, f"{what}: a")
        assert_within(logp, lp, e_lp, f"{what}: logp")


@gpu
@pytest.mark.parametrize("A,det,D,H,B,keep,variant", ACTOR_CASES)
def test_actor_forward_sample(A, det, D, H, B, keep, variant, path):
    impl = impl_of(path)
    st, X, eps, noise, clip = actor_inputs(A, det, D, H, B, variant, seed=A * 1000 + D * 10 + H + B + int(det))
    O = A if det else 2 * A
    P = params_dev(st)
    ldx = D + 2
    Xd = X.to(DEV)
    epsd, noised = (None if t is None else t.to(DEV) for t in (eps, noise))
    h1, h2 = torch.full((B, H), float("nan"), device=DEV), torch.full((B, H), float("nan"), device=DEV)
    out = nan_with_tail(B * O)
    col0, lda = 5, A + 8                                    # a is a column block of a wider cat(s, a)-like matrix
    Xa = torch.full((B + 1, lda), MARK, device=DEV)
    Xa[:B, col0:col0 + A] = float("nan")
    logp = None if det else nan_with_tail(B)
    tanh_out = nan_with_tail(B * A) if det else None

    def run():
        L().actor_forward_sample(*wptrs(P), D, H, A, int(det), Xd.data_ptr(), ldx, B, h1.data_ptr(), h2.data_ptr(), keep,
                                 out.data_ptr(), ptr(epsd), ptr(noised), SIGMA, clip, LO, HI, Xa[:, col0:].data_ptr(), lda,
                                 ptr(logp), ptr(tanh_out), impl, S())

    names = profiled_kernels(run)
    want = output_kernel(path, D, H, O)
    assert_ran(names, want, absent=("head_forward_kernel",) if want == "mlp3_forward_kernel" else ("mlp3_forward_kernel",))
    h1_ref, h2_ref, out_ref = ref_mlp(st, 0, X[:, :D])
    if want == "mlp3_forward_kernel" and not keep:
        assert bool(torch.isnan(h1).all()) and bool(torch.isnan(h2).all()), "keep_hidden=0 wrote h1 / h2"
    if keep or want != "mlp3_forward_kernel":
        assert_mlp_close(h1.cpu(), h1_ref, "h1")
        assert_mlp_close(h2.cpu(), h2_ref, "h2")
    assert_tail(out, B * O, "out")
    outk = out[: B * O].view(B, O).cpu()
    assert_mlp_close(outk, out_ref, "out")
    Xa = Xa.cpu()
    outside = torch.ones_like(Xa, dtype=torch.bool)
    outside[:B, col0:col0 + A] = False
    assert bool((Xa[outside] == MARK).all()), "a: written outside its column block"
    a = Xa[:B, col0:col0 + A]
    if logp is not None:
        assert_tail(logp, B, "logp")
        logp = logp[:B].cpu()
    if tanh_out is not None:
        assert_tail(tanh_out, B * A, "tanh_out")
        tanh_out = tanh_out[: B * A].view(B, A).cpu()
    check_head(det, outk, eps, noise, clip, a, logp, tanh_out, path)
    if variant == "saturate" and B > 1:
        x = f64(outk[:, :2]) + f64(eps[:, :2]) * torch.exp(LO + 0.5 * (HI - LO) * (torch.tanh(f64(outk[:, A:A + 2])) + 1.0))
        assert bool((x < -50).any()), "test data: no sample deep in the softplus threshold branch"


# ------------------------------------------------------------------------------------------------ D: row-local policy
ROWS_SHAPES = [(1, 63, 64), (8, 56, 256), (8, 17, 128), (1, 17, 256)]   # A, D, H (D + A = 64 in the first two)
ROWS_MODES = ["stochastic", "det", "det-noise-clip", "det-noise-noclip"]
ROWS_CASES = [(A, D, H, B, mode) for i, B in enumerate((1, 5, 8, 9, 16, 17, 300)) for j, mode in enumerate(ROWS_MODES)
              for (A, D, H) in [ROWS_SHAPES[(i + j) % len(ROWS_SHAPES)]]]


@gpu
@pytest.mark.parametrize("A,D,H,B,mode", ROWS_CASES)
def test_policy_rows(A, D, H, B, mode):
    det = mode != "stochastic"
    variant = {"stochastic": "plain", "det": "eps", "det-noise-clip": "eps+noise-clip", "det-noise-noclip": "noise-noclip"}[mode]
    st, X, eps, noise, clip = actor_inputs(A, det, D, H, B, variant, seed=A * 31 + D + H + B)
    O = A if det else 2 * A
    assert L().rows_supported(D, H, O) == 1
    P = params_dev(st)
    ldx = D + 2
    Xd = X.to(DEV)
    epsd, noised = (None if t is None else t.to(DEV) for t in (eps, noise))
    col0, lda = 3, A + 5
    res = {}
    for who in ("rows", "forward_sample"):
        out = nan_with_tail(B * O)
        Xa = torch.full((B + 1, lda), MARK, device=DEV)
        logp = None if det else nan_with_tail(B)
        tanh_out = nan_with_tail(B * A) if det else None
        if who == "rows":
            names = profiled_kernels(lambda: L().policy_rows(
                *wptrs(P), D, H, A, int(det), Xd.data_ptr(), ldx, B, out.data_ptr(), ptr(epsd), ptr(noised), SIGMA, clip, LO,
                HI, Xa[:, col0:].data_ptr(), lda, ptr(logp), ptr(tanh_out), S()))
            assert_ran(names, "mlp_rows_kernel", absent=("head_forward_kernel", "mlp3_forward_kernel"))
        else:
            h1, h2 = torch.empty((B, H), device=DEV), torch.empty((B, H), device=DEV)
            L().actor_forward_sample(*wptrs(P), D, H, A, int(det), Xd.data_ptr(), ldx, B, h1.data_ptr(), h2.data_ptr(), 0,
                                     out.data_ptr(), ptr(epsd), ptr(noised), SIGMA, clip, LO, HI, Xa[:, col0:].data_ptr(), lda,
                                     ptr(logp), ptr(tanh_out), 1, S())
        torch.cuda.synchronize()
        assert_tail(out, B * O, f"{who} out")
        Xa = Xa.cpu()
        outside = torch.ones_like(Xa, dtype=torch.bool)
        outside[:B, col0:col0 + A] = False
        assert bool((Xa[outside] == MARK).all()), f"{who}: a written outside its column block"
        if logp is not None:
            assert_tail(logp, B, f"{who} logp")
            logp = logp[:B].cpu()
        if tanh_out is not None:
            assert_tail(tanh_out, B * A, f"{who} tanh_out")
            tanh_out = tanh_out[: B * A].view(B, A).cpu()
        outk = out[: B * O].view(B, O).cpu()
        a = Xa[:B, col0:col0 + A]
        res[who] = (outk, a, logp)
        assert_mlp_close(outk, ref_mlp(st, 0, X[:, :D])[2], f"{who} out")
        check_head(det, outk, eps, noise, clip, a, logp, tanh_out, who)
    (o1, a1, l1), (o2, a2, l2) = res["rows"], res["forward_sample"]
    gu.assert_close(o1.numpy(), o2.numpy(), 1e-5, 2e-6 * max(1.0, float(o2.abs().max())), "rows vs forward_sample: out")
    gu.assert_close(a1.numpy(), a2.numpy(), 0.0, 2e-5, "rows vs forward_sample: a")
    if not det:
        gu.assert_close(l1.numpy(), l2.numpy(), 1e-4, 1e-4, "rows vs forward_sample: logp")


@gpu
def test_host_side_rejections():
    """Arguments outside an entry point's range come back as error codes before anything is launched."""
    D, H = 56, 64
    st = uo.MLPStack(1, D, H, 18).random_init(torch.Generator().manual_seed(1))
    P = params_dev(st)
    x = torch.zeros(4, 64, device=DEV)
    a = torch.zeros(4, 16, device=DEV)
    eps = torch.zeros(4, 16, device=DEV)

    def rows(D_, A):
        return L().policy_rows.raw(*wptrs(P), D_, H, A, 0, x.data_ptr(), 64, 4, None, eps.data_ptr(), None, 0.0, 0.0, LO, HI,
                                   a.data_ptr(), 16, None, None, S())

    assert rows(D, 9) == -1                                 # SSAC_E_BADARG: A > 8
    assert rows(57, 8) == -2                                # SSAC_E_UNSUPPORTED: D + A > 64
    assert rows(D - 1, 8) == 0
    N, B = 2, 4
    stc = uo.MLPStack(N, 8, 32, 1).random_init(torch.Generator().manual_seed(2))
    Pc = params_dev(stc)
    h = torch.zeros(N, B, 32, device=DEV)
    q, dq, qt = torch.zeros(N, B, device=DEV), torch.zeros(N, B, device=DEV), torch.zeros(2, B, device=DEV)
    one, pa = torch.zeros(B, device=DEV), torch.tensor([0.0, 1.0, 1.0, 0.0], device=DEV)
    rc = critic_call(Pc, N, 8, 32, x, 64, B, h, h, q, None, None, None, pa, 1, 1, 0, dq, None, 2, 2, qt=qt, M=2, r=one, d=one,
                     raw=True)
    assert rc == -1                                         # SSAC_E_BADARG: in-place TD target with PopArt
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ E: small kernels
@gpu
@pytest.mark.parametrize("N", [1, 2, 10])
@pytest.mark.parametrize("E,with_logp,popart", [(1, True, None), (3, True, 1), (3, False, 0), (2, False, 1)])
def test_actor_loss_seed(N, E, with_logp, popart):
    gen = torch.Generator().manual_seed(N * 10 + E)
    B = 300
    q = torch.randn(N, B, generator=gen)
    if N > 1:   # exact ties: the seed goes to the net the reference's CPU min picks
        q[N - 1, :40] = q[0, :40]
        q[:, 40:60] = q[0, 40:60]
        q[1, 60:80] = q[:, 60:80].min(0).values
    logp = torch.randn(B, generator=gen) if with_logp else None
    la = torch.tensor([math.log(0.3)])
    pa = torch.tensor([0.2, 1.3, 1.7, -0.3]) if popart is not None else None
    pop = int(popart or 0)
    qd, lad = q.to(DEV), la.to(DEV)
    lpd, pad = (None if t is None else t.to(DEV) for t in (logp, pa))
    vals, dq = nan_with_tail(B), nan_with_tail(N * B)
    loss = torch.tensor([0.5], device=DEV)
    L().actor_loss_seed(qd.data_ptr(), N, B, ptr(lpd), lad.data_ptr(), ptr(pad), pop, E, vals.data_ptr(), dq.data_ptr(),
                        loss.data_ptr(), S())
    torch.cuda.synchronize()
    assert_tail(vals, B, "vals")
    assert_tail(dq, N * B, "dq")
    m, arg = torch.stack(list(q), 0).min(0)
    assert torch.equal(ref_arg_min(q), arg)
    pw, pb = (float(pa[2]), float(pa[3])) if pop else (1.0, 0.0)
    seed = -pw / (E * B)
    dqk = dq[: N * B].view(N, B).cpu()
    onehot = torch.zeros(N, B, dtype=torch.bool)
    onehot[arg, torch.arange(B)] = True
    assert torch.equal(dqk != 0, onehot), "seed routed to another net than torch.min's arg-min"
    assert bool((dqk[~onehot] == 0).all())
    assert_within(dqk[onehot], torch.full((B,), seed, dtype=torch.float64), 2 * U * abs(seed), "seed")
    v_ref = pw * f64(m) + pb
    assert_within(vals[:B].cpu(), v_ref, 2 * U * (v_ref.abs() + abs(pw) * f64(m).abs()), "vals")
    alpha = math.exp(float(la))
    ent = alpha * f64(logp) if with_logp else torch.zeros(B, dtype=torch.float64)
    terms = v_ref - ent
    want = 0.5 - float(terms.mean()) / E
    e_terms = 4 * U * (v_ref.abs() + abs(pw) * f64(m).abs() + ent.abs() + terms.abs())
    assert_within(loss.cpu()[0], want, sum_bound(terms, e_terms) / (B * E) + 4 * U * (abs(want) + 0.5), "loss (+=)")


@gpu
def test_sum_groups_strided():
    gen = torch.Generator().manual_seed(3)
    G, B, D, col0, A = 3, 37, 23, 17, 6
    lddx = D + 5                                            # lddx > col0 + A
    dx = torch.randn(G, B, lddx, generator=gen)
    out = nan_with_tail(B * A)
    dxd = dx.to(DEV)
    L().sum_groups(dxd.data_ptr(), G, B, lddx, col0, A, out.data_ptr(), S())
    torch.cuda.synchronize()
    assert_tail(out, B * A, "out")
    sel = f64(dx[:, :, col0:col0 + A])
    assert_within(out[: B * A].view(B, A).cpu(), sel.sum(0), G * U * sel.abs().sum(0), "sum over groups")


@gpu
def test_dr3_dot_overwrites():
    gen = torch.Generator().manual_seed(4)
    N, B, H = 10, 1024, 1024
    f = torch.relu(torch.randn(N, B, H, generator=gen))
    f1 = torch.relu(torch.randn(N, B, H, generator=gen))
    fd, f1d = f.to(DEV), f1.to(DEV)
    out = torch.tensor([5.0, MARK], device=DEV)
    for _ in range(2):   # the second call must not see the first one's result
        L().dr3_dot(fd.data_ptr(), f1d.data_ptr(), N, B, H, out.data_ptr(), S())
    torch.cuda.synchronize()
    prod = f64(f) * f64(f1)
    want = float(prod.sum(-1).mean())
    n = N * B * H
    grid = min((n + 255) // 256, 2 * 148)                   # dr3_dot_kernel: grid-stride loop, block tree, one atomic per block
    depth = -(-n // (grid * 256)) + 16 + grid
    assert_within(out.cpu()[0], want, depth * U * float(prod.sum()) / (N * B) + 2 * U * want, "dr3 dot product")
    assert float(out[1]) == MARK


@gpu
def test_alpha_step_matches_torch_adam():
    """10 steps of ssac_alpha_step against torch.optim.Adam on the fp32 scalar (what the reference runs) and against a
    float64 re-statement; mean(logp + target_entropy) changes sign along the way."""
    B, te, lr, b1, b2, eps = 256, -6.0, 3e-2, 0.5, 0.999, 1e-8
    gen = torch.Generator().manual_seed(5)
    la0 = math.log(0.1)
    la_t = torch.tensor([la0], requires_grad=True)
    opt = torch.optim.Adam([la_t], lr=lr, betas=(b1, b2), eps=eps)
    la_d = torch.tensor([la0, MARK], device=DEV)
    state = torch.zeros(2, device=DEV)
    ctl = torch.tensor([0, 7], dtype=torch.int32, device=DEV)
    logs = torch.full((3,), MARK, device=DEV)
    p64, m64, v64 = float(torch.tensor(la0)), 0.0, 0.0
    means = []
    for t in range(1, 11):
        logp = torch.randn(B, generator=gen) * 0.5 + (6.5 if t % 3 else 5.2)
        lpd = logp.to(DEV)
        L().alpha_step(la_d.data_ptr(), lpd.data_ptr(), B, te, state.data_ptr(), ctl.data_ptr(), lr, b1, b2, eps,
                       logs.data_ptr(), S())
        la_prev = float(la_t.detach())
        opt.zero_grad()
        loss_t = -(la_t * (logp + te).detach()).mean()
        loss_t.backward()
        g64 = -float(f64(logp + te).mean())
        means.append(-g64)
        loss64 = -p64 * (-g64)
        p64, m64, v64 = ref_adam_scalar(p64, g64, m64, v64, t, lr, b1, b2, eps)
        opt.step()
        torch.cuda.synchronize()
        la_k, st_k, lg = f64(la_d.cpu()), f64(state.cpu()), f64(logs.cpu())
        ts = opt.state[la_t]
        assert ctl.cpu().tolist() == [t, 7], f"step {t}: ctl"
        assert float(la_k[1]) == MARK and float(lg[2]) == MARK
        assert_within(la_k[0], float(la_t.detach()), 4 * t * U * abs(float(la_t.detach())) + 1e-3 * lr * U, f"step {t}: log_alpha vs torch Adam")
        assert_within(st_k, [float(ts["exp_avg"]), float(ts["exp_avg_sq"])],
                      [16 * U * abs(float(ts["exp_avg"])) + 1e-30, 16 * U * float(ts["exp_avg_sq"]) + 1e-30],
                      f"step {t}: Adam state vs torch")
        e_loss = 2 * B * U * abs(la_prev) * float(f64(logp + te).abs().mean()) + 4 * U * abs(float(loss_t.detach()))
        assert_within(lg[0], float(loss_t.detach()), e_loss, f"step {t}: alpha loss")
        assert_within(lg[1], math.exp(float(la_k[0])), 3 * U * math.exp(float(la_k[0])), f"step {t}: alpha")
        assert_within(la_k[0], p64, 8 * t * U * abs(p64), f"step {t}: log_alpha vs float64")
        assert_within(st_k, [m64, v64], [1e-5 * abs(m64), 1e-5 * v64], f"step {t}: Adam state vs float64")
        assert_within(lg[0], loss64, 1e-5 * abs(loss64), f"step {t}: alpha loss vs float64")
    assert min(means) < 0 < max(means), "test data: mean(logp + target_entropy) never changed sign"


@gpu
@pytest.mark.parametrize("with_popart", [False, True])
def test_min_over_nets(with_popart):
    gen = torch.Generator().manual_seed(6)
    N, B = 4, 301
    q = torch.randn(N, B, generator=gen)
    q[2, :30] = q[0, :30]
    pa = torch.tensor([0.2, 1.3, 1.7, -0.3]) if with_popart else None
    out = nan_with_tail(B)
    qd = q.to(DEV)
    pad = None if pa is None else pa.to(DEV)
    L().min_over_nets(qd.data_ptr(), N, B, ptr(pad), out.data_ptr(), S())
    torch.cuda.synchronize()
    assert_tail(out, B, "out")
    want = torch.stack(list(q), 0).min(0).values
    if pa is not None:
        want = pa[2] * want + pa[3]                       # two fp32 roundings, as in agent.py:37-38
    assert torch.equal(out[:B].cpu(), want)


@gpu
def test_det_head_backward_strided():
    gen = torch.Generator().manual_seed(7)
    B, A, ldda = 129, 6, 11
    th = torch.tanh(torch.randn(B, A, generator=gen) * 2)
    da = torch.randn(B, ldda, generator=gen)
    out = nan_with_tail(B * A)
    thd, dad = th.to(DEV), da.to(DEV)
    L().det_head_backward(thd.data_ptr(), dad.data_ptr(), ldda, B, A, out.data_ptr(), S())
    torch.cuda.synchronize()
    assert_tail(out, B * A, "dout")
    g = f64(da[:, :A])
    want = g * (1.0 - f64(th) ** 2)
    assert_within(out[: B * A].view(B, A).cpu(), want, 3 * U * g.abs(), "dout = da (1 - tanh^2)")


@gpu
def test_scale_by_dev_bit_exact():
    gen = torch.Generator().manual_seed(8)
    n, off = 1_000_003, 3
    x0 = torch.randn(n + off + 1, generator=gen)
    s = torch.tensor([0.37])
    xd, sd = x0.to(DEV), s.to(DEV)
    L().scale_by_dev(xd.data_ptr() + 4 * off, n, sd.data_ptr(), S())
    torch.cuda.synchronize()
    xk = xd.cpu()
    assert torch.equal(xk[off:off + n], s * x0[off:off + n])
    assert torch.equal(xk[:off], x0[:off]) and torch.equal(xk[off + n:], x0[off + n:])


@gpu
def test_polyak_multi_bit_exact_table():
    """A multi-million-element tensor (every thread loops: the grid is capped at 4 x 148 blocks), a 1-element tensor and a
    view at an odd element offset, in one table."""
    gen = torch.Generator().manual_seed(9)
    tau = 0.005
    sizes = [3_000_001, 1, 777]
    offs = [0, 0, 5]
    tgt0 = [torch.randn(n + o + 2, generator=gen) for n, o in zip(sizes, offs)]
    src0 = [torch.randn(n + o + 2, generator=gen) for n, o in zip(sizes, offs)]
    tgt, src = [t.to(DEV) for t in tgt0], [s.to(DEV) for s in src0]
    table = torch.tensor([[t.data_ptr() + 4 * o, s.data_ptr() + 4 * o, n] for t, s, n, o in zip(tgt, src, sizes, offs)],
                         dtype=torch.int64, device=DEV)
    L().polyak_multi(table.data_ptr(), len(sizes), max(sizes), tau, S())
    torch.cuda.synchronize()
    for t0, s0, t, n, o in zip(tgt0, src0, tgt, sizes, offs):
        got = t.cpu()
        assert torch.equal(got[o:o + n], t0[o:o + n] * (1.0 - tau) + s0[o:o + n] * tau), f"numel {n}"
        assert torch.equal(got[:o], t0[:o]) and torch.equal(got[o + n:], t0[o + n:]), f"numel {n}: written outside"

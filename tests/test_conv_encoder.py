"""N3: the native DrQ pixel encoder (csrc/ssac_conv.cu behind nets.cnns.BigPixelEncoder) against

* the golden vectors of the unmodified reference module (tests/golden/encoder.npz), through the C ABI, layer by layer
  (every activation and every per-layer gradient is compared with oracle/encoder_oracle.py, which test_oracle_golden.py
  pins against the same fixture), and through the drop-in module + autograd;
* the oracle at the BASELINE geometry (9 x 84 x 84, out_dim 50).

Tolerance: north_star's rtol 1e-4 (+ atol 1e-4 of the tensor's largest magnitude: sums of thousands of 3xTF32 products of
either sign).  CPU part: the library exports the entry points and plans its workspace.
"""
import ctypes

import numpy as np
import pytest
import torch

import golden_util as gu
from oracle import encoder_oracle as eo

RTOL = 1e-4


def _close(got, want, what, rtol=RTOL, rel_atol=1e-4, flip_frac=0.0):
    """flip_frac: fraction of elements allowed to disagree -- a pre-activation within rounding of zero lands on either
    side of the ReLU in two correct fp32 forwards (DESIGN.md 4), which switches single elements of dL/dz on or off."""
    want = np.asarray(want, dtype=np.float64)
    atol = rel_atol * max(float(np.abs(want).max()), 1e-30)
    if flip_frac:
        bad = np.abs(np.asarray(got, dtype=np.float64) - want) > atol + rtol * np.abs(want)
        assert bad.sum() <= flip_frac * bad.size, f"{what}: {int(bad.sum())} of {bad.size} elements disagree"
        return
    gu.assert_close(got, want, rtol, atol, what)


def test_workspace_plan_cpu():
    """No GPU needed: the plan is host arithmetic (and the symbols exist)."""
    from super_sac_b200 import _lib

    lib = _lib.lib()
    n = ctypes.c_int64()
    lib.conv_encoder_ws_floats(512, 9, 84, 84, 50, 1, ctypes.byref(n))
    off = (ctypes.c_int64 * 32)()
    lib.conv_encoder_ws_offsets(512, 9, 84, 84, 50, 1, off)
    rows, pitch = [off[i] for i in range(16, 20)], [off[i] for i in range(20, 24)]
    kf, kfp, ks, nsplit, total = [off[i] for i in range(24, 29)]
    assert rows == pitch == [42, 41, 39, 37]      # layer l works on its input grid: s2d 42, then the valid outputs 41 / 39 / 37
    assert kf == 37 * 37 * 32 and kfp == ks * nsplit >= kf and ks % 32 == 0
    assert total == n.value and all(off[i] % 256 == 0 for i in range(16))
    with pytest.raises(_lib.SsacError):
        lib.conv_encoder_ws_floats(4, 17, 84, 84, 50, 1, ctypes.byref(n))   # 4C must fit 64 channels
    with pytest.raises(_lib.SsacError):
        lib.conv_encoder_ws_floats(4, 9, 83, 84, 50, 1, ctypes.byref(n))


def test_encoder_entry_point_fails_loudly_without_a_device():
    """No GPU (or bad arguments): an error code and a message, never a silent CPU path."""
    if torch.cuda.is_available():
        pytest.skip("this check is for machines without a GPU")
    from super_sac_b200 import _lib

    ptrs = _lib.host_array(ctypes.c_void_p, [0] * 12)
    with pytest.raises(_lib.SsacError):
        _lib.lib().conv_encoder_forward(None, 4, 3, 20, 20, 10, ptrs, None, 0, None, None)


class _Native:
    """The encoder through the C ABI with a test-owned workspace (so intermediates can be inspected)."""

    def __init__(self, params, B, C, H, W, O, save=1):
        from super_sac_b200 import _lib

        self.lib, self._lib = _lib.lib(), _lib
        self.dims = (B, C, H, W, O)
        self.save = save
        self.params = [torch.as_tensor(np.asarray(params[n])).float().cuda().contiguous() for n in eo.PARAM_NAMES]
        n = ctypes.c_int64()
        self.lib.conv_encoder_ws_floats(B, C, H, W, O, save, ctypes.byref(n))
        self.ws = torch.zeros(n.value, device="cuda")
        off = (ctypes.c_int64 * 32)()
        self.lib.conv_encoder_ws_offsets(B, C, H, W, O, save, off)
        self.off = list(off)
        self.rows, self.pitch = [0] + self.off[16:20], [0] + self.off[20:24]     # grid of layer l = 1..4
        self.out = torch.empty(B, O, device="cuda")
        self.grads = [torch.full_like(p, float("nan")) for p in self.params]

    def _ptrs(self, ts):
        return self._lib.host_array(ctypes.c_void_p, [t.data_ptr() for t in ts])

    def forward(self, obs):
        B, C, H, W, O = self.dims
        self.obs = torch.as_tensor(np.asarray(obs)).float().cuda().contiguous()
        self.lib.conv_encoder_forward(self.obs.data_ptr(), B, C, H, W, O, self._ptrs(self.params), self.ws.data_ptr(),
                                      self.save, self.out.data_ptr(), self._lib.stream_ptr())
        torch.cuda.synchronize()
        return self.out.cpu().numpy()

    def backward(self, dout):
        B, C, H, W, O = self.dims
        d = torch.as_tensor(np.asarray(dout)).float().cuda().contiguous()
        self.lib.conv_encoder_backward(d.data_ptr(), self.out.data_ptr(), self.obs.data_ptr(), B, C, H, W, O, self._ptrs(self.params),
                                       self.ws.data_ptr(), self._ptrs(self.grads), self._lib.stream_ptr())
        torch.cuda.synchronize()
        return {n: g.cpu().numpy() for n, g in zip(eo.PARAM_NAMES, self.grads)}

    def act(self, layer):
        """Output of conv layer `layer` as NCHW (valid region only): y1..y3 are stored compacted on the next layer's grid,
        y4 on layer 4's own grid."""
        B = self.dims[0]
        g = min(layer + 1, 4)
        R, P = self.rows[g], self.pitch[g]
        o = self.off[layer]
        x = self.ws[o:o + B * R * P * 32].view(B, R, P, 32)
        if layer == 4:
            x = x[:, :R - 2, :P - 2, :]
        return x.permute(0, 3, 1, 2).contiguous().cpu().numpy()

    def dz(self, layer):
        """dL/d(pre-activation) of conv layer `layer`: stored on that layer's grid; returns (valid region as NCHW, full view)."""
        B = self.dims[0]
        R, P = self.rows[layer], self.pitch[layer]
        o = self.off[4 + layer]
        full = self.ws[o:o + B * R * P * 32].view(B, R, P, 32)
        v_h, v_w = (R - 1, P - 1) if layer == 1 else (R - 2, P - 2)
        return full[:, :v_h, :v_w, :].permute(0, 3, 1, 2).contiguous().cpu().numpy(), full, (v_h, v_w)


def _native_masks(nat, cache, tag):
    """The ReLU patterns of the native forward; where they differ from the oracle's, the oracle's activation is within
    rounding of zero (DESIGN.md 4) -- and that happens for a handful of elements only."""
    masks = {}
    for l in range(1, 5):
        got = nat.act(l)
        want = cache["acts"][l].numpy()
        _close(got, want, f"{tag} y{l}")
        masks[l] = got > 0
        diff = masks[l] != (want > 0)
        assert diff.sum() <= 1e-5 * diff.size + 2, f"{tag} y{l}: {int(diff.sum())} ReLU decisions differ"
        if diff.any():
            assert np.abs(want[diff]).max() <= 1e-4 * np.abs(want).max() and np.abs(got[diff]).max() <= 1e-4 * np.abs(want).max()
    return masks


def _check_layers(nat, cache, g, tag):
    for l in (4, 3, 2, 1):
        got, full, (v_h, v_w) = nat.dz(l)
        _close(got, g[f"dz{l}"].numpy(), f"{tag} dz{l}")
        assert float(full[:, v_h:, :, :].abs().max()) == 0.0 and float(full[:, :, v_w:, :].abs().max()) == 0.0, \
            f"{tag} dz{l}: gradient outside the valid region"


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["rgb20", "stack24"])
def test_encoder_golden_through_c_abi(tag):
    fx = gu.load("encoder")
    params = gu.sub(fx, f"{tag}/params")
    obs = fx[f"{tag}/obs"].astype(np.float32)
    B, C, H, W = obs.shape
    O = fx[f"{tag}/out"].shape[1]
    nat = _Native(params, B, C, H, W, O)
    out = nat.forward(obs)
    ref_out, cache = eo.forward(params, obs)
    # layer by layer against the oracle first (localises a failure), then the reference's own numbers
    masks = _native_masks(nat, cache, tag)
    g_or = eo.backward(cache, fx[f"{tag}/dout"], masks)
    _close(out, fx[f"{tag}/out"], f"{tag} out")
    grads = nat.backward(fx[f"{tag}/dout"])
    _check_layers(nat, cache, g_or, tag)
    want = gu.sub(fx, f"{tag}/grads")
    for n in reversed(eo.PARAM_NAMES):
        _close(grads[n], want[n], f"{tag} grad {n}")
    # a second pass over the same (now dirty) workspace gives the same bits: nothing leaks through the padding
    out2 = nat.forward(obs)
    grads2 = nat.backward(fx[f"{tag}/dout"])
    assert np.array_equal(out, out2)
    for n in eo.PARAM_NAMES:
        assert np.array_equal(grads[n], grads2[n]), n
    # the no-grad variant (ping-pong buffers) computes the same forward
    nat0 = _Native(params, B, C, H, W, O, save=0)
    assert np.array_equal(nat0.forward(obs), out)


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["rgb20", "stack24"])
def test_encoder_module_autograd_matches_reference(tag):
    """The drop-in module: forward + loss.backward() fill .grad like the reference's autograd does; a deepcopy (the target
    encoder, main.py:321) runs without grad on its own workspace."""
    import copy

    from super_sac_b200.nets import cnns

    fx = gu.load("encoder")
    obs = fx[f"{tag}/obs"]
    B, C, H, W = obs.shape
    O = fx[f"{tag}/out"].shape[1]
    enc = cnns.BigPixelEncoder((C, H, W), out_dim=O)
    enc.load_state_dict({k: torch.as_tensor(v) for k, v in gu.sub(fx, f"{tag}/params").items()})
    enc.cuda()
    x = torch.as_tensor(obs).cuda().float()
    y = enc(x)
    _close(y.detach().cpu().numpy(), fx[f"{tag}/out"], f"{tag} module out")
    (y * torch.as_tensor(fx[f"{tag}/dout"]).cuda()).sum().backward()
    want = gu.sub(fx, f"{tag}/grads")
    for n, p in enc.named_parameters():
        _close(p.grad.cpu().numpy(), want[n], f"{tag} module grad {n}")
    tgt = copy.deepcopy(enc)
    with torch.no_grad():
        y2 = tgt(x)
    assert torch.equal(y2, y.detach())
    # uint8 observations are accepted as they come out of the replay ring
    with torch.no_grad():
        assert torch.equal(enc(torch.as_tensor(obs).cuda()), y.detach())


@pytest.mark.gpu
@pytest.mark.parametrize("B", [64, 512])
def test_encoder_baseline_geometry_against_oracle(B):
    """BASELINE config 4: 9 x 84 x 84 uint8 frames, out_dim 50 (B = 512 is the bench's batch)."""
    rng = np.random.default_rng(5)
    torch.manual_seed(5)
    C, H, W, O = 9, 84, 84, 50
    from super_sac_b200.nets import cnns

    enc = cnns.BigPixelEncoder((C, H, W), out_dim=O)
    with torch.no_grad():
        for p in enc.parameters():
            p.add_(0.02 * torch.randn_like(p))
    params = {k: v.detach().numpy() for k, v in enc.named_parameters()}
    obs = rng.integers(0, 256, (B, C, H, W)).astype(np.float32)
    dout = rng.standard_normal((B, O)).astype(np.float32)
    torch.set_num_threads(max(1, torch.get_num_threads()))
    ref_out, cache = eo.forward(params, obs)
    nat = _Native(params, B, C, H, W, O)
    out = nat.forward(obs)
    masks = _native_masks(nat, cache, f"B{B}")
    g = eo.backward(cache, dout, masks)   # both sides differentiate through the same ReLU pattern
    _close(out, ref_out.numpy(), "out")
    grads = nat.backward(dout)
    _check_layers(nat, cache, g, f"B{B}")
    for n in reversed(eo.PARAM_NAMES):
        _close(grads[n], g[n].numpy(), f"grad {n}")


@pytest.mark.gpu
def test_fused_encoder_optimizer_step_matches_torch():
    """clip_grad_norm_ + torch.optim.Adam.step() over the encoder's parameters (learning.py:122-131) == ssac_sumsq +
    ssac_adam_step over its flat gradient buffer (_encoder_opt.fused_step), step after step, and the optimiser's state
    (what a checkpoint saves) is the one torch would have produced."""
    from super_sac_b200 import _encoder_opt, nets
    from super_sac_b200.nets import cnns

    class Enc(nets.Encoder):   # experiments/dmc/train_dmc_from_pixels.py:15-27
        def __init__(self):
            super().__init__()
            self.net = cnns.BigPixelEncoder((3, 20, 20), 10)

        @property
        def embedding_dim(self):
            return 10

        def forward(self, obs_dict):
            return self.net(obs_dict["obs"])

    torch.manual_seed(3)
    a = Enc().cuda()
    with torch.no_grad():
        for p in a.parameters():
            p.add_(0.05 * torch.randn_like(p))
    import copy

    b = copy.deepcopy(a)
    oa = torch.optim.Adam(a.parameters(), lr=1e-3)
    ob = torch.optim.Adam(b.parameters(), lr=1e-3)
    for step in range(4):
        obs = {"obs": torch.randint(0, 256, (6, 3, 20, 20), device="cuda").float()}
        w = torch.randn(6, 10, device="cuda") * (30.0 if step % 2 else 0.3)    # clipping active on odd steps
        for enc, opt in ((a, oa), (b, ob)):
            opt.zero_grad()
            (enc(obs) * w).sum().backward()
        if step == 2:   # autograd may hand a parameter a COPY of the gradient instead of adopting the flat view: the fused
            for p in list(a.net.parameters())[::2]:          # step then moves it into the flat buffer first
                p.grad = p.grad.clone()
        assert _encoder_opt.fused_step(a, oa, 5.0) is a.net
        assert all(p.grad.data_ptr() == a.net._flat_grad.data_ptr() + 4 * o for p, o in zip(a.net._native_params(), a.net._flat_off))
        torch.nn.utils.clip_grad_norm_(b.parameters(), 5.0)
        ob.step()
        for (n, pa), pb in zip(a.named_parameters(), b.parameters()):
            _close(pa.detach().cpu().numpy(), pb.detach().cpu().numpy(), f"step {step} {n}", rtol=2e-6, rel_atol=1e-6)
            if pa.grad is not None:   # clip_grad_norm_ scales .grad in place: so does the fused step
                _close(pa.grad.cpu().numpy(), pb.grad.cpu().numpy(), f"step {step} grad {n}", rtol=2e-6, rel_atol=1e-6)
    sa, sb = oa.state_dict()["state"], ob.state_dict()["state"]
    for k in sb:
        if k in sa or len(sb[k]):
            assert float(sa[k]["step"]) == float(sb[k]["step"]) == 4.0
            _close(sa[k]["exp_avg"].cpu().numpy(), sb[k]["exp_avg"].cpu().numpy(), f"exp_avg {k}", rtol=2e-6, rel_atol=1e-6)
            _close(sa[k]["exp_avg_sq"].cpu().numpy(), sb[k]["exp_avg_sq"].cpu().numpy(), f"exp_avg_sq {k}", rtol=2e-6, rel_atol=1e-6)
    # two backward passes before a step: the second one accumulates (in place, into the flat buffer) like autograd always does
    oa.zero_grad()
    (a(obs) * w).sum().backward()
    g1 = a.net.conv2.weight.grad.clone()
    (a(obs) * w).sum().backward()
    _close(a.net.conv2.weight.grad.cpu().numpy(), 2.0 * g1.cpu().numpy(), "accumulated gradient", rtol=1e-6, rel_atol=1e-7)
    assert _encoder_opt.eligible(a, oa) is a.net


@pytest.fixture
def conv_halo(request):
    """ssac_set_conv_halo(mode) for the duration of one test, then the default (3) again."""
    from super_sac_b200 import _lib

    _lib.lib().set_conv_halo(request.param)
    yield request.param
    _lib.lib().set_conv_halo(3)


@pytest.mark.gpu
@pytest.mark.parametrize("conv_halo", [3, 0], ids=["halo", "per-tap"], indirect=True)
@pytest.mark.parametrize("B,C,H,W,O", [(1, 9, 84, 84, 50), (2, 1, 16, 16, 8), (3, 16, 20, 28, 64), (7, 4, 32, 18, 33)])
def test_encoder_edge_geometries_against_oracle(B, C, H, W, O, conv_halo):
    """Batch of one (the acting path), one channel, the widest channel count (4C = 64), non-square images, the smallest
    image (a single valid output pixel in the last layer), an odd output width.  Each with the default kernel choice
    (halo tiles wherever the halo box fits, as it does at these sizes) and with the per-tap kernels forced (mode 0: the
    fallback for images whose halo box does not fit)."""
    from super_sac_b200.nets import cnns

    rng = np.random.default_rng(B * 1000 + C)
    torch.manual_seed(B * 1000 + C)
    enc = cnns.BigPixelEncoder((C, H, W), out_dim=O)
    with torch.no_grad():
        for p in enc.parameters():
            p.add_(0.05 * torch.randn_like(p))
    params = {k: v.detach().numpy() for k, v in enc.named_parameters()}
    obs = rng.integers(0, 256, (B, C, H, W)).astype(np.float32)
    dout = rng.standard_normal((B, O)).astype(np.float32)
    ref_out, cache = eo.forward(params, obs)
    nat = _Native(params, B, C, H, W, O)
    out = nat.forward(obs)
    masks = _native_masks(nat, cache, f"{B}x{C}x{H}x{W}")
    g = eo.backward(cache, dout, masks)
    _close(out, ref_out.numpy(), "out")
    grads = nat.backward(dout)
    for n in reversed(eo.PARAM_NAMES):
        _close(grads[n], g[n].numpy(), f"grad {n}")


@pytest.mark.gpu
def test_update_entry_points_with_native_encoder_fused_vs_torch_optimizer(monkeypatch):
    """critic_update and offline_actor_update(update_encoder=True) on an agent whose encoder is the native BigPixelEncoder:
    the fused clip + Adam over the flat buffers gives the parameters the torch calls give (same kernels everywhere else),
    and one optimiser keeps one kind of state whichever entry point stepped it."""
    import copy
    import math
    from itertools import chain

    import super_sac_b200 as ssb
    from super_sac_b200 import _rng, augmentations, learning, nets
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

    def build():
        torch.manual_seed(11)
        ssb.manual_seed(11)
        agent = ssb.Agent(act_space_size=3, encoder=Enc(), actor_network_cls=nets.mlps.ContinuousStochasticActor,
                          critic_network_cls=nets.mlps.ContinuousCritic, ensemble_size=1, num_critics=2, hidden_size=32,
                          auto_rescale_targets=False, log_std_low=-5.0, log_std_high=2.0)
        agent.to("cuda")
        target = copy.deepcopy(agent)
        rng = np.random.default_rng(11)
        n = 64
        buf = ssb.replay.ReplayBuffer(n, device="cuda")
        buf.load_experience({"pixels": rng.integers(0, 256, (n, 3, 20, 20), dtype=np.uint8)}, rng.uniform(-0.9, 0.9, (n, 3)).astype(np.float32),
                            rng.standard_normal(n).astype(np.float32), {"pixels": rng.integers(0, 256, (n, 3, 20, 20), dtype=np.uint8)},
                            rng.uniform(size=n) < 0.05)
        c_opt = torch.optim.Adam(chain(*(c.parameters() for c in agent.critics)), lr=3e-4)
        a_opt = torch.optim.Adam(chain(*(a.parameters() for a in agent.actors)), lr=3e-4)
        e_opt = torch.optim.Adam(agent.encoder.parameters(), lr=1e-3)
        la = torch.Tensor([math.log(0.1)]).cuda()
        la.requires_grad = True
        return agent, target, buf, c_opt, a_opt, e_opt, [la]

    def run(mode):
        monkeypatch.setenv("SSAC_ENCODER_OPT", mode)
        agent, target, buf, c_opt, a_opt, e_opt, las = build()
        B = 16
        aug = augmentations.AugmentationSequence([augmentations.IdentityAug(B)])
        for _ in range(2):
            learning.critic_update(buffer=buf, agent=agent, target_agent=target, critic_optimizer=c_opt, encoder_optimizer=e_opt,
                                   log_alphas=las, batch_size=B, gamma=0.99, critic_clip=None, encoder_clip=0.5,
                                   target_critic_ensemble_n=2, weighted_bellman_temp=None, weight_type=None, pop=False,
                                   augmenter=aug, encoder_lambda=0.0, random_process=None, noise_clip=None, aug_mix=0.0)
            learning.offline_actor_update(buffer=buf, agent=agent, actor_optimizer=a_opt, encoder_optimizer=e_opt, batch_size=B,
                                          actor_clip=None, update_encoder=True, encoder_clip=0.5, augmenter=aug, actor_lambda=0.0,
                                          aug_mix=0.0, per=False, filter_=False)
        torch.cuda.synchronize()
        st = e_opt.state[agent.encoder.net.conv2.weight]
        return {k: v.detach().cpu().numpy().copy() for k, v in agent.encoder.net.named_parameters()}, float(st["step"])

    fused, fs = run("fused")
    plain, ps = run("torch")
    assert fs == ps == 4.0      # two critic updates + two offline actor updates, each stepping the encoder once
    for k in plain:
        _close(fused[k], plain[k], f"encoder {k}", rtol=1e-5, rel_atol=1e-5)


@pytest.mark.gpu
def test_encoder_training_drift_against_cpu_module():
    """10 Adam steps of the encoder alone (a fixed regression problem) on the native kernels + fused optimiser step against the
    same module trained by PyTorch on the CPU (the reference's arithmetic: fp32 conv / linear / LayerNorm, torch.optim.Adam):
    every parameter within rtol 1e-4 + 1e-5.  Measured on this very problem (tools/probes/encoder_drift_probe2.py): the
    trajectories agree to 2.4e-6 for ten steps (PyTorch-cuDNN vs PyTorch-CPU: 1.6e-6); between steps 10 and 20 the problem
    turns chaotic for ANY two fp32 implementations (cuDNN vs CPU 3.3e-4, native vs CPU 7.0e-4 at step 20, and 1.5e-2 vs
    3.9e-3 by step 60 on a sibling instance), while the fused optimiser step stays within 3e-7 of torch.optim.Adam fed the
    same gradients -- so a longer horizon would test the problem's conditioning, not the kernels."""
    import copy

    from super_sac_b200 import _encoder_opt, nets
    from super_sac_b200.nets import cnns

    class Enc(nets.Encoder):
        def __init__(self):
            super().__init__()
            self.net = cnns.BigPixelEncoder((3, 20, 20), 10)

        @property
        def embedding_dim(self):
            return 10

        def forward(self, obs_dict):
            return self.net(obs_dict["obs"])

    torch.manual_seed(21)
    cpu = Enc()
    with torch.no_grad():
        for p in cpu.parameters():
            p.add_(0.05 * torch.randn_like(p))
    gpu = copy.deepcopy(cpu).cuda()
    lr = 1e-3
    oc, og = torch.optim.Adam(cpu.parameters(), lr=lr), torch.optim.Adam(gpu.parameters(), lr=lr)
    rng = np.random.default_rng(21)
    obs = torch.as_tensor(rng.integers(0, 256, (24, 3, 20, 20)).astype(np.float32))
    tgt = torch.as_tensor(rng.uniform(-0.8, 0.8, (24, 10)).astype(np.float32))
    obs_g, tgt_g = obs.cuda(), tgt.cuda()
    torch.set_num_threads(1)
    l0 = float(((cpu({"obs": obs}) - tgt) ** 2).mean())
    for step in range(10):
        oc.zero_grad()
        ((cpu({"obs": obs}) - tgt) ** 2).mean().backward()
        oc.step()
        og.zero_grad()
        ((gpu({"obs": obs_g}) - tgt_g) ** 2).mean().backward()
        assert _encoder_opt.fused_step(gpu, og, None) is gpu.net
    for (n, pc), pg in zip(cpu.net.named_parameters(), gpu.net.parameters()):
        gu.assert_close(pg.detach().cpu().numpy(), pc.detach().numpy(), 1e-4, 1e-5, f"after 10 steps: {n}")
    lc = float(((cpu({"obs": obs}) - tgt) ** 2).mean())
    lg = float(((gpu({"obs": obs_g}) - tgt_g) ** 2).mean())
    assert lc < 0.7 * l0 and abs(lc - lg) <= 1e-4 * abs(lc) + 1e-6      # it trains, and by the same amount on both sides


@pytest.mark.gpu
def test_encoder_rejects_observations_of_another_geometry():
    from super_sac_b200.nets import cnns

    enc = cnns.BigPixelEncoder((3, 20, 20), 10).cuda()
    with pytest.raises(ValueError):
        enc(torch.zeros(2, 3, 24, 24, device="cuda"))
    with pytest.raises(ValueError):
        enc(torch.zeros(2, 4, 20, 20, device="cuda"))
    assert enc(torch.zeros(2, 3, 20, 20, device="cuda")).shape == (2, 10)


@pytest.mark.gpu
def test_auto_graphed_pixel_update_follows_the_annealed_noise_scale():
    """enable_auto_graphs() on the DrQv2-shaped update (native encoder + fused optimiser step, deterministic actor with the
    exploration-noise process): the replayed graphs give the bits the eager calls give, while the acting path keeps
    annealing sigma between the updates (the kernels read it from device memory)."""
    import copy
    import math
    from itertools import chain

    import super_sac_b200 as ssb
    from super_sac_b200 import augmentations, graphed, learning, learning_utils as lu, nets
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

    class Space:
        low, high, shape = -np.ones(3, np.float32), np.ones(3, np.float32), (3,)

    def run(graphs):
        torch.manual_seed(5)
        ssb.manual_seed(5)
        agent = ssb.Agent(act_space_size=3, encoder=Enc(), actor_network_cls=nets.mlps.ContinuousDeterministicActor,
                          critic_network_cls=nets.mlps.ContinuousCritic, ensemble_size=1, num_critics=2, hidden_size=32,
                          auto_rescale_targets=False)
        agent.to("cuda")
        target = copy.deepcopy(agent)
        rng = np.random.default_rng(5)
        n, B = 64, 16
        buf = ssb.replay.ReplayBuffer(n, device="cuda")
        buf.load_experience({"pixels": rng.integers(0, 256, (n, 3, 20, 20), dtype=np.uint8)}, rng.uniform(-0.9, 0.9, (n, 3)).astype(np.float32),
                            rng.standard_normal(n).astype(np.float32), {"pixels": rng.integers(0, 256, (n, 3, 20, 20), dtype=np.uint8)},
                            rng.uniform(size=n) < 0.05)
        c_opt = torch.optim.Adam(chain(*(c.parameters() for c in agent.critics)), lr=3e-4)
        a_opt = torch.optim.Adam(chain(*(a.parameters() for a in agent.actors)), lr=3e-4)
        e_opt = torch.optim.Adam(agent.encoder.parameters(), lr=1e-3)
        la = torch.Tensor([math.log(1e-15)]).cuda()
        la.requires_grad = True
        noise = lu.GaussianExplorationNoise(Space(), start_scale=1.0, final_scale=0.1, steps_annealed=10)
        aug = augmentations.AugmentationSequence([augmentations.Drqv2Aug(B)])
        graphed.enable_auto_graphs(graphs)
        losses = []
        try:
            for step in range(7):
                logs, rds = learning.critic_update(
                    buffer=buf, agent=agent, target_agent=target, critic_optimizer=c_opt, encoder_optimizer=e_opt, log_alphas=[la],
                    batch_size=B, gamma=0.99, critic_clip=None, encoder_clip=5.0, target_critic_ensemble_n=2,
                    weighted_bellman_temp=None, weight_type=None, pop=False, augmenter=aug, encoder_lambda=0.0,
                    random_process=noise, noise_clip=0.3, aug_mix=1.0)
                for ac, tc in zip(agent.critics, target.critics):
                    lu.soft_update(tc, ac, 0.01)
                lu.soft_update(target.encoder, agent.encoder, 1.0)
                learning.online_actor_update(buffer=buf, agent=agent, pop=False, actor_optimizer=a_opt, log_alphas=[la], batch_size=B,
                                             clip=None, random_process=noise, noise_clip=0.3, augmenter=aug, aug_mix=1.0,
                                             premade_replay_dicts=rds)
                losses.append(float(logs["losses/critic_overall_loss"]))
                noise.sample(np.zeros(3, np.float32), update_schedule=True)     # the acting path anneals sigma (main.py:350)
            torch.cuda.synchronize()
            captured = sorted(k[0] for k, e in graphed._auto["cache"].items() if any(sl.graph is not None for sl in e.slots))
            assert captured == (["actor", "critic"] if graphs else []), captured    # both entry points really replay graphs
        finally:
            graphed.enable_auto_graphs(False)
        st = e_opt.state[agent.encoder.net.conv2.weight]
        return ([p.detach().clone() for p in chain(agent.encoder.net.parameters(), agent.critics[0].parameters(), agent.actors[0].parameters())],
                losses, float(st["step"]), noise.current_scale)

    eager, le, se, sc_e = run(False)
    graph, lg, sg, sc_g = run(True)
    assert se == sg == 7.0 and sc_e == sc_g and abs(sc_e - 0.37) < 1e-6
    assert le == lg, (le, lg)
    for a, b in zip(eager, graph):
        assert torch.equal(a, b)

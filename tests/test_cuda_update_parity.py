"""GPU parity of the drop-in update functions against the reference's golden vectors (run with -m gpu on a B200).

The same fixtures that pin the oracle (tests/test_oracle_golden.py) are replayed through
super_sac_b200.learning.{critic_update, online_actor_update, alpha_update} + learning_utils.soft_update with the
reference's indices / subsets / eps / noise injected.  Tolerance: north_star's fp32 rtol 1e-4 (plus small atol for
near-zero entries; post-Adam parameters get an atol tied to the learning rate, SURVEY 7.3); Polyak is bit-exact
given equal inputs, so target nets are compared at the same tolerance as the online nets they track.
"""
import numpy as np
import pytest
import torch

import golden_util as gu

pytestmark = pytest.mark.gpu

RTOL = 1e-4


def _cmp_stack(got, want, what, rtol=RTOL, atol=1e-6):
    for n in ("W1", "b1", "W2", "b2", "W3", "b3"):
        gu.assert_close(got[n], want[n], rtol, atol, f"{what}.{n}")


def _cmp_logs(logs, want, what):
    for k, v in want.items():
        k2 = k.replace("|", "/")
        if k2.startswith("gradients/"):
            continue
        assert k2 in logs, f"{what}: missing log key {k2}"
        gu.assert_close(float(logs[k2]), float(v), 2e-4, 2e-5, f"{what} log {k2}")


@pytest.mark.parametrize("impl", ["tcgen05", "ffma"])
@pytest.mark.parametrize("case", gu.UPDATE_CASES)
def test_update_matches_reference(case, impl):
    import cuda_util as cu
    import super_sac_b200 as ssb
    from super_sac_b200 import _rng, augmentations, learning, learning_utils as lu

    ssb.set_mlp_impl(impl)
    fx = gu.load("update_" + case)
    cfg, agent, target = cu.agent_from_fixture(fx)
    E, N, M, B, A = cfg["E"], cfg["N"], cfg["M"], cfg["B"], cfg["A"]
    det = cfg.get("deterministic", False)
    buf = cu.buffer_from_fixture(fx)
    critic_opt, actor_opt, enc_opt, log_alphas, alpha_opts = cu.optimizers(agent, cfg)
    sigma = cfg.get("noise_sigma")
    random_process = None
    if sigma is not None:
        random_process = lu.GaussianExplorationNoise(cu.ActionSpace(A), start_scale=sigma, final_scale=min(sigma, 0.1))
    augmenter = augmentations.AugmentationSequence([augmentations.IdentityAug(B)])
    softmax_w = cfg.get("weight_type") == "softmax" and E > 1

    rec = {}
    o_td, o_bw = lu.compute_td_targets, lu.compute_backup_weights

    def td_rec(*a_, **k_):
        res = o_td(*a_, **k_)
        rec.setdefault("td", []).append(res[0])
        return res

    def bw_rec(*a_, **k_):
        res = o_bw(*a_, **k_)
        rec.setdefault("w", []).append(res)
        return res

    lu.compute_td_targets, lu.compute_backup_weights = td_rec, bw_rec
    old_src = _rng.set_source(_rng.ScriptedSource())
    try:
        replay_dicts = None
        for t in range(cfg["steps"]):
            src = _rng.ScriptedSource()
            _rng.set_source(src)
            r = gu.sub(fx, f"step{t}/rand")
            for i in range(E):
                src.push("indices", r["idx"][i])
                src.push("subsets", r["subsets"][i].astype(np.int32))
                if not det:
                    src.push("normal", r["eps"][i])
                if sigma is not None:
                    src.push("normal", r["noise"][i])
                if softmax_w and not det:
                    for j in range(E):
                        src.push("normal", r["weight_eps"][i][j])
            rec.clear()
            logs, replay_dicts = learning.critic_update(
                buffer=buf, agent=agent, target_agent=target, critic_optimizer=critic_opt, encoder_optimizer=enc_opt,
                log_alphas=log_alphas, batch_size=B, gamma=cfg.get("gamma", 0.99), critic_clip=cfg.get("critic_clip"),
                encoder_clip=cfg.get("encoder_clip"), target_critic_ensemble_n=M,
                weighted_bellman_temp=cfg.get("weight_temp"), weight_type=cfg.get("weight_type"), pop=cfg.get("pop", False),
                augmenter=augmenter, encoder_lambda=0.0, aug_mix=0.0, discrete=False, random_process=random_process,
                noise_clip=cfg.get("noise_clip"), per=False, update_priorities=False, dr3_coeff=cfg.get("dr3_coeff", 0.0))
            assert src.empty(), "not every scripted draw was consumed"
            for i in range(E):
                gu.assert_close(rec["td"][i].cpu().numpy(), fx[f"step{t}/td_target/{i}"], RTOL, 1e-5, f"step{t} td_target[{i}]")
                w = rec["w"][i]
                w = w.cpu().numpy() if torch.is_tensor(w) else np.array(w, dtype=np.float32)
                gu.assert_close(w, fx[f"step{t}/weights/{i}"], RTOL, 1e-5, f"step{t} weights[{i}]")
            _cmp_stack(cu.grads_of(agent._critic_arena), gu.sub(fx, f"step{t}/critic_grads"), f"step{t} critic_grads",
                       rtol=RTOL, atol=2e-7)
            _cmp_logs(logs, gu.sub(fx, f"step{t}/logs"), f"step{t}")
            assert "gradients/critic_random_grad" in logs and "gradients/encoder_criticloss_grad_norm" in logs
            if (t + cfg.get("step0", 0)) % cfg.get("target_delay", 1) == 0:
                for ac, tc in zip(agent.critics, target.critics):
                    lu.soft_update(tc, ac, cfg.get("tau", 0.005))
                lu.soft_update(target.encoder, agent.encoder, cfg.get("encoder_tau", 0.01))
            lr = cfg.get("critic_lr", 3e-4)
            _cmp_stack(cu.stack_of(agent._critic_arena), gu.sub(fx, f"step{t}/critics"), f"step{t} critics", atol=lr * 0.05)
            _cmp_stack(cu.stack_of(target._critic_arena), gu.sub(fx, f"step{t}/target_critics"), f"step{t} target_critics",
                       atol=lr * 0.05)
            want_pop = gu.sub(fx, f"step{t}/popart")
            for i, p in enumerate(agent.popart):
                if not p:
                    continue
                for n in ("mu", "nu", "w", "b"):
                    gu.assert_close(getattr(p, n).cpu().numpy(), want_pop[f"{i}/{n}"], RTOL, 1e-6, f"step{t} popart[{i}].{n}")
                assert int(p._stable) == int(want_pop[f"{i}/stable"])
            if cfg.get("encoder") == "shared":
                want = gu.sub(fx, f"step{t}/encoder")
                for k, v in agent.encoder.state_dict().items():
                    gu.assert_close(v.cpu().numpy(), want[k], RTOL, 1e-4 * 0.05, f"step{t} encoder.{k}")
                want = gu.sub(fx, f"step{t}/target_encoder")
                for k, v in target.encoder.state_dict().items():
                    gu.assert_close(v.cpu().numpy(), want[k], RTOL, 1e-4 * 0.05, f"step{t} target_encoder.{k}")

        # ---- actor update on the last critic batch (reuse_replay_dicts) ----
        src = _rng.ScriptedSource()
        _rng.set_source(src)
        r = gu.sub(fx, "actor/rand")
        for i in range(E):
            src.push("normal", r["eps"][i])
            if sigma is not None:
                src.push("normal", r["noise"][i])
        alogs = learning.online_actor_update(
            buffer=buf, agent=agent, pop=cfg.get("pop", False), actor_optimizer=actor_opt, log_alphas=log_alphas,
            batch_size=B, clip=cfg.get("actor_clip"), random_process=random_process, noise_clip=cfg.get("noise_clip"),
            augmenter=augmenter, aug_mix=0.0, premade_replay_dicts=replay_dicts, per=False, discrete=False,
            use_baseline=False)
        assert src.empty()
        _cmp_stack(cu.grads_of(agent._actor_arena), gu.sub(fx, "actor/grads"), "actor grads", rtol=RTOL, atol=2e-7)
        _cmp_stack(cu.stack_of(agent._actor_arena), gu.sub(fx, "actor/actors"), "actors", atol=3e-4 * 0.05)
        _cmp_logs(alogs, gu.sub(fx, "actor/logs"), "actor")
        if cfg.get("alpha_update", True):
            src = _rng.ScriptedSource()
            _rng.set_source(src)
            r = gu.sub(fx, "alpha/rand")
            if not det:
                for i in range(E):
                    src.push("normal", r["eps"][i])
            llogs = learning.alpha_update(
                buffer=buf, agent=agent, optimizers=alpha_opts, batch_size=B, log_alphas=log_alphas, augmenter=augmenter,
                aug_mix=0.0, target_entropy=-float(A), premade_replay_dicts=replay_dicts, discrete=False)
            for i, la in enumerate(log_alphas):
                gu.assert_close(la.detach().cpu().numpy(), fx[f"alpha/log_alphas/{i}"], 1e-5, 1e-6, f"log_alpha[{i}]")
            _cmp_logs(llogs, gu.sub(fx, "alpha/logs"), "alpha")
    finally:
        lu.compute_td_targets, lu.compute_backup_weights = o_td, o_bw
        _rng.set_source(old_src)
        ssb.set_mlp_impl("tcgen05")


def test_afbc_matches_reference():
    """offline_actor_update (advantage-filtered BC, learning.py:144-219) with prioritised sampling and the priority
    refresh of learning_utils.py:288-295, against the reference's golden vectors (tests/golden/afbc.npz)."""
    import random as pyrandom

    import cuda_util as cu
    import super_sac_b200 as ssb
    from super_sac_b200 import _rng, augmentations, learning, learning_utils as lu, nets

    fx = gu.load("afbc")
    cfg = gu.cfg_of(fx)
    E, N, S, A, H, B = cfg["E"], cfg["N"], cfg["S"], cfg["A"], cfg["H"], cfg["B"]
    agent = ssb.Agent(act_space_size=A, encoder=cu.IdentityEncoder(S), actor_network_cls=nets.mlps.ContinuousStochasticActor,
                      critic_network_cls=nets.mlps.ContinuousCritic, ensemble_size=E, num_critics=N, hidden_size=H,
                      auto_rescale_targets=True, log_std_low=-5.0, log_std_high=2.0)
    agent.to("cuda")
    cu.load_stack(agent._actor_arena, gu.sub(fx, "init/actors"))
    cu.load_stack(agent._critic_arena, gu.sub(fx, "init/critics"))
    pst = gu.sub(fx, "init/popart")
    for i, p in enumerate(agent.popart):
        p.mu, p.nu, p.w, p.b = pst[f"{i}/mu"], pst[f"{i}/nu"], pst[f"{i}/w"], pst[f"{i}/b"]
    b = gu.sub(fx, "buffer")
    buf = ssb.replay.ReplayBuffer(64, alpha=0.6, beta=1.0, device="cuda")
    buf.push({"obs": b["s"]}, b["a"], b["r"][:, None], {"obs": b["s1"]}, b["d"][:, None], priorities=b["priorities"])
    from itertools import chain

    actor_opt = torch.optim.Adam(chain(*(a.parameters() for a in agent.actors)), lr=3e-4, betas=(0.9, 0.999))
    enc_opt = torch.optim.Adam(agent.encoder.parameters(), lr=1e-4)
    augmenter = augmentations.AugmentationSequence([augmentations.IdentityAug(B)])
    old_src = _rng.set_source(_rng.ScriptedSource())
    o_choice = pyrandom.choice
    try:
        for step in range(2):
            r = gu.sub(fx, f"step{step}/rand")
            src = _rng.ScriptedSource()
            _rng.set_source(src)
            for i in range(E):
                src.push("uniform01", r["u"][i])
                for e in r["adv_eps"][i]:
                    src.push("normal", e)
            for e in r["prio_eps"]:
                src.push("normal", e)
            member = int(r["prio_member"])
            pyrandom.choice = lambda seq: (list(seq)[member] if isinstance(seq, range) else o_choice(seq))
            logs = learning.offline_actor_update(
                buffer=buf, agent=agent, actor_optimizer=actor_opt, encoder_optimizer=enc_opt, batch_size=B, actor_clip=40.0,
                update_encoder=False, encoder_clip=40.0, augmenter=augmenter, actor_lambda=0.0, aug_mix=0.0,
                premade_replay_dicts=None, per=True, discrete=False, filter_=True)
            pyrandom.choice = o_choice
            assert src.empty()
            _cmp_stack(cu.grads_of(agent._actor_arena), gu.sub(fx, f"step{step}/actor_grads"), f"step{step} actor grads", atol=2e-7)
            _cmp_stack(cu.stack_of(agent._actor_arena), gu.sub(fx, f"step{step}/actors"), f"step{step} actors", atol=3e-4 * 0.05)
            _cmp_logs(logs, gu.sub(fx, f"step{step}/logs"), f"afbc step{step}")
            tr = gu.sub(fx, f"step{step}/trees")
            gu.assert_close(buf._it_sum.cpu().numpy(), tr["sum_tree"], 1e-4, 1e-8, "sum tree")
            fin = np.isfinite(tr["min_tree"])
            assert np.array_equal(np.isfinite(buf._it_min.cpu().numpy()), fin)
            gu.assert_close(buf._it_min.cpu().numpy()[fin], tr["min_tree"][fin], 1e-4, 1e-8, "min tree")
            assert abs(buf._max_priority - float(tr["max_priority"])) <= 1e-4 * float(tr["max_priority"])
    finally:
        pyrandom.choice = o_choice
        _rng.set_source(old_src)


def test_pixel_critic_update_matches_oracle():
    """BASELINE config 4 in miniature: uint8 frames in the device ring, fused gather + DrQ (v1, exact) shift, a conv
    encoder (user plugin, PyTorch/cuDNN) trained through grad(s_rep), deterministic actor + TD3 noise, n-step gamma.
    Checked against the CPU oracle on the same draws (the encoder runs in PyTorch on both sides)."""
    import copy

    import cuda_util as cu
    import super_sac_b200 as ssb
    from oracle import aug_oracle as ao
    from oracle import update_oracle as uo
    from super_sac_b200 import _rng, augmentations, learning, learning_utils as lu, nets

    class TinyPixelEncoder(nets.Encoder):
        def __init__(self, c, hw, out_dim=10):
            super().__init__()
            self.conv1 = torch.nn.Conv2d(c, 8, 3, stride=2)
            self.conv2 = torch.nn.Conv2d(8, 8, 3, stride=1)
            n = ((hw - 3) // 2 + 1) - 2
            self.fc = torch.nn.Linear(8 * n * n, out_dim)
            self.ln = torch.nn.LayerNorm(out_dim)
            self._dim = out_dim

        @property
        def embedding_dim(self):
            return self._dim

        def forward(self, obs):
            x = obs["pixels"] / 255.0 - 0.5
            x = torch.relu(self.conv2(torch.relu(self.conv1(x))))
            return torch.tanh(self.ln(self.fc(x.flatten(1))))

    rng = np.random.default_rng(5)
    torch.manual_seed(5)
    C, HW, A, Hd, B, nbuf, N = 3, 20, 3, 64, 16, 40, 2
    enc = TinyPixelEncoder(C, HW)
    agent = ssb.Agent(act_space_size=A, encoder=enc, actor_network_cls=nets.mlps.ContinuousDeterministicActor,
                      critic_network_cls=nets.mlps.ContinuousCritic, ensemble_size=1, num_critics=N, hidden_size=Hd,
                      auto_rescale_targets=False)
    for arena in (agent._actor_arena, agent._critic_arena):
        arena.flat.add_(0.02 * torch.randn_like(arena.flat))
    # oracle twin (CPU) before anything moves
    o_agent = uo.OracleAgent(1, N, enc.embedding_dim, A, Hd, deterministic=True, encoder=copy.deepcopy(enc))
    for n in uo.PARAM_NAMES:
        getattr(o_agent.actors, n).copy_(agent._actor_arena.p[n])
        getattr(o_agent.critics, n).copy_(agent._critic_arena.p[n])
    o_target = o_agent.clone()
    agent.to("cuda")
    target = copy.deepcopy(agent)
    s = rng.integers(0, 256, (nbuf, C, HW, HW), dtype=np.uint8)
    s1 = rng.integers(0, 256, (nbuf, C, HW, HW), dtype=np.uint8)
    a = rng.uniform(-1, 1, (nbuf, A)).astype(np.float32)
    r = rng.standard_normal(nbuf).astype(np.float32)
    d = rng.uniform(size=nbuf) < 0.1
    buf = ssb.replay.ReplayBuffer(nbuf, device="cuda")
    buf.load_experience({"pixels": s}, a, r, {"pixels": s1}, d)
    from itertools import chain

    critic_opt = torch.optim.Adam(chain(*(c.parameters() for c in agent.critics)), lr=1e-4)
    enc_opt = torch.optim.Adam(agent.encoder.parameters(), lr=1e-4)
    o_opt = uo.Adam(o_agent.critics.tensors(), lr=1e-4)
    o_enc_opt = torch.optim.Adam(o_agent.encoder.parameters(), lr=1e-4)
    log_alphas = [torch.tensor([-30.0], device="cuda", requires_grad=True)]
    noise_proc = lu.GaussianExplorationNoise(cu.ActionSpace(A), start_scale=0.6, final_scale=0.1)
    augmenter = augmentations.AugmentationSequence([augmentations.DrqNoNoiseAug(B)])
    gamma = 0.99**3
    old_src = _rng.set_source(_rng.ScriptedSource())
    try:
        for step in range(2):
            idx = rng.integers(0, nbuf, B)
            shift = rng.integers(0, 8, (B, 2))
            noise = rng.standard_normal((B, A)).astype(np.float32)
            subset = rng.permutation(N)[:2]
            src = _rng.ScriptedSource()
            _rng.set_source(src)
            src.push("indices", idx).push("shifts", shift.astype(np.int32)).push("normal", noise).push("subsets", subset.astype(np.int32))
            logs, _ = learning.critic_update(
                buffer=buf, agent=agent, target_agent=target, critic_optimizer=critic_opt, encoder_optimizer=enc_opt,
                log_alphas=log_alphas, batch_size=B, gamma=gamma, critic_clip=None, encoder_clip=None,
                target_critic_ensemble_n=2, weighted_bellman_temp=None, weight_type=None, pop=False, augmenter=augmenter,
                encoder_lambda=0.0, random_process=noise_proc, noise_clip=0.3, aug_mix=1.0)
            assert src.empty()
            for ac, tc in zip(agent.critics, target.critics):
                lu.soft_update(tc, ac, 0.01)
            lu.soft_update(target.encoder, agent.encoder, 1.0)
            # oracle on the same draws
            t32 = lambda x: torch.as_tensor(np.asarray(x, dtype=np.float32))
            o = {"pixels": t32(ao.drq_v1_crop(s[idx], shift[:, 0], shift[:, 1]))}
            o1 = {"pixels": t32(ao.drq_v1_crop(s1[idx], shift[:, 0], shift[:, 1]))}
            batch = (o, t32(a[idx]), t32(r[idx]).reshape(-1, 1), o1, t32(d[idx]).reshape(-1, 1))
            hp = dict(gamma=gamma, noise_sigma=0.6, noise_clip=0.3)
            ologs, aux = uo.critic_update(o_agent, o_target, [batch], [dict(eps=None, noise=t32(noise), subset=[int(x) for x in subset])],
                                          hp, [torch.tensor([-30.0])], o_opt, o_enc_opt)
            uo.soft_update(o_target.critics.tensors(), o_agent.critics.tensors(), 0.01)
            uo.soft_update([p.data for p in o_target.encoder.parameters()], [p.data for p in o_agent.encoder.parameters()], 1.0)
            for n in uo.PARAM_NAMES:
                gu.assert_close(agent._critic_arena.g[n].cpu().numpy(), getattr(aux["grads"], n).numpy(), 2e-4, 2e-6, f"step{step} grad {n}")
                gu.assert_close(agent._critic_arena.p[n].cpu().numpy(), getattr(o_agent.critics, n).numpy(), 1e-4, 1e-4 * 0.05, f"step{step} critics {n}")
                gu.assert_close(target._critic_arena.p[n].cpu().numpy(), getattr(o_target.critics, n).numpy(), 1e-4, 1e-4 * 0.05, f"step{step} target {n}")
            for (k, v), (_, w) in zip(agent.encoder.state_dict().items(), o_agent.encoder.state_dict().items()):
                gu.assert_close(v.cpu().numpy(), w.numpy(), 2e-4, 1e-4 * 0.05, f"step{step} encoder {k}")
            for v, w in zip(target.encoder.parameters(), agent.encoder.parameters()):
                assert torch.equal(v, w)  # encoder_tau = 1.0 is a copy
            gu.assert_close(logs["losses/critic_overall_loss"], ologs["losses/critic_overall_loss"], 2e-4, 1e-6, "loss")
    finally:
        _rng.set_source(old_src)


def test_sharded_update_equals_single_gpu():
    """SURVEY §8e: critics sharded over 2 GPUs (NCCL all-gather of target Q / Q(s,pi), all-reduce of dL/da) give the
    single-GPU result.  Needs 2 GPUs on the box (skipped otherwise); the host logic is covered on CPU by
    tests/test_parallel_gloo.py."""
    import os
    import subprocess
    import sys

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29517", os.path.join(root, "tests", "dist_sharded_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "[rank 0] sharded critics" in res.stdout and "[rank 1] sharded critics" in res.stdout
    assert "[rank 0] sharded members" in res.stdout and "[rank 1] sharded members" in res.stdout   # SUNRISE, C3


def test_auto_graph_replay_equals_eager():
    """graphed.enable_auto_graphs(): from the third identical call on, critic_update / online_actor_update replay a
    captured CUDA graph.  Same Philox seed => the replayed run must reproduce the eager run bit for bit (same kernels,
    device-side step / rng counters), and return the same log keys."""
    import copy
    from itertools import chain

    import cuda_util as cu
    import super_sac_b200 as ssb
    from super_sac_b200 import augmentations, graphed, learning, learning_utils as lu, nets

    def run(auto):
        ssb.manual_seed(11)
        torch.manual_seed(11)
        agent = ssb.Agent(act_space_size=6, encoder=cu.IdentityEncoder(17), actor_network_cls=nets.mlps.ContinuousStochasticActor,
                          critic_network_cls=nets.mlps.ContinuousCritic, ensemble_size=1, num_critics=4, hidden_size=64,
                          auto_rescale_targets=False, log_std_low=-5.0, log_std_high=2.0)
        agent.to("cuda")
        target = copy.deepcopy(agent)
        rng = np.random.default_rng(0)
        buf = ssb.replay.ReplayBuffer(2048, device="cuda")
        buf.load_experience({"obs": rng.standard_normal((2048, 17), dtype=np.float32)}, rng.uniform(-1, 1, (2048, 6)).astype(np.float32),
                            rng.standard_normal(2048, dtype=np.float32), {"obs": rng.standard_normal((2048, 17), dtype=np.float32)},
                            rng.uniform(size=2048) < 0.05)
        c_opt = torch.optim.Adam(chain(*(c.parameters() for c in agent.critics)), lr=3e-4)
        a_opt = torch.optim.Adam(chain(*(a.parameters() for a in agent.actors)), lr=3e-4)
        e_opt = torch.optim.Adam(agent.encoder.parameters(), lr=1e-4)
        la = [torch.tensor([-2.3], device="cuda", requires_grad=True)]
        aug = augmentations.AugmentationSequence([augmentations.IdentityAug(64)])
        graphed.enable_auto_graphs(auto)
        try:
            for k in range(7):
                logs, rds = learning.critic_update(
                    buffer=buf, agent=agent, target_agent=target, critic_optimizer=c_opt, encoder_optimizer=e_opt, log_alphas=la,
                    batch_size=64, gamma=0.99, critic_clip=None, encoder_clip=None, target_critic_ensemble_n=2,
                    weighted_bellman_temp=None, weight_type=None, pop=False, augmenter=aug, encoder_lambda=0.0,
                    random_process=None, noise_clip=None, aug_mix=0.0)
                if k % 2 == 0:
                    lu.soft_update(target.critics[0], agent.critics[0], 0.005)
                alogs = learning.online_actor_update(
                    buffer=buf, agent=agent, pop=False, actor_optimizer=a_opt, log_alphas=la, batch_size=64, clip=None,
                    random_process=None, noise_clip=None, augmenter=aug, aug_mix=0.0, premade_replay_dicts=rds)
        finally:
            graphed.enable_auto_graphs(False)
        assert c_opt._ssac_flat_adam.steps == 7 and int(c_opt._ssac_flat_adam.ctl[0]) == 7
        assert buf.total_sample_calls == 7
        return agent, target, logs, alogs

    a0, t0, l0, al0 = run(False)
    a1, t1, l1, al1 = run(True)
    assert torch.equal(a0._critic_arena.flat, a1._critic_arena.flat)
    assert torch.equal(t0._critic_arena.flat, t1._critic_arena.flat)
    assert torch.equal(a0._actor_arena.flat, a1._actor_arena.flat)
    assert set(l0.keys()) == set(l1.keys()) and set(al0.keys()) == set(al1.keys())
    for k in l0:
        gu.assert_close(float(l1[k]), float(l0[k]), 1e-5, 1e-7, f"log {k}")


@pytest.mark.parametrize("shape", [(4, 64, 64), (10, 256, 256)], ids=["small", "redq"])
def test_cross_call_pipelined_updates_equal_eager(shape):
    """graphed.enable_auto_graphs(pipeline=True): consecutive critic_update calls overlap on the device (two alternating
    captures on two streams, ordered by external event nodes), with a buffer.push before every update, a Polyak step after
    every second one and an actor + temperature update every fifth -- exactly the calls a training loop makes.  Same Philox
    seed => bit-identical parameters and replay ring, same logged scalars as the eager run."""
    import copy
    from itertools import chain

    import cuda_util as cu
    import super_sac_b200 as ssb
    from super_sac_b200 import augmentations, graphed, learning, learning_utils as lu, nets

    N, H, B = shape
    steps = 23

    def run(mode):
        ssb.manual_seed(13)
        torch.manual_seed(13)
        agent = ssb.Agent(act_space_size=6, encoder=cu.IdentityEncoder(17), actor_network_cls=nets.mlps.ContinuousStochasticActor,
                          critic_network_cls=nets.mlps.ContinuousCritic, ensemble_size=1, num_critics=N, hidden_size=H,
                          auto_rescale_targets=False, log_std_low=-5.0, log_std_high=2.0)
        agent.to("cuda")
        target = copy.deepcopy(agent)
        rng = np.random.default_rng(0)
        n = 512   # small ring: pushes wrap around and overwrite rows that are being sampled
        buf = ssb.replay.ReplayBuffer(n, device="cuda")
        buf.load_experience({"obs": rng.standard_normal((n - 7, 17), dtype=np.float32)}, rng.uniform(-1, 1, (n - 7, 6)).astype(np.float32),
                            rng.standard_normal(n - 7, dtype=np.float32), {"obs": rng.standard_normal((n - 7, 17), dtype=np.float32)},
                            rng.uniform(size=n - 7) < 0.05)
        c_opt = torch.optim.Adam(chain(*(c.parameters() for c in agent.critics)), lr=3e-4)
        a_opt = torch.optim.Adam(chain(*(a.parameters() for a in agent.actors)), lr=3e-4)
        e_opt = torch.optim.Adam(agent.encoder.parameters(), lr=1e-4)
        la = [torch.tensor([-2.3], device="cuda", requires_grad=True)]
        al_opt = [torch.optim.Adam([la[0]], lr=1e-4, betas=(0.5, 0.999))]
        aug = augmentations.AugmentationSequence([augmentations.IdentityAug(B)])
        tr = np.random.default_rng(1)
        graphed.enable_auto_graphs(mode != "eager", pipeline=(mode == "pipeline"))
        all_logs = []
        try:
            for k in range(steps):
                buf.push({"obs": tr.standard_normal(17, dtype=np.float32)}, tr.uniform(-1, 1, 6).astype(np.float32), float(tr.standard_normal()),
                         {"obs": tr.standard_normal(17, dtype=np.float32)}, bool(tr.uniform() < 0.1))
                logs, rds = learning.critic_update(
                    buffer=buf, agent=agent, target_agent=target, critic_optimizer=c_opt, encoder_optimizer=e_opt, log_alphas=la,
                    batch_size=B, gamma=0.99, critic_clip=None, encoder_clip=None, target_critic_ensemble_n=2,
                    weighted_bellman_temp=None, weight_type=None, pop=False, augmenter=aug, encoder_lambda=0.0,
                    random_process=None, noise_clip=None, aug_mix=0.0)
                all_logs.append(logs)
                if k % 2 == 0:
                    lu.soft_update(target.critics[0], agent.critics[0], 0.005)
                if k % 5 == 4:
                    learning.online_actor_update(
                        buffer=buf, agent=agent, pop=False, actor_optimizer=a_opt, log_alphas=la, batch_size=B, clip=None,
                        random_process=None, noise_clip=None, augmenter=aug, aug_mix=0.0, premade_replay_dicts=rds)
                    learning.alpha_update(buffer=buf, agent=agent, optimizers=al_opt, batch_size=B, log_alphas=la, augmenter=aug,
                                          aug_mix=0.0, target_entropy=-6.0, premade_replay_dicts=rds, discrete=False)
            all_logs = [dict(l) for l in all_logs]   # (lazy logs resolve here)
            graphed.join()
            torch.cuda.synchronize()
        finally:
            graphed.enable_auto_graphs(False)
        assert c_opt._ssac_flat_adam.steps == steps and int(c_opt._ssac_flat_adam.ctl[0]) == steps
        return agent, target, la, buf, all_logs

    a0, t0, la0, b0, l0 = run("eager")
    a1, t1, la1, b1, l1 = run("pipeline")
    assert torch.equal(a0._critic_arena.flat, a1._critic_arena.flat)
    assert torch.equal(t0._critic_arena.flat, t1._critic_arena.flat)
    assert torch.equal(a0._actor_arena.flat, a1._actor_arena.flat)
    assert torch.equal(la0[0], la1[0])
    assert torch.equal(b0._storage.s_stack["obs"], b1._storage.s_stack["obs"])
    for k, (x, y) in enumerate(zip(l0, l1)):
        assert set(x.keys()) == set(y.keys())
        for key in x:
            if key.startswith("gradients/"):
                continue   # the logged member is a host-side random.choice (frozen at capture)
            gu.assert_close(float(y[key]), float(x[key]), 1e-5, 1e-7, f"step {k} log {key}")


@pytest.mark.parametrize("captured,pop", [(False, False), (True, False), (False, True), (True, True)],
                         ids=["eager", "graph", "eager-popart", "graph-popart"])
def test_pipelined_update_block_equals_sequential(captured, pop):
    """lu.pipelined_updates(): the target side of update k+1 runs next to update k's backward / Adam on its own stream.
    Same kernels, same draw order, event-ordered where data flows => a block of UTD updates (+ Polyak every 2nd, + one
    actor and one temperature update, as main.py:380-543 runs them) must reproduce the sequential schedule bit for bit.
    With PopArt the critic updates take the serial schedule inside the block (the next TD target rescales the PopArt
    layer this update's loss seed still reads)."""
    import copy
    from itertools import chain

    import cuda_util as cu
    import super_sac_b200 as ssb
    from super_sac_b200 import augmentations, graphed, learning, learning_utils as lu, nets

    def build():
        ssb.manual_seed(5)
        torch.manual_seed(5)
        agent = ssb.Agent(act_space_size=6, encoder=cu.IdentityEncoder(17), actor_network_cls=nets.mlps.ContinuousStochasticActor,
                          critic_network_cls=nets.mlps.ContinuousCritic, ensemble_size=1, num_critics=10, hidden_size=256,
                          auto_rescale_targets=pop, log_std_low=-5.0, log_std_high=2.0)
        agent.to("cuda")
        target = copy.deepcopy(agent)
        rng = np.random.default_rng(0)
        n = 4096
        buf = ssb.replay.ReplayBuffer(n, device="cuda")
        buf.load_experience({"obs": rng.standard_normal((n, 17), dtype=np.float32)}, rng.uniform(-1, 1, (n, 6)).astype(np.float32),
                            rng.standard_normal(n, dtype=np.float32), {"obs": rng.standard_normal((n, 17), dtype=np.float32)},
                            rng.uniform(size=n) < 0.05)
        c_opt = torch.optim.Adam(chain(*(c.parameters() for c in agent.critics)), lr=3e-4)
        a_opt = torch.optim.Adam(chain(*(a.parameters() for a in agent.actors)), lr=3e-4)
        e_opt = torch.optim.Adam(agent.encoder.parameters(), lr=1e-4)
        la = [torch.tensor([-2.3], device="cuda", requires_grad=True)]
        al_opt = [torch.optim.Adam([la[0]], lr=1e-4, betas=(0.5, 0.999))]
        aug = augmentations.AugmentationSequence([augmentations.IdentityAug(256)])

        def block(pipelined):
            ctx = lu.pipelined_updates() if pipelined else contextlib.nullcontext()
            with ctx:
                for k in range(6):
                    logs, rds = learning._critic_update_impl(
                        buffer=buf, agent=agent, target_agent=target, critic_optimizer=c_opt, encoder_optimizer=e_opt,
                        log_alphas=la, batch_size=256, gamma=0.99, critic_clip=None, encoder_clip=None,
                        target_critic_ensemble_n=2, weighted_bellman_temp=None, weight_type=None, pop=pop, augmenter=aug,
                        encoder_lambda=0.0, random_process=None, noise_clip=None, aug_mix=0.0)
                    if k % 2 == 0:
                        lu.soft_update(target.critics[0], agent.critics[0], 0.005)
                learning._online_actor_update_impl(
                    buffer=buf, agent=agent, pop=pop, actor_optimizer=a_opt, log_alphas=la, batch_size=256, clip=None,
                    random_process=None, noise_clip=None, augmenter=aug, aug_mix=0.0, premade_replay_dicts=rds)
                learning.alpha_update(buffer=buf, agent=agent, optimizers=al_opt, batch_size=256, log_alphas=la, augmenter=aug,
                                      aug_mix=0.0, target_entropy=-6.0, premade_replay_dicts=rds, discrete=False)
            return logs

        return agent, target, la, block

    import contextlib

    a0, t0, la0, block0 = build()
    for _ in range(5):
        l0 = block0(False)
    l0 = dict(l0.fetch(keep=True)) if hasattr(l0, "fetch") else dict(l0)
    a1, t1, la1, block1 = build()
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
    assert torch.equal(a0._critic_arena.flat, a1._critic_arena.flat)
    assert torch.equal(t0._critic_arena.flat, t1._critic_arena.flat)
    assert torch.equal(a0._actor_arena.flat, a1._actor_arena.flat)
    assert torch.equal(la0[0], la1[0])
    for p0, p1 in zip(a0.popart, a1.popart):
        assert bool(p0) == bool(p1) == pop
        if pop:
            assert torch.equal(p0._state, p1._state) and torch.equal(p0._ctl, p1._ctl)
    assert set(l0.keys()) == set(l1.keys())
    for k in l0:
        gu.assert_close(float(l1[k]), float(l0[k]), 1e-5, 1e-7, f"log {k}")


def test_module_views_and_kernels_agree_on_the_acting_path():
    """The nn.Modules the reference API exposes (Agent.forward / sample_action, critics[i](s, a)) are views into the
    parameter arenas the kernels read: after a fused update both must see the same parameters, and the PyTorch forward of
    the modules must equal the kernel forward (SURVEY 8f N1: acting path)."""
    import cuda_util as cu
    import super_sac_b200 as ssb
    from super_sac_b200 import learning_utils as lu, nets

    torch.manual_seed(3)
    S, A, H, N, B = 17, 6, 256, 10, 64
    agent = ssb.Agent(act_space_size=A, encoder=cu.IdentityEncoder(S), actor_network_cls=nets.mlps.ContinuousStochasticActor,
                      critic_network_cls=nets.mlps.ContinuousCritic, ensemble_size=1, num_critics=N, hidden_size=H,
                      auto_rescale_targets=False, log_std_low=-5.0, log_std_high=2.0)
    agent.to(ssb.device)
    dev = agent._critic_arena.device
    with torch.no_grad():   # perturb through the arena, read through the modules
        agent._critic_arena.flat.mul_(1.5)
        agent._actor_arena.flat.add_(0.01)
    s = torch.randn(B, S, device=dev)
    a = torch.rand(B, A, device=dev) * 2 - 1
    with torch.no_grad():
        q_mod = torch.stack([net(s, a) for net in agent.critics[0].nets], dim=0)          # PyTorch path, [N,B,1]
        mu_mod = agent.actors[0](s).mean                                                   # tanh(mu)
    X = torch.cat((s, a), dim=1).contiguous()
    q_ker = lu._critic_values(agent, 0, N, X, B)
    gu.assert_close(q_ker.cpu().numpy(), q_mod.cpu().numpy(), 1e-4, 2e-5, "critics: kernel vs nn.Module")
    out, _, _ = lu._actor_forward(agent, 0, X, B, S, A)
    gu.assert_close(torch.tanh(out[0, :, :A]).cpu().numpy(), mu_mod.cpu().numpy(), 1e-4, 2e-5, "actor mean: kernel vs nn.Module")
    obs = {"obs": s[0].cpu().numpy()}
    act = agent.forward(obs)
    assert act.shape == (A,) and np.all(np.abs(act) <= 1.0)
    gu.assert_close(act, mu_mod[0].cpu().numpy(), 1e-4, 2e-5, "Agent.forward")
    smp = agent.sample_action(obs)
    assert smp.shape == (A,) and np.all(np.abs(smp) <= 1.0)

"""SAC-Discrete ensembles sharded over two ranks, on CPU: a world-2 gloo group whose ranks each run
super_sac_b200.discrete UNCHANGED on CPU tensors against the numpy emulation of the C ABI (tests/emulated_abi.py, as in
tests/test_discrete_host.py).  The exchanges fall back to torch.distributed collectives.  Every rank must reproduce the
golden vectors of the unmodified reference for the nets and members it owns, and the replicated state (actor,
temperature, PopArt) must be equal on both ranks.

- ``critics``: update_discrete_sac, N = 3 critics over 2 ranks (2 + 1), DR3 (the golden's clip of 40 does not engage).
- ``members``: update_discrete_sunrise_popart, 2 members over 2 ranks, sunrise weights and PopArt.
- ``offline``: the discrete_afbc golden (filtered BC, indirect advantage, priority refresh, filter statistics), critics
  sharded, with Python's ``random`` seeded differently on each rank.
- ``offline-members``: the discrete_afbc golden, one member per rank (the filter's mean policy over every rank's actors).
- ``clip``: global-norm clipping where it engages (clip 1e-3), sharded against the unsharded update on the same draws.
"""
import os
import socket
import traceback

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

RTOL = 1e-4


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _emulate():
    """The fixture of test_discrete_host.py, for a spawned rank (which ends with its case)."""
    from emulated_abi import EmulatedLib
    from super_sac_b200 import _lib, _logs, _ops

    emu = EmulatedLib()
    _lib._lib = emu
    _lib.stream_ptr = lambda: 0
    _ops.check_cuda = lambda *t: None
    torch.cuda.is_current_stream_capturing = lambda: False

    def fetch(self, keep=False, synced=False):
        host = self._buf[: self._n].tolist()
        for key, slot, transform in self._pending:
            if isinstance(transform, _logs._Multi):
                self[key] = transform.fn(*[host[s_] for s_ in slot])
                continue
            val = sum(host[s_] for s_ in slot) if isinstance(slot, (list, tuple)) else host[slot]
            self[key] = transform(val) if transform is not None else val
        self._pending = []
        return self

    _logs.DeviceLogs.fetch = fetch
    return emu


def _cmp_logs(logs, want, what, keep):
    """Every golden key that ``keep(key)`` selects must be logged with the golden value (gradient norms: present)."""
    import golden_util as gu

    for k, v in want.items():
        k2 = k.replace("|", "/")
        if not keep(k2):
            continue
        assert k2 in logs, f"{what}: missing log key {k2}"
        if not k2.startswith("gradients/"):
            gu.assert_close(float(logs[k2]), float(v), 2e-4, 2e-5, f"{what} log {k2}")


def _member_of(key):
    """The member a per-member log key belongs to (``..._<i>``), else None."""
    tail = key.rsplit("_", 1)[-1]
    return int(tail) if tail.isdigit() else None


def _same_on_all_ranks(t, what):
    t = t.detach().reshape(-1).clone()
    lst = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(lst, t)
    assert all(torch.equal(x, lst[0]) for x in lst), f"{what} differs between ranks"


def _agent(fx, E, N, popart):
    import golden_util as gu
    import super_sac_b200 as ssb
    from super_sac_b200 import nets
    from test_discrete_host import IdentityEncoder

    cfg = gu.cfg_of(fx)
    return ssb.Agent(act_space_size=cfg["A"], encoder=IdentityEncoder(cfg["S"]), actor_network_cls=nets.mlps.DiscreteActor,
                     critic_network_cls=nets.mlps.DiscreteCritic, discrete=True, ensemble_size=E, num_critics=N,
                     hidden_size=cfg["H"], auto_rescale_targets=popart)


def _rows_of(d, rows):
    return {k: v[rows] for k, v in d.items()}


def _sampler(bufd, S):
    """sample_move_and_augment over the golden buffer: the scripted indices, the packed [s | a] state batch."""
    from super_sac_b200 import _rng, learning_utils as lu

    def fake_sample(buffer, batch_size, augmenter, aug_mix, per=True, _idx=None):
        idx = torch.empty(batch_size, dtype=torch.int64)
        _rng.source().indices(idx, len(bufd["a"]))
        ix = idx.numpy()
        XA = torch.as_tensor(np.concatenate([bufd["s"][ix], bufd["a"][ix]], 1).astype(np.float32))
        X1 = torch.as_tensor(np.concatenate([bufd["s1"][ix], np.zeros((batch_size, 1), np.float32)], 1))
        rd = lu.ReplayDict()
        rd["primary_batch"] = ({"obs": XA[:, :S]}, XA[:, S:], torch.as_tensor(bufd["r"][ix]).reshape(-1, 1),
                               {"obs": X1[:, :S]}, torch.as_tensor(bufd["d"][ix]).reshape(-1, 1))
        rd["priority_idxs"], rd["imp_weights"] = idx, torch.ones(1)
        return rd

    return fake_sample


def _update_case(case, rank):
    """update_discrete_sac (critics sharded) or update_discrete_sunrise_popart (members sharded): the critic updates of
    every golden step, then the actor and the temperature update, as test_discrete_host runs them."""
    import copy
    import math
    from itertools import chain

    import golden_util as gu
    from super_sac_b200 import _rng, augmentations, learning, learning_utils as lu, parallel
    from test_discrete_host import _cmp_stack, _load_stack

    fx = gu.load("update_" + case)
    cfg = gu.cfg_of(fx)
    Eg, Ng, M, S, B = cfg["E"], cfg["N"], cfg["M"], cfg["S"], cfg["B"]
    if case == "discrete_sac":
        lo, hi = parallel.enable_critic_sharding(Ng)
        members, nets_ = [0], np.arange(lo, hi)                  # E = 1: nets [lo, hi) of the one member
        E, N, last = 1, hi - lo, hi == Ng
    else:
        lo, hi = parallel.enable_member_sharding(Eg)
        members, nets_ = list(range(lo, hi)), np.arange(lo * Ng, hi * Ng)
        E, N, last = hi - lo, Ng, hi == Eg
    agent = _agent(fx, E, N, cfg.get("popart", False))
    _load_stack(agent._actor_arena, _rows_of(gu.sub(fx, "init/actors"), members))
    _load_stack(agent._critic_arena, _rows_of(gu.sub(fx, "init/critics"), nets_))
    pst = gu.sub(fx, "init/popart")
    for i, p in enumerate(agent.popart):
        if p:
            g = members[i]
            p.mu, p.nu, p.w, p.b = pst[f"{g}/mu"], pst[f"{g}/nu"], pst[f"{g}/w"], pst[f"{g}/b"]
            p._t = int(pst[f"{g}/t"])
    target = copy.deepcopy(agent)
    _load_stack(target._critic_arena, _rows_of(gu.sub(fx, "init/target_critics"), nets_))
    critic_opt = torch.optim.Adam(chain(*(c.parameters() for c in agent.critics)), lr=3e-4, betas=(0.9, 0.999))
    actor_opt = torch.optim.Adam(chain(*(a.parameters() for a in agent.actors)), lr=3e-4, betas=(0.9, 0.999))
    enc_opt = torch.optim.Adam(agent.encoder.parameters(), lr=1e-4)
    log_alphas, alpha_opts = [], []
    for _ in range(E):
        la = torch.Tensor([math.log(cfg.get("init_alpha", 0.1))])
        la.requires_grad = True
        log_alphas.append(la)
        alpha_opts.append(torch.optim.Adam([la], lr=1e-4, betas=(0.5, 0.999)))
    augmenter = augmentations.AugmentationSequence([augmentations.IdentityAug(B)])
    bufd = gu.sub(fx, "buffer")

    lu.sample_move_and_augment = _sampler(bufd, S)
    rec = {}
    o_td, o_bw = lu.compute_td_targets, lu.compute_backup_weights
    lu.compute_td_targets = lambda *a, **k: rec.setdefault("td", []).append(o_td(*a, **k)) or rec["td"][-1]
    lu.compute_backup_weights = lambda *a, **k: rec.setdefault("w", []).append(o_bw(*a, **k)) or rec["w"][-1]

    def mine(key):   # per-member keys of the members this rank owns; the sunrise weights of the last member
        m = _member_of(key)
        if key.startswith("bellman_weights/"):
            return last
        return m is None or m in members

    replay_dicts = None
    for t in range(cfg["steps"]):
        src = _rng.ScriptedSource()
        _rng.set_source(src)
        r = gu.sub(fx, f"step{t}/rand")
        for g in members:
            src.push("indices", r["idx"][g])
            src.push("subsets", r["subsets"][g].astype(np.int32))
        rec.clear()
        logs, replay_dicts = learning.critic_update(
            buffer=None, agent=agent, target_agent=target, critic_optimizer=critic_opt, encoder_optimizer=enc_opt,
            log_alphas=log_alphas, batch_size=B, gamma=cfg.get("gamma", 0.99), critic_clip=cfg.get("critic_clip"),
            encoder_clip=cfg.get("encoder_clip"), target_critic_ensemble_n=M, weighted_bellman_temp=cfg.get("weight_temp"),
            weight_type=cfg.get("weight_type"), pop=cfg.get("pop", False), augmenter=augmenter, encoder_lambda=0.0,
            aug_mix=0.0, discrete=True, random_process=None, noise_clip=None, per=False, update_priorities=False,
            dr3_coeff=cfg.get("dr3_coeff", 0.0))
        assert src.empty(), "not every scripted draw was consumed"
        for i, g in enumerate(members):
            gu.assert_close(rec["td"][i][0].numpy(), fx[f"step{t}/td_target/{g}"], RTOL, 1e-5, f"step{t} td_target[{g}]")
            w = rec["w"][i]
            w = w.numpy() if torch.is_tensor(w) else np.array(w, dtype=np.float32)
            gu.assert_close(w, fx[f"step{t}/weights/{g}"], RTOL, 1e-5, f"step{t} weights[{g}]")
            if case == "discrete_sac":
                _same_on_all_ranks(rec["td"][i][0], f"step{t} td_target[{g}]")
        _cmp_stack(agent._critic_arena.g, _rows_of(gu.sub(fx, f"step{t}/critic_grads"), nets_), f"step{t} critic_grads",
                   atol=2e-7)
        _cmp_logs(logs, gu.sub(fx, f"step{t}/logs"), f"step{t}", mine)
        with torch.no_grad():
            tf, sf = target._critic_arena.flat, agent._critic_arena.flat
            tf.copy_(tf * (1.0 - cfg.get("tau", 0.005)) + sf * cfg.get("tau", 0.005))
        _cmp_stack(agent._critic_arena.p, _rows_of(gu.sub(fx, f"step{t}/critics"), nets_), f"step{t} critics",
                   atol=3e-4 * 0.05)
        want_pop = gu.sub(fx, f"step{t}/popart")
        for i, p in enumerate(agent.popart):
            if p:
                for n in ("mu", "nu", "w", "b"):
                    gu.assert_close(getattr(p, n).numpy(), want_pop[f"{members[i]}/{n}"], RTOL, 1e-6,
                                    f"step{t} popart[{members[i]}].{n}")
    alogs = learning.online_actor_update(
        buffer=None, agent=agent, pop=cfg.get("pop", False), actor_optimizer=actor_opt, log_alphas=log_alphas,
        batch_size=B, clip=cfg.get("actor_clip"), random_process=None, noise_clip=None, augmenter=augmenter, aug_mix=0.0,
        premade_replay_dicts=replay_dicts, per=False, discrete=True, use_baseline=False)
    _cmp_stack(agent._actor_arena.g, _rows_of(gu.sub(fx, "actor/grads"), members), "actor grads", atol=2e-7)
    _cmp_stack(agent._actor_arena.p, _rows_of(gu.sub(fx, "actor/actors"), members), "actors", atol=3e-4 * 0.05)
    _cmp_logs(alogs, gu.sub(fx, "actor/logs"), "actor", mine)
    llogs = learning.alpha_update(
        buffer=None, agent=agent, optimizers=alpha_opts, batch_size=B, log_alphas=log_alphas, augmenter=augmenter,
        aug_mix=0.0, target_entropy=float(fx["alpha/target_entropy"]), premade_replay_dicts=replay_dicts, discrete=True)
    for i, la in enumerate(log_alphas):
        gu.assert_close(la.detach().numpy(), fx[f"alpha/log_alphas/{members[i]}"], 1e-6, 1e-7, f"log_alpha[{members[i]}]")
    _cmp_logs(llogs, gu.sub(fx, "alpha/logs"), "alpha", mine)
    if case == "discrete_sac":   # replicated state: the same bits on every rank
        _same_on_all_ranks(agent._actor_arena.flat, "actor")
        _same_on_all_ranks(log_alphas[0], "log_alpha")
        # (the logged gradient norm is each rank's own critics', as in the continuous path)
        _same_on_all_ranks(torch.tensor([float(logs[k]) for k in sorted(logs) if not k.startswith("gradients/")]),
                           "critic logs")
    return lo, hi


def _clip_case(rank):
    """Global-norm clipping under critic sharding where it engages: the update_discrete_sac draws with a clip of 1e-3 (the
    golden's 40 never engages), DR3 on.  The sharded critics, the clip norm and the logged loss must equal the unsharded
    update on the same draws."""
    import copy
    from itertools import chain

    import golden_util as gu
    from super_sac_b200 import _arena, _rng, augmentations, learning, learning_utils as lu, parallel
    from test_discrete_host import _load_stack

    fx = gu.load("update_discrete_sac")
    cfg = gu.cfg_of(fx)
    Ng, M, S, B, clip = cfg["N"], cfg["M"], cfg["S"], cfg["B"], 1e-3
    lu.sample_move_and_augment = _sampler(gu.sub(fx, "buffer"), S)

    def run(sharded):
        lo, hi = parallel.enable_critic_sharding(Ng) if sharded else (0, Ng)
        agent = _agent(fx, 1, hi - lo, False)
        _load_stack(agent._actor_arena, gu.sub(fx, "init/actors"))
        _load_stack(agent._critic_arena, _rows_of(gu.sub(fx, "init/critics"), np.arange(lo, hi)))
        target = copy.deepcopy(agent)
        _load_stack(target._critic_arena, _rows_of(gu.sub(fx, "init/target_critics"), np.arange(lo, hi)))
        opt = torch.optim.Adam(chain(*(c.parameters() for c in agent.critics)), lr=3e-4)
        la = torch.tensor([np.log(0.1)], dtype=torch.float32, requires_grad=True)
        aug = augmentations.AugmentationSequence([augmentations.IdentityAug(B)])
        gsq, losses = [], []
        for t in range(cfg["steps"]):
            src = _rng.ScriptedSource()
            _rng.set_source(src)
            r = gu.sub(fx, f"step{t}/rand")
            src.push("indices", r["idx"][0]).push("subsets", r["subsets"][0].astype(np.int32))
            logs, _ = learning.critic_update(
                buffer=None, agent=agent, target_agent=target, critic_optimizer=opt,
                encoder_optimizer=torch.optim.Adam(agent.encoder.parameters()), log_alphas=[la], batch_size=B, gamma=0.99,
                critic_clip=clip, encoder_clip=None, target_critic_ensemble_n=M, weighted_bellman_temp=None,
                weight_type=None, pop=False, augmenter=aug, encoder_lambda=0.0, aug_mix=0.0, discrete=True,
                random_process=None, noise_clip=None, per=False, update_priorities=False,
                dr3_coeff=cfg.get("dr3_coeff", 0.0))
            gsq.append(float(_arena.FlatAdam.attach(opt, agent._critic_arena).gnorm_sq))
            losses.append(logs["losses/critic_overall_loss"])
        parallel.disable()
        return agent, np.array(gsq), np.array(losses), lo, hi

    full, gsq_f, loss_f, _, _ = run(False)
    shard, gsq_s, loss_s, lo, hi = run(True)
    assert np.all(gsq_f > 100 * clip * clip), f"the clip does not engage: |g|^2 = {gsq_f}"
    gu.assert_close(gsq_s, gsq_f, RTOL, 0.0, "global clip norm |g|^2")
    gu.assert_close(loss_s, loss_f, RTOL, 1e-7, "logged loss")
    for n in ("W1", "b1", "W2", "b2", "W3", "b3"):
        gu.assert_close(shard._critic_arena.p[n].numpy(), full._critic_arena.p[n][lo:hi].numpy(), RTOL, 1e-7,
                        f"clipped critics {n}")
    return lo, hi


def _offline_case(rank, members=False):
    """discrete_afbc with the critics of both members sharded over the ranks: the advantage filter's Q_min gathers every
    rank's critics; actor, Adam, the priority refresh and the filter statistics run replicated -- with Python's
    ``random`` seeded differently on each rank, whose member draws differ.  ``members``: one member per rank instead;
    the filter's mean policy gathers every rank's actors."""
    import random
    from itertools import chain

    import golden_util as gu
    from super_sac_b200 import _rng, augmentations, learning, learning_utils as lu, parallel
    from test_discrete_host import _cmp_stack, _load_stack

    fx = gu.load("discrete_afbc")
    cfg = gu.cfg_of(fx)
    Eg, Ng, S, B = cfg["E"], cfg["N"], cfg["S"], cfg["B"]
    if members:
        lo, hi = parallel.enable_member_sharding(Eg)
        mem, E, N, nets_ = list(range(lo, hi)), hi - lo, Ng, np.arange(lo * Ng, hi * Ng)
    else:
        lo, hi = parallel.enable_critic_sharding(Ng)
        mem, E, N = list(range(Eg)), Eg, hi - lo
        nets_ = np.concatenate([np.arange(i * Ng + lo, i * Ng + hi) for i in range(Eg)])
    agent = _agent(fx, E, N, True)
    _load_stack(agent._actor_arena, _rows_of(gu.sub(fx, "init/actors"), mem))
    _load_stack(agent._critic_arena, _rows_of(gu.sub(fx, "init/critics"), nets_))
    pst = gu.sub(fx, "init/popart")
    for i, p in enumerate(agent.popart):
        g = mem[i]
        p.mu, p.nu, p.w, p.b = pst[f"{g}/mu"], pst[f"{g}/nu"], pst[f"{g}/w"], pst[f"{g}/b"]
        p._t = int(pst[f"{g}/t"])
    bufd, idx = gu.sub(fx, "buffer"), fx["rand/idx"]

    def make_rd(ix):
        XA = torch.as_tensor(np.concatenate([bufd["s"][ix], bufd["a"][ix]], 1).astype(np.float32))
        rd = lu.ReplayDict()
        rd["primary_batch"] = ({"obs": XA[:, :S]}, XA[:, S:], None, None, None)
        rd["priority_idxs"], rd["imp_weights"] = torch.as_tensor(ix), torch.ones(1)
        return rd

    if members:   # the mean policy needs every rank's actors: only offline_actor_update exchanges them
        with pytest.raises(NotImplementedError, match="every rank's actors"):
            agent.adv_estimator(make_rd(idx[lo])["primary_batch"][0], make_rd(idx[lo])["primary_batch"][1], 0)
    for i in range(E if not members else 0):   # agent.adv_estimator(o, a, i): Q_min over both ranks' critics
        rd = make_rd(idx[i])
        adv = agent.adv_estimator(rd["primary_batch"][0], rd["primary_batch"][1], i)
        gu.assert_close(adv.numpy(), fx[f"adv/{i}"], RTOL, 1e-6, f"adv[{i}]")

    def fake_sample(buffer, batch_size, augmenter, aug_mix, per=True, _idx=None):
        ix = torch.empty(batch_size, dtype=torch.int64)
        _rng.source().indices(ix, len(bufd["a"]))
        return make_rd(ix.numpy())

    lu.sample_move_and_augment = fake_sample
    actor_opt = torch.optim.Adam(chain(*(a.parameters() for a in agent.actors)), lr=3e-4, betas=(0.9, 0.999))
    enc_opt = torch.optim.Adam(agent.encoder.parameters(), lr=1e-4)
    augmenter = augmentations.AugmentationSequence([augmentations.IdentityAug(B)])
    src = _rng.ScriptedSource()
    _rng.set_source(src)
    for g in mem:
        src.push("indices", idx[g])
    logs = learning.offline_actor_update(
        buffer=None, agent=agent, actor_optimizer=actor_opt, encoder_optimizer=enc_opt, batch_size=B,
        actor_clip=cfg["actor_clip"], update_encoder=False, encoder_clip=None, augmenter=augmenter, actor_lambda=0.0,
        aug_mix=0.0, premade_replay_dicts=None, per=False, discrete=True, filter_=True)
    assert src.empty()
    _cmp_stack(agent._actor_arena.g, _rows_of(gu.sub(fx, "actor/grads"), mem), "actor grads", atol=2e-7)
    _cmp_stack(agent._actor_arena.p, _rows_of(gu.sub(fx, "actor/actors"), mem), "actors", atol=3e-4 * 0.05)
    _cmp_logs(logs, gu.sub(fx, "actor/logs"), "offline actor", lambda k: _member_of(k) is None or _member_of(k) in mem)
    if members:
        return lo, hi

    class Buf:
        def update_priorities(self, idxs, prios):
            self.idxs, self.prios = idxs, prios

    buf = Buf()
    # the golden's draw is random.seed(7)'s (member 1); seed 8 draws member 0: rank 0's pick must hold on every rank
    random.seed(7 if rank == 0 else 8)
    lu.adjust_priorities({}, make_rd(idx[-1]), agent, buf)
    assert np.array_equal(np.asarray(buf.idxs), fx["priorities/idxs"])
    gu.assert_close(buf.prios.numpy(), fx["priorities/values"], 1e-5, 1e-6, "priorities")
    _same_on_all_ranks(agent._actor_arena.flat, "actor")
    _same_on_all_ranks(buf.prios, "priorities")
    src.push("indices", idx[0])
    random.seed(7 if rank == 0 else 8)
    _same_on_all_ranks(torch.tensor([lu.compute_filter_stats(None, agent, augmenter, B)]), "filter statistics")
    return lo, hi


def _worker(rank, world, port, case, out_q):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from super_sac_b200 import parallel

    try:
        emu = _emulate()
        if case == "clip":
            lo, hi = _clip_case(rank)
        elif case.startswith("discrete_afbc"):
            lo, hi = _offline_case(rank, members=case.endswith("members"))
        else:
            lo, hi = _update_case(case, rank)
        assert "discrete_value" in emu.calls or case.startswith("discrete_afbc")
        out_q.put((rank, lo, hi, None))
    except Exception:  # noqa: BLE001  (reported by the parent)
        out_q.put((rank, None, None, traceback.format_exc()))
    finally:
        parallel.disable()
        dist.destroy_process_group()


@pytest.mark.parametrize("case,ranges", [
    ("discrete_sac", [(0, 0, 2), (1, 2, 3)]),                 # critics 0,1 | 2
    ("discrete_sunrise_popart", [(0, 0, 1), (1, 1, 2)]),      # member 0 | member 1
    ("discrete_afbc", [(0, 0, 1), (1, 1, 2)]),                # critic 0 | critic 1 of both members
    ("discrete_afbc_members", [(0, 0, 1), (1, 1, 2)]),        # member 0 | member 1
    ("clip", [(0, 0, 2), (1, 2, 3)]),                         # critics 0,1 | 2, against the unsharded update
], ids=["critics", "members", "offline", "offline-members", "clip"])
def test_sharded_discrete_update_matches_golden_world2_gloo(case, ranges):
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, case, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = sorted(q.get(timeout=300) for _ in range(world))
    for p in procs:
        p.join(120)
    errors = [err for *_, err in got if err]
    assert not errors, "\n".join(errors)
    assert all(p.exitcode == 0 for p in procs)
    assert [g[:3] for g in got] == ranges


def test_sharded_discrete_limits_fail_loudly(monkeypatch):
    """What sharded discrete ensembles do not cover raises: more than one member under critic sharding, both partitionings
    at once, a trainable encoder, softmax weights, and the priority refresh of member-sharded ensembles."""
    import super_sac_b200 as ssb
    from emulated_abi import EmulatedLib
    from super_sac_b200 import _lib, _ops, discrete, nets
    from test_discrete_host import IdentityEncoder

    monkeypatch.setattr(_lib, "_lib", EmulatedLib())
    monkeypatch.setattr(_lib, "stream_ptr", lambda: 0)
    monkeypatch.setattr(_ops, "check_cuda", lambda *t: None)
    monkeypatch.setenv("MASTER_ADDR", "127.0.0.1")
    monkeypatch.setenv("MASTER_PORT", str(_free_port()))
    dist.init_process_group("gloo", rank=0, world_size=1)
    from super_sac_b200 import parallel

    def agent(E, enc=None):
        return ssb.Agent(act_space_size=4, encoder=enc or IdentityEncoder(3), actor_network_cls=nets.mlps.DiscreteActor,
                         critic_network_cls=nets.mlps.DiscreteCritic, discrete=True, ensemble_size=E, num_critics=2,
                         hidden_size=16)

    def critic(ag, **kw):
        args = dict(buffer=None, agent=ag, target_agent=ag, critic_optimizer=None, encoder_optimizer=None, log_alphas=[],
                    batch_size=4, gamma=0.99, critic_clip=None, encoder_clip=None, target_critic_ensemble_n=2,
                    weighted_bellman_temp=None, weight_type=None, pop=False, augmenter=None, encoder_lambda=0.0,
                    aug_mix=0.0, per=False, update_priorities=False, dr3_coeff=0.0)
        args.update(kw)
        return discrete.critic_update(**args)

    class Trainable(IdentityEncoder):
        def __init__(self, dim):
            super().__init__(dim)
            self.proj = torch.nn.Linear(dim, dim)

    try:
        parallel.enable_critic_sharding(2)
        with pytest.raises(NotImplementedError, match="one member"):
            critic(agent(2))
        with pytest.raises(NotImplementedError, match="trainable"):
            critic(agent(1, Trainable(3)))
        with pytest.raises(NotImplementedError, match="cannot be combined"):
            parallel.enable_member_sharding(2)
        parallel.disable()
        parallel.enable_member_sharding(2)
        with pytest.raises(NotImplementedError, match="priority refresh"):
            critic(agent(2), update_priorities=True)
        with pytest.raises(NotImplementedError, match="sunrise"):
            critic(agent(2), weight_type="softmax", weighted_bellman_temp=10.0)
        with pytest.raises(NotImplementedError, match="priority refresh"):
            discrete.offline_actor_update(None, agent(2), None, None, 4, None, False, None, None, 0.0, 0.0, None, True, True)
    finally:
        parallel.disable()
        dist.destroy_process_group()

"""Prioritised replay over the frame-deduplicated n-step ring (NStepReplayBuffer(prioritized=True)).

Until the first start is evicted, the v-th start of the ring is the v-th tuple the reference's deque pushes (main.py:353-365)
and its tree leaf is v: the ring must then be bit-identical to a classic prioritised ReplayBuffer loaded with those tuples in
push order -- trees, draws, weights, batches and whole updates.  After evictions the trees are checked against a numpy model
of the live transitions, and the draw against the priorities."""
import copy
from itertools import chain

import numpy as np
import pytest
import torch

from test_nstep_replay import make_stream, reference_nstep_tuples

pytestmark = pytest.mark.gpu
DEV = "cuda"
ALPHA, BETA = 0.6, 0.4


def _discrete_actions(steps, A):
    return [(s, np.asarray([float(i % A)], np.float32), r, s1, t, o) for i, (s, _, r, s1, t, o) in enumerate(steps)]


def fill_pair(kind, reward_f32, n_step=3, gamma=0.97, n_steps=300, size=4096, seed=0, on_push=None, discrete_actions=0):
    """The same one-step stream into NStepReplayBuffer(prioritized=True) and, one reference tuple at the moment its window
    completes, into a classic prioritised ReplayBuffer.  on_push(nb, cb, t) runs after every push."""
    import super_sac_b200 as ssb

    rng = np.random.default_rng(seed)
    steps = make_stream(kind, n_steps, rng, reward_f32)
    if discrete_actions:
        steps = _discrete_actions(steps, discrete_actions)
    want = reference_nstep_tuples(steps, n_step, gamma)
    nb = ssb.replay.NStepReplayBuffer(size, n_step=n_step, gamma=gamma, frame_stack=3 if kind == "pixels" else 1, device=DEV,
                                      prioritized=True, alpha=ALPHA, beta=BETA)
    cb = ssb.replay.ReplayBuffer(size, alpha=ALPHA, beta=BETA, device=DEV)
    for t, (s, a, r, s1, term, over) in enumerate(steps):
        nb.push(s, a, r, s1, term, terminate_traj=over)
        while len(cb) < len(nb):
            ws, wa, wr, ws1, wd = want[len(cb)]
            cb.push(ws, wa, wr, ws1, wd)
        if on_push is not None:
            on_push(nb, cb, t)
    assert nb._v_tail == 0 and len(nb) == len(cb) == len(want)
    return nb, cb, rng


def trees_equal(nb, cb):
    return torch.equal(nb._it_sum, cb._it_sum) and torch.equal(nb._it_min, cb._it_min)


@pytest.mark.parametrize("reward_f32", [False, True], ids=["float64-rewards", "float32-rewards"])
@pytest.mark.parametrize("kind", ["flat", "pixels"])
def test_trees_before_eviction_equal_classic_per(kind, reward_f32):
    upd = np.random.default_rng(11)
    checked = []

    def on_push(nb, cb, t):
        torch.cuda.synchronize()
        if cb._it_sum is None:   # no window complete yet: no classic storage, the ring's trees are still empty
            assert len(nb) == 0 and not bool(nb._it_sum.any()) and bool(torch.isinf(nb._it_min).all())
            return
        assert trees_equal(nb, cb), f"push {t}"
        n = len(nb)
        if t % 17 == 16 and n >= 4:
            ids = upd.integers(0, n, 24)   # duplicates: the last write of a leaf wins
            pr = upd.uniform(0.01, 3.0, 24)
            if t % 2:
                for buf in (nb, cb):
                    buf.update_priorities(ids, pr)
            else:
                ids_d, pr_d = torch.from_numpy(ids).to(DEV), torch.from_numpy(pr).to(DEV)
                for buf in (nb, cb):
                    buf.update_priorities(ids_d, pr_d)
            torch.cuda.synchronize()
            assert trees_equal(nb, cb), f"update after push {t}"
            assert nb._max_priority == cb._max_priority
            checked.append(t)

    fill_pair(kind, reward_f32, on_push=on_push)
    assert len(checked) > 5


@pytest.mark.parametrize("kind", ["flat", "pixels"])
def test_sampling_before_eviction_equals_classic_per(kind):
    from super_sac_b200 import _rng, augmentations, learning_utils as lu

    nb, cb, rng = fill_pair(kind, False, seed=5)
    ids = rng.integers(0, len(nb), 200)
    pr = rng.uniform(0.05, 2.0, 200)
    for buf in (nb, cb):
        buf.update_priorities(ids, pr)
    B = 128
    u = rng.uniform(0.0, 1.0, B)
    u[:3] = [0.0, np.nextafter(1.0, 0.0), 0.5]
    outs = []
    for buf in (cb, nb):
        src = _rng.ScriptedSource()
        old = _rng.set_source(src)
        try:
            src.push("uniform01", u)
            outs.append(buf.sample(B))
        finally:
            _rng.set_source(old)
    torch.cuda.synchronize()
    (b0, w0, i0), (b1, w1, i1) = outs
    assert np.array_equal(i0, i1)
    assert torch.equal(w0, w1)
    (s0, a0, r0, p0, d0), (s1, a1, r1, p1, d1) = b0, b1
    for key in s0:
        assert torch.equal(s0[key], s1[key]) and torch.equal(p0[key], p1[key]), key
    assert torch.equal(a0, a1) and torch.equal(r0, r1) and torch.equal(d0, d1)

    if kind == "pixels":
        augm = augmentations.AugmentationSequence([augmentations.Drqv2Aug(B)], keys=["pixels"])
        shift = rng.integers(0, 9, (B, 2)).astype(np.int32)
    else:
        augm = augmentations.AugmentationSequence([augmentations.IdentityAug(B)])
        shift = None
    rds = []
    for buf in (cb, nb):
        src = _rng.ScriptedSource()
        old = _rng.set_source(src)
        try:
            src.push("uniform01", u[::-1].copy())
            if shift is not None:
                src.push("shifts", shift)
            rds.append(lu.sample_move_and_augment(buffer=buf, batch_size=B, augmenter=augm, aug_mix=0.75, per=True))
            assert src.empty()
        finally:
            _rng.set_source(old)
    torch.cuda.synchronize()
    c, n = rds
    assert torch.equal(c["priority_idxs"], n["priority_idxs"])
    assert n["imp_weights"].dtype == torch.float64 and torch.equal(c["imp_weights"], n["imp_weights"])
    (o0, a0, r0, q0, d0), (o1, a1, r1, q1, d1) = c["primary_batch"], n["primary_batch"]
    for key in o0:
        assert torch.equal(o0[key], o1[key]) and torch.equal(q0[key], q1[key]), key
    assert torch.equal(a0, a1) and torch.equal(r0, r1) and torch.equal(d0, d1)


def _continuous_agent():
    import cuda_util as cu
    import super_sac_b200 as ssb
    from super_sac_b200 import nets

    return ssb.Agent(act_space_size=2, encoder=cu.IdentityEncoder(5), actor_network_cls=nets.mlps.ContinuousStochasticActor,
                     critic_network_cls=nets.mlps.ContinuousCritic, ensemble_size=1, num_critics=4, hidden_size=64,
                     auto_rescale_targets=False, log_std_low=-5.0, log_std_high=2.0)


def _discrete_agent(A):
    import cuda_util as cu
    import super_sac_b200 as ssb
    from super_sac_b200 import nets

    return ssb.Agent(act_space_size=A, encoder=cu.IdentityEncoder(5), actor_network_cls=nets.mlps.DiscreteActor,
                     critic_network_cls=nets.mlps.DiscreteCritic, discrete=True, ensemble_size=1, num_critics=2,
                     hidden_size=64, auto_rescale_targets=False)


@pytest.mark.parametrize("discrete", [False, True], ids=["continuous", "discrete"])
def test_per_updates_before_eviction_equal_classic_per(discrete):
    """Six critic_update(per=True, update_priorities=True) calls (Polyak every second one), plus one
    offline_actor_update(per=True) for the continuous agent: parameters and trees bit-identical to the classic buffer."""
    import super_sac_b200 as ssb
    from super_sac_b200 import augmentations, learning, learning_utils as lu

    A, n_step, gamma, B = 3, 3, 0.99, 64
    nb, cb, _ = fill_pair("flat", False, n_step=n_step, gamma=gamma, n_steps=600, seed=3, discrete_actions=A if discrete else 0)

    def run(buf):
        ssb.manual_seed(21)
        torch.manual_seed(21)
        agent = _discrete_agent(A) if discrete else _continuous_agent()
        agent.to(DEV)
        target = copy.deepcopy(agent)
        c_opt = torch.optim.Adam(chain(*(c.parameters() for c in agent.critics)), lr=3e-4)
        e_opt = torch.optim.Adam(agent.encoder.parameters(), lr=1e-4)
        la = [torch.tensor([-2.3], device=DEV, requires_grad=True)]
        aug = augmentations.AugmentationSequence([augmentations.IdentityAug(B)])
        for k in range(6):
            learning.critic_update(
                buffer=buf, agent=agent, target_agent=target, critic_optimizer=c_opt, encoder_optimizer=e_opt, log_alphas=la,
                batch_size=B, gamma=gamma ** n_step, critic_clip=None, encoder_clip=None, target_critic_ensemble_n=2,
                weighted_bellman_temp=None, weight_type=None, pop=False, augmenter=aug, encoder_lambda=0.0,
                random_process=None, noise_clip=None, aug_mix=0.0, discrete=discrete, per=True, update_priorities=True)
            if k % 2 == 0:
                lu.soft_update(target.critics[0], agent.critics[0], 0.005)
        out = [agent._critic_arena.flat.clone(), target._critic_arena.flat.clone()]
        if not discrete:
            a_opt = torch.optim.Adam(chain(*(a.parameters() for a in agent.actors)), lr=1e-4)
            learning.offline_actor_update(buffer=buf, agent=agent, actor_optimizer=a_opt, encoder_optimizer=e_opt,
                                          batch_size=B, actor_clip=None, update_encoder=False, encoder_clip=None,
                                          augmenter=aug, actor_lambda=0.0, aug_mix=0.0, per=True, filter_=True)
            out.append(agent._actor_arena.flat.clone())
        torch.cuda.synchronize()
        return out + [buf._it_sum.clone(), buf._it_min.clone()]

    want, got = run(cb), run(nb)
    assert not torch.equal(want[-2], torch.zeros_like(want[-2]))
    names = ["critics", "targets"] + ([] if discrete else ["actors"]) + ["sum tree", "min tree"]
    for name, x, y in zip(names, want, got):
        assert torch.equal(x, y), name


# ---- after eviction ---------------------------------------------------------------------------------------------------
def _live_slots(nb):
    return [v % nb._maxsize for v in range(nb._v_tail, nb._v_head)]


def _check_against_model(nb, model):
    """model: slot -> p ** alpha of the transition in it.  Leaves: live -> that value (sum and min), dead -> (0, +inf);
    every internal node = its recomputed children."""
    torch.cuda.synchronize()
    S, M = nb._it_sum.cpu().numpy(), nb._it_min.cpu().numpy()
    cap2 = nb._capacity
    live = set(_live_slots(nb))
    for leaf in range(cap2):
        if leaf in live:
            want = model[leaf]
            assert S[cap2 + leaf] == want and M[cap2 + leaf] == want, leaf
        else:
            assert S[cap2 + leaf] == 0.0 and M[cap2 + leaf] == np.inf, leaf
    nodes = np.arange(1, cap2)
    assert np.array_equal(S[nodes], S[2 * nodes] + S[2 * nodes + 1])
    assert np.array_equal(M[nodes], np.fmin(M[2 * nodes], M[2 * nodes + 1]))
    return S, M, live


def _evicting_stream(n_steps, seed):
    rng = np.random.default_rng(seed)
    return make_stream("pixels", n_steps, rng, reward_f32=False), rng


def test_after_eviction_trees_draws_and_stale_updates():
    import super_sac_b200 as ssb
    from super_sac_b200 import _rng

    steps, rng = _evicting_stream(3000, 17)
    size = 61
    nb = ssb.replay.NStepReplayBuffer(size, n_step=5, gamma=0.97, frame_stack=3, frame_capacity=70, device=DEV,
                                      prioritized=True, alpha=ALPHA, beta=BETA)
    model = {}           # slot -> p ** alpha of the live transition in it
    max_p = 1.0
    ssb.manual_seed(5)
    torch.manual_seed(5)
    n_checks = 0
    for t, (s, a, r, s1, term, over) in enumerate(steps):
        v0 = nb._v_head
        nb.push(s, a, r, s1, term, terminate_traj=over)
        for v in range(v0, nb._v_head):
            model[v % size] = max_p ** ALPHA   # what the push writes (replay.py:129)
        if t > 100 and t % 37 == 0 and len(nb) >= 8:
            B = 64
            batch, w, ids = nb.sample(B)
            live = _live_slots(nb)
            assert set(ids.tolist()) <= set(live), "a dead slot was drawn"
            # weights: replay.py:173-176 with N = number of live transitions
            S, M, _ = _check_against_model(nb, model)
            N = len(live)
            p_min = M[1] / S[1]
            want_w = (S[nb._capacity + ids] / S[1] * N) ** (-BETA) / (p_min * N) ** (-BETA)
            np.testing.assert_allclose(w.cpu().numpy(), want_w, rtol=1e-12, atol=0)
            # the batch rows are the transitions in those slots (FIFO position (slot - v_tail) mod size)
            alls = nb.get_all_transitions()
            j = (ids - nb._v_tail) % size
            torch.cuda.synchronize()
            for key in batch[0]:
                assert torch.equal(batch[0][key], alls[0][key][torch.from_numpy(j).to(DEV)]), key
            assert torch.equal(batch[2], alls[2][torch.from_numpy(j).to(DEV)])
            # new priorities for the drawn ids (numpy path: the same float64 pow as the model)
            pr = rng.uniform(0.05, 4.0, B)
            nb.update_priorities(ids, pr)
            for i, v in zip(ids.tolist(), (pr**ALPHA).tolist()):   # the same float64 pow as update_priorities
                model[i] = v
            max_p = max(max_p, float(pr.max()))
            _check_against_model(nb, model)
            n_checks += 1
    assert nb._v_tail > 20 * size, "the FIFO of starts must wrap many times"
    assert n_checks > 50

    # boundary draws: u just below 1 and u = 1 (mass = the whole root) never return a dead slot; u = 1 descends to the
    # right end, where dead leaves sit (size 61 < 64 leaves), and is moved to the live leaf with the largest index
    live = _live_slots(nb)
    src = _rng.ScriptedSource()
    old = _rng.set_source(src)
    try:
        src.push("uniform01", np.asarray([np.nextafter(1.0, 0.0), 1.0, 0.0, 1.0 - 1e-12]))
        _, _, ids = nb.sample(4)
    finally:
        _rng.set_source(old)
    assert set(ids.tolist()) <= set(live)
    assert ids[1] == max(live)

    # a stale update: the oldest live transition is evicted by the next pushes; its slot is not reused yet
    oldest_v = nb._v_tail
    slot = oldest_v % size
    k = 0
    more, _ = _evicting_stream(400, 99)
    while nb._v_tail <= oldest_v:
        s, a, r, s1, term, over = more[k % len(more)]
        nb.push(s, a, r, s1, term, terminate_traj=True)   # every step its own episode: no window completes (n_step 5)
        k += 1
    assert nb._v_head < oldest_v + size and slot not in _live_slots(nb)
    torch.cuda.synchronize()
    before = nb._it_sum.clone(), nb._it_min.clone()
    nb.update_priorities(np.asarray([slot]), np.asarray([3.0]))
    nb.update_priorities(torch.tensor([slot, slot], device=DEV), torch.tensor([2.0, 7.0], dtype=torch.float64, device=DEV))
    torch.cuda.synchronize()
    assert torch.equal(before[0], nb._it_sum) and torch.equal(before[1], nb._it_min)


def test_boundary_rule_on_a_hand_built_tree():
    """The kernel's rule for a descent that ends on a dead leaf, on exact (dyadic) trees: u = 1 walks to the right end."""
    import super_sac_b200 as ssb

    L = ssb._lib.lib()
    cap2, size = 8, 7

    def draw(tail, n, u):
        leaf_sum = np.zeros(cap2)
        live = [(tail + i) % size for i in range(n)]
        leaf_sum[live] = 0.5
        S = np.zeros(2 * cap2)
        M = np.full(2 * cap2, np.inf)
        S[cap2:] = leaf_sum
        M[cap2:][live] = 0.5
        for node in range(cap2 - 1, 0, -1):
            S[node] = S[2 * node] + S[2 * node + 1]
            M[node] = min(M[2 * node], M[2 * node + 1])
        St, Mt = torch.from_numpy(S).to(DEV), torch.from_numpy(M).to(DEV)
        scal = torch.tensor([n, tail % size, 1], dtype=torch.int64, device=DEV)
        ut = torch.tensor(u, dtype=torch.float64, device=DEV)
        B = ut.numel()
        vr = torch.arange(size, dtype=torch.int64, device=DEV)
        rew = torch.zeros(size, dtype=torch.float64, device=DEV)
        gp = torch.ones(1, dtype=torch.float64, device=DEV)
        o = [torch.empty(B, dtype=torch.int64, device=DEV) for _ in range(4)]
        w = torch.empty(B, dtype=torch.float64, device=DEV)
        R = torch.empty(B, dtype=torch.float32, device=DEV)
        L.nstep_tree_sample(St.data_ptr(), Mt.data_ptr(), cap2, size, scal.data_ptr(), ut.data_ptr(), B, 1.0, o[0].data_ptr(),
                            o[1].data_ptr(), w.data_ptr(), vr.data_ptr(), 1, rew.data_ptr(), None, gp.data_ptr(), None,
                            o[2].data_ptr(), o[3].data_ptr(), R.data_ptr(), None, None, ssb._lib.stream_ptr())
        torch.cuda.synchronize()
        return o[0].cpu().numpy(), o[1].cpu().numpy(), live

    # live [2, 5): u = 1 ends on leaf 7 (padding) -> the largest live leaf below it, 4; FIFO position 2
    slots, j, live = draw(2, 3, [1.0, 0.0, 0.5])
    assert slots[0] == 4 and j[0] == 2 and set(slots.tolist()) <= set(live)
    # wrapped live range {5, 6, 0, 1}: leaf 7 -> 6
    slots, j, live = draw(5, 4, [1.0, 0.0, 0.99])
    assert slots[0] == 6 and j[0] == 1 and set(slots.tolist()) <= set(live)
    # full ring: every leaf below 7 is live -> 6
    slots, _, _ = draw(3, 7, [1.0])
    assert slots[0] == 6


def test_draw_frequencies_follow_the_priorities():
    """2^16 seeded draws after many evictions: chi-square against p ** alpha of the live transitions."""
    from scipy import stats

    import super_sac_b200 as ssb

    steps, rng = _evicting_stream(1500, 23)
    size = 61
    nb = ssb.replay.NStepReplayBuffer(size, n_step=5, gamma=0.97, frame_stack=3, frame_capacity=70, device=DEV,
                                      prioritized=True, alpha=ALPHA, beta=BETA)
    for s, a, r, s1, term, over in steps:
        nb.push(s, a, r, s1, term, terminate_traj=over)
    assert nb._v_tail > 0
    live = _live_slots(nb)
    pr = rng.uniform(0.1, 5.0, len(live))
    nb.update_priorities(np.asarray(live), pr)
    torch.manual_seed(1234)
    counts = np.zeros(size, dtype=np.int64)
    for _ in range(64):
        res, _ = nb.sample_per(1024)
        counts += np.bincount(res["slot"].cpu().numpy(), minlength=size)
    assert counts.sum() == 65536
    assert counts[[i for i in range(size) if i not in set(live)]].sum() == 0
    p = pr ** ALPHA
    expected = p / p.sum() * 65536
    _, pval = stats.chisquare(counts[live], expected)
    assert pval > 1e-3, pval


def test_uniform_ring_still_refuses_priorities():
    import super_sac_b200 as ssb
    from super_sac_b200 import augmentations, learning_utils as lu

    buf = ssb.replay.NStepReplayBuffer(256, n_step=2, device=DEV)
    rng = np.random.default_rng(0)
    for s, a, r, s1, term, over in make_stream("flat", 80, rng, reward_f32=False):
        buf.push(s, a, r, s1, term, terminate_traj=over)
    with pytest.raises(NotImplementedError):
        buf.sample(8)
    with pytest.raises(NotImplementedError):
        buf.update_priorities(np.asarray([0]), np.asarray([1.0]))
    aug = augmentations.AugmentationSequence([augmentations.IdentityAug(8)])
    with pytest.raises(NotImplementedError, match="prioritized=True"):
        lu.sample_move_and_augment(buffer=buf, batch_size=8, augmenter=aug, aug_mix=0.0, per=True)
    rd = lu.sample_move_and_augment(buffer=buf, batch_size=8, augmenter=aug, aug_mix=0.0, per=False)
    assert rd["primary_batch"][0]["obs"].shape == (8, 5)

"""SAC-Discrete updates (SURVEY 8f N4): the ``discrete=True`` branches of reference learning.py:18-141 (critic),
:344-421 (actor), :222-263 (temperature) and learning_utils.py:322-328 (TD target), :373-376 (sunrise weights).

Same flat arenas, grouped MLP launches (ssac_mlp_forward / ssac_mlp_backward with O = number of actions: every critic
net emits its whole Q row), fused Adam and device-side logs as the continuous path in learning.py; the categorical
arithmetic around the networks (softmax, expectation over actions, gather at the taken action and its scatter back into
the dense output gradient) runs in the ssac_discrete_* kernels (csrc/ssac_discrete.cu).  Members run in series.  Nothing
here allocates by host state, reads back or decides on the host (except the logged member, ``random.choice``, frozen at
capture as in the continuous path), so ``learning.critic_update`` / ``online_actor_update`` replay these functions as
CUDA graphs under ``graphed.enable_auto_graphs()``; inside ``lu.pipelined_updates()`` the target side of a one-member
critic update runs on the block's front stream (as in learning._critic_update_impl).  The offline (AFBC) actor update
with the indirect advantage filter (adv_estimator.py:45-56) and the priority refresh are here too.  Not implemented
(raise): softmax Bellman weights (they draw Categorical samples), the invariance regularisers.

Sharded ensembles (parallel.py) exchange through the same sites as the continuous path -- peer stores on GPUs,
torch.distributed collectives otherwise -- and follow the same rules (learning_utils' shared pieces: global loss
normalisation, global clip norms, global member ids in the log keys, logged values summed over / taken from the owning
rank):

- critics over ranks (``enable_critic_sharding``, one member): actor, temperature, PopArt and batch stay replicated.
  The TD target gathers the REDQ subset's target rows [M,B,A] from every rank (on the front stream inside
  ``lu.pipelined_updates()``), the actor update and the advantage filter every rank's online rows [N_global,B,A]; no
  gradient crosses ranks (the discrete actor loss takes none through the critics).
- members over ranks (``enable_member_sharding``): each rank runs its members.  The sunrise weights gather every
  member's batch, run the local target critics over all of them and gather the values back (``_member_target_q``); the
  offline filter does the same with the actors for the mean policy (``_member_policies``).
- the member that rates a batch for the priority refresh / filter statistics (the reference's ``random.choice``) is
  rank 0's draw on every rank when the critics are sharded (parallel.same_member_choice).
- not covered (raise): more than one member in the critic update under critic sharding, an encoder with trainable
  parameters; with members sharded, the priority refresh, compute_filter_stats and direct advantage-estimator calls.

Only the member bodies are this module's own.  The skeleton around them -- pipeline eligibility, member batches, the
member loop, the encoder step, the logged gradient norms, the temperature step, the DR3 term and the ends of the critic
and actor updates -- is learning_utils' "shared pieces of the updates", which learning.py uses as well.
"""
import contextlib

import torch

from . import _arena, _lib, _logs, _ops, _rng, parallel
from . import learning_utils as lu


def _rows(rep):
    """(tensor, row stride) of a [B, S] fp32 device matrix the kernels can read in place (unit column stride)."""
    rep = rep.detach()
    if rep.dtype != torch.float32 or rep.dim() != 2 or rep.stride(1) != 1:
        rep = rep.float().contiguous()
    _ops.check_cuda(rep)
    return rep, rep.stride(0)


def _forward(arena, g0, G, X, ldx, B, net_index=None, keep=False):
    """y [G,B,O] of nets g0..g0+G (or the ``net_index`` subset relative to g0) on the rows of X."""
    dev = X.device
    h1 = torch.empty((G, B, arena.H), dtype=torch.float32, device=dev)
    h2 = torch.empty_like(h1)
    y = torch.empty((G, B, arena.O), dtype=torch.float32, device=dev)
    _ops.mlp_forward(arena, g0, G, X, B, h1, h2, y, ldx=ldx, net_index=net_index, keep_hidden=keep)
    return (y, h1, h2) if keep else y


def _actions(a, B):
    """The taken actions as a dense float [B] vector holding the indices (replay row [B,1], ``a.long()`` in the reference)."""
    return a.reshape(B).float().contiguous()


def _check(agent):
    if not agent.discrete:
        raise ValueError("discrete=True needs an Agent built with discrete=True")
    if parallel.sharded() and lu._encoder_trainable(agent):
        raise NotImplementedError("sharded discrete ensembles need an encoder without trainable parameters: every rank "
                                  "would train its replica on its own share of the gradients and the replicas would drift")
    _ops.check_cuda(agent._critic_arena.flat)


def _global_q(q_local, site):
    """Critics sharded over ranks: this rank's nets' Q rows [n_local, B, A] -> every net's [N_global, B, A]."""
    return parallel.all_gather_q(q_local, site=site) if parallel.critics_sharded() else q_local


def compute_td_targets(logs, replay_dict, agent, target_agent, ensemble_idx, ensemble_n, log_alphas, pop, gamma):
    """learning_utils.py:298-354 with discrete=True: y = r + gamma (1-d) E_{a~pi(s1)}[min_M Q_target(s1, a) - alpha log pi(a|s1)],
    PopArt as in the continuous branch.  Returns (y [B,1], (s1_rep, None)): the reference hands back the policy's
    probabilities in the second slot (:328), which nothing on the update path reads -- they never leave the kernel here."""
    dlogs, user_logs = _logs.as_device_logs(logs, agent._critic_arena.device)
    i, M = ensemble_idx, ensemble_n
    o, a, r, o1, d = replay_dict["primary_batch"]
    aa, N = agent._actor_arena, agent.num_critics
    A = agent.act_space_size
    # REDQ subset: drawn over the GLOBAL ensemble when the critics are sharded over ranks (replicated Philox state)
    pool = parallel.n_global(N)
    assert 0 < M <= pool
    L, stream = _lib.lib(), _lib.stream_ptr()
    with torch.no_grad():
        s1_rep = target_agent.encoder(o1)
    X1, ld1 = _rows(s1_rep)
    B, dev = X1.shape[0], X1.device
    # the subset is drawn before the actor forward: the single-kernel forward reads net_index ahead of its PDL wait,
    # which needs the draw at least two launches back (ssac_mlp_fused.cu).  The actor forward draws nothing, so the
    # random numbers are the same as in the reference's order (policy, then subset).
    subset = torch.empty(M, dtype=torch.int32, device=dev)
    _rng.source().subsets(subset, pool, M)                                  # agent.py:29
    logits = _forward(aa, i, 1, X1, ld1, B)
    if lu.pipeline() is not None:
        lu.pipeline().front_wait_polyak()   # the target critics' parameters: the only thing this side reads that Polyak writes
    if parallel.critics_sharded():
        # every rank evaluates its own target critics and gathers the subset's rows [M,B,A] (in subset order): the state
        # value, the TD target and the PopArt update are then the same on every rank.  Inside lu.pipelined_updates() the
        # put and the wait run on the front stream with the rest of this side.
        qt = parallel.all_gather_q(_forward(target_agent._critic_arena, i * N, N, X1, ld1, B), site="target_q",
                                   select=subset)
    else:
        qt = _forward(target_agent._critic_arena, i * N, M, X1, ld1, B, net_index=subset)   # [M,B,A]
    v = torch.empty(B, dtype=torch.float32, device=dev)
    ev, eslot = dlogs.slots(1)                                              # zero-initialised with the buffer
    L.discrete_value(logits.data_ptr(), qt.data_ptr(), M, B, A, log_alphas[i].data_ptr(), v.data_ptr(), ev.data_ptr(), stream)
    popart = agent.popart[i]
    y = torch.empty((B, 1), dtype=torch.float32, device=dev)
    lv, slot = dlogs.slots(3)
    # PopArt de-normalisation, r + gamma (1-d) v, statistics update and re-normalisation: the continuous kernel with the
    # state value in the place of min Q - alpha logp (M = 1, no entropy term: it is inside v already)
    L.td_target(v.data_ptr(), 1, B, None, log_alphas[i].data_ptr(), r.data_ptr(), d.data_ptr(), float(gamma),
                popart.state_ptr() if popart else None, popart.ctl_ptr() if popart else None, int(bool(pop)),
                float(popart.beta) if popart else 0.0, int(popart.min_steps) if popart else 0, y.data_ptr(), lv.data_ptr(),
                stream)
    g = parallel.member_id(i)
    dlogs.defer(f"td_targets/mean_td_target_{g}", slot)
    dlogs.defer(f"td_targets/std_td_target_{g}", slot + 1)
    dlogs.defer(f"td_targets/entropy_bonus_{g}", eslot)
    if user_logs is not None:
        user_logs.update(dlogs.finalize())
    return y, (s1_rep, None)


def compute_backup_weights(logs, replay_dict, agent, target_agent, weight_type, weight_temp, batch_size, _q_sel=None):
    """learning_utils.py:357-398 with discrete=True: sunrise weights from the std over members of min_N Q_target(s, a_b).
    ``_q_sel`` [E_global*N, B]: every target net's Q at the taken actions of this member's batch, already gathered over
    the ranks (members sharded over ranks: ``_member_target_q``)."""
    E, N = parallel.members_global(agent.ensemble_size), agent.num_critics
    if weight_type is None or weight_temp is None or E == 1:
        return 1.0
    if weight_type != "sunrise":
        raise NotImplementedError("discrete agents: only the sunrise Bellman weights are implemented "
                                  "(softmax weights draw Categorical samples)")
    dlogs, user_logs = _logs.as_device_logs(logs, agent._critic_arena.device)
    L, stream = _lib.lib(), _lib.stream_ptr()
    if _q_sel is not None:
        q_sel, B, dev = _q_sel, _q_sel.shape[1], _q_sel.device
    elif parallel.members_sharded():
        raise NotImplementedError("member-sharded ensembles: the sunrise weights are exchanged inside critic_update")
    else:
        o, a, *_ = replay_dict["primary_batch"]
        A = agent.act_space_size
        with torch.no_grad():
            s_rep = target_agent.encoder(o)
        X, ld = _rows(s_rep)
        B, dev = X.shape[0], X.device
        q_all = _forward(target_agent._critic_arena, 0, E * N, X, ld, B)        # every target net's Q row: one launch
        q_sel = torch.empty((E * N, B), dtype=torch.float32, device=dev)
        act = _actions(a, B)
        L.discrete_gather_q(q_all.data_ptr(), act.data_ptr(), E * N, B, A, q_sel.data_ptr(), stream)
    w = torch.empty((B, 1), dtype=torch.float32, device=dev)
    lv, slot = dlogs.slots(4)
    L.backup_weights(q_sel.data_ptr(), E, N, B, float(weight_temp), 0, w.data_ptr(), lv.data_ptr(), stream)
    for j, name in enumerate(("mean", "max", "min", "std")):
        dlogs.defer(f"bellman_weights/{name}", slot + j)
    if user_logs is not None:
        user_logs.update(dlogs.finalize())
    return w


def _member_target_q(rds, target_agent, N, B):
    """Members sharded over ranks: every target net of every rank on every member's batch, at the batch's actions ->
    [E_global*N, E_global, B] (global net order, then global member order).  Two exchanges: the local batches' states
    and actions to every rank, then each rank's values back; in between one grouped forward of the local target critics
    over all E_global*B gathered rows and one gather at the taken actions."""
    E, A = len(rds), target_agent.act_space_size
    Xs, acts = [], []
    for rd in rds:
        o, a, *_ = rd["primary_batch"]
        with torch.no_grad():
            Xs.append(_rows(target_agent.encoder(o))[0])
        acts.append(_actions(a, B))
    x_all = parallel.all_gather_members(torch.stack(Xs))                    # [En,B,S]
    act_all = parallel.all_gather_members(torch.stack(acts))                # [En,B]
    En, S = x_all.shape[0], x_all.shape[2]
    q = _forward(target_agent._critic_arena, 0, E * N, x_all.view(En * B, S), S, En * B)   # [E*N, En*B, A]
    q_sel = torch.empty((E * N, En, B), dtype=torch.float32, device=q.device)
    _lib.lib().discrete_gather_q(q.data_ptr(), act_all.data_ptr(), E * N, En * B, A, q_sel.data_ptr(), _lib.stream_ptr())
    return parallel.all_gather_members(q_sel)                               # [En*N, En, B]


def critic_update(buffer, agent, target_agent, critic_optimizer, encoder_optimizer, log_alphas, batch_size, gamma,
                  critic_clip, encoder_clip, target_critic_ensemble_n, weighted_bellman_temp, weight_type, pop, augmenter,
                  encoder_lambda, aug_mix, per, update_priorities, dr3_coeff):
    """learning.py:18-141 with discrete=True."""
    _check(agent)
    if encoder_lambda:
        raise NotImplementedError("encoder invariance regulariser (lambda = 0 in every shipped config) is out of scope")
    ca = agent._critic_arena
    dev = ca.device
    L, stream = _lib.lib(), _lib.stream_ptr()
    E, N, B, A = agent.ensemble_size, agent.num_critics, batch_size, agent.act_space_size
    if parallel.critics_sharded() and E != 1:
        raise NotImplementedError("critic sharding covers one member (REDQ / SAC shapes); SUNRISE members shard as a whole")
    if parallel.members_sharded() and update_priorities:
        raise NotImplementedError("member-sharded ensembles: the priority refresh needs every actor on the batch")
    if parallel.members_sharded() and weight_type not in (None, "sunrise") and weighted_bellman_temp is not None:
        raise NotImplementedError("discrete agents: only the sunrise Bellman weights are implemented "
                                  "(softmax weights draw Categorical samples)")
    # loss normalisation over the GLOBAL ensemble: all members when members are sharded over ranks, all critics when the
    # critics are (each rank then holds a share of the loss and of the DR3 mean; the shares are summed below)
    En = parallel.members_global(E)
    # Inside lu.pipelined_updates(): the target side (draws, gather, actor logits and target-critic subset on s1, state
    # value, TD target -- and, critics sharded over ranks, the exchange of the target values) runs on the front stream,
    # the online side on the caller's (eligibility: lu._critic_pipeline).
    pipe = lu._critic_pipeline(agent, per, update_priorities, weight_type)
    if pipe is not None:
        main = torch.cuda.current_stream(dev)
        pipe.front_wait_dep(main)
    with (torch.cuda.stream(pipe.front) if pipe is not None else contextlib.nullcontext()):
        logs = _logs.DeviceLogs(dev)   # (zeroed on the stream that writes it first)
    if pipe is not None:
        pipe.keep.append(logs)
    loss_all, loss_slot = logs.slots(2 * E)   # per member: {loss contribution, mean td error of its last net}
    opt = _arena.FlatAdam.attach(critic_optimizer, ca)
    enc_outs = []
    presampled, q_weights = None, None
    if parallel.members_sharded() and weight_type is not None and weighted_bellman_temp is not None and En > 1:
        # every local member samples first; then the exchange of _member_target_q (the draws of a member-sharded rank are
        # its own: only their order within the rank moves)
        presampled = [lu.sample_move_and_augment(buffer=buffer, batch_size=B, augmenter=augmenter, aug_mix=aug_mix, per=per)
                      for _ in range(E)]
        q_weights = _member_target_q(presampled, target_agent, N, B)
        g_lo = parallel.my_range()[0]

    def member_step(i):
        loss_v = loss_all[2 * i:2 * i + 2]
        with (torch.cuda.stream(pipe.front) if pipe is not None else contextlib.nullcontext()):
            rd = presampled[i] if presampled is not None else lu.sample_move_and_augment(
                buffer=buffer, batch_size=B, augmenter=augmenter, aug_mix=aug_mix, per=per)
            if pipe is not None:
                batch_ready = torch.cuda.Event()
                batch_ready.record(pipe.front)
            td_target, (s1_rep, _) = lu.compute_td_targets(
                logs=logs, replay_dict=rd, agent=agent, target_agent=target_agent, ensemble_idx=i,
                ensemble_n=target_critic_ensemble_n, log_alphas=log_alphas, pop=pop, gamma=gamma, random_process=None,
                noise_clip=None, discrete=True)
            if pipe is not None:
                target_ready = torch.cuda.Event()
                target_ready.record(pipe.front)
                pipe.keep.append((rd, td_target, s1_rep))
        if pipe is not None:
            main.wait_event(batch_ready)
        w = lu.compute_backup_weights(logs=logs, replay_dict=rd, agent=agent, target_agent=target_agent,
                                      weight_type=weight_type, weight_temp=weighted_bellman_temp, batch_size=B, discrete=True,
                                      _q_all=None if q_weights is None else q_weights[:, g_lo + i].contiguous())
        o, a, *_ = rd["primary_batch"]
        s_rep = agent.encoder(o)
        need_ds = torch.is_tensor(s_rep) and s_rep.requires_grad
        X, ld = _rows(s_rep)
        S = X.shape[1]
        act = _actions(a, B)
        q, h1, h2 = _forward(ca, i * N, N, X, ld, B, keep=True)               # [N,B,A]: every net's whole Q row
        popart = agent.popart[i]
        imp = rd["imp_weights"].float().contiguous() if per else None          # per=False: ones(1), i.e. no weighting
        dy = torch.empty((N, B, A), dtype=torch.float32, device=dev)
        if pipe is not None:
            main.wait_event(target_ready)
        L.discrete_critic_loss_seed(q.data_ptr(), N, B, A, act.data_ptr(), td_target.data_ptr(),
                                    w.data_ptr() if torch.is_tensor(w) else None, None if imp is None else imp.data_ptr(),
                                    popart.state_ptr() if popart else None, int(bool(pop)), En, parallel.n_global(N),
                                    dy.data_ptr(), loss_v.data_ptr(), stream)
        extra, extra_scale, f1 = None, 0.0, None
        if dr3_coeff > 0:
            # DR3 (learning.py:100-108): second forward on s1; both feature sets carry gradient
            X1, ld1 = _rows(s1_rep)
            _, h1b, h2b = _forward(ca, i * N, N, X1, ld1, B, keep=True)
            extra_scale = lu._dr3_term(logs, ca, i, N, B, E, h2, h2b, dr3_coeff, loss_v)
            extra, f1 = h2b, (X1, ld1, h1b, h2b)
        dxg = torch.empty((N, B, S), dtype=torch.float32, device=dev) if need_ds else None
        _ops.mlp_backward(ca, i * N, N, X, B, h1, h2, dy, ldx=ld, dh2_extra=extra, extra_scale=extra_scale, want_dw=True,
                          accumulate=False, dx=dxg, lddx=S)
        if f1 is not None:
            X1, ld1, h1b, h2b = f1
            _ops.mlp_backward(ca, i * N, N, X1, B, h1b, h2b, None, ldx=ld1, dh2_extra=h2, extra_scale=extra_scale,
                              want_dw=True, accumulate=True)
        if need_ds:
            enc_outs.append((s_rep, dxg.sum(0)))
        return rd

    replay_dicts = lu._run_members(E, dev, False, member_step)
    return lu._critic_tail(logs, loss_all, loss_slot, replay_dicts, buffer, agent, opt, pipe, critic_clip, encoder_optimizer,
                           encoder_clip, enc_outs, update_priorities)


def online_actor_update(buffer, agent, pop, actor_optimizer, log_alphas, batch_size, clip, augmenter, aug_mix,
                        premade_replay_dicts, per):
    """learning.py:344-421 with discrete=True: the critics are evaluated without gradient (:384-387), so the backward
    is the actor's own MLP only."""
    _check(agent)
    lu.pipeline_barrier()
    aa, ca = agent._actor_arena, agent._critic_arena
    dev = aa.device
    L, stream = _lib.lib(), _lib.stream_ptr()
    E, N, B, A = agent.ensemble_size, agent.num_critics, batch_size, agent.act_space_size
    En = parallel.members_global(E)
    logs = _logs.DeviceLogs(dev)
    loss_all, loss_slot = logs.slots(E)
    opt = _arena.FlatAdam.attach(actor_optimizer, aa)

    def member_step(i):
        rd = lu._member_replay_dict(premade_replay_dicts, i, buffer, B, augmenter, aug_mix, per)
        o, *_ = rd["primary_batch"]
        with torch.no_grad():  # actor gradients do not train the encoder (learning.py:378-380)
            s_rep = agent.encoder(o)
        X, ld = _rows(s_rep)
        logits, h1, h2 = _forward(aa, i, 1, X, ld, B, keep=True)
        # [N,B,A]; critics sharded over ranks: every rank's rows gathered.  No gradient flows back through the critics
        # (learning.py:384-387), so nothing else is exchanged: the actor backward and Adam run replicated
        q = _global_q(_forward(ca, i * N, N, X, ld, B), "actor_q")
        popart = agent.popart[i]
        dlogits = torch.empty((1, B, A), dtype=torch.float32, device=dev)
        L.discrete_actor_seed(logits.data_ptr(), q.data_ptr(), q.shape[0], B, A, log_alphas[i].data_ptr(),
                              popart.state_ptr() if popart else None, int(bool(pop)), En, dlogits.data_ptr(),
                              loss_all[i:i + 1].data_ptr(), stream)
        _ops.mlp_backward(aa, i, 1, X, B, h1, h2, dlogits, ldx=ld, want_dw=True, accumulate=False)

    lu._run_members(E, dev, False, member_step)
    lu._actor_tail(logs, aa, opt, clip, E, "gradients/random_actor_online_grad", loss_all)
    logs.defer("losses/actor_pg_loss", [loss_slot + i for i in range(E)])
    return logs.finalize()


def alpha_update(buffer, agent, optimizers, batch_size, log_alphas, augmenter, aug_mix, target_entropy,
                 premade_replay_dicts):
    """learning.py:222-263 with discrete=True: logp = sum_a p log p (the policy's negative entropy, :252-253)."""
    _check(agent)
    lu.pipeline_barrier()
    aa = agent._actor_arena
    dev = aa.device
    L, stream = _lib.lib(), _lib.stream_ptr()
    E, B, A = agent.ensemble_size, batch_size, agent.act_space_size
    logs = _logs.DeviceLogs(dev)

    def member_step(i):
        rd = lu._member_replay_dict(premade_replay_dicts, i, buffer, B, augmenter, aug_mix, False)
        o, *_ = rd["primary_batch"]
        with torch.no_grad():
            s_rep = agent.encoder(o)
        X, ld = _rows(s_rep)
        logits = _forward(aa, i, 1, X, ld, B)
        plogp = torch.empty(B, dtype=torch.float32, device=dev)
        L.discrete_neg_entropy(logits.data_ptr(), B, A, plogp.data_ptr(), stream)
        lu._alpha_step(logs, i, optimizers[i], log_alphas[i], plogp, B, target_entropy)

    lu._run_members(E, dev, False, member_step)
    return logs.finalize()


def _advantage(agent, replay_dict, ensemble_idx, want_priority=False, logits_all=None):
    """Indirect advantage of a discrete agent (adv_estimator.py:45-56): A(s,a) = Q_min(s,a) - sum_a' pibar(a'|s) Q_min(s,a')
    with pibar the mean policy of ALL actors and Q_min member ``ensemble_idx``'s critics (+ its PopArt layer).  Critics
    sharded over ranks: Q_min runs over every rank's critics (one all-gather).  Members sharded over ranks: the caller
    hands every rank's actors' logits on this batch as ``logits_all`` [E_global, B, A] (``_member_policies``).
    Returns (adv [B], mask [B], priority float64 [B] or None) like learning_utils._advantage."""
    _check(agent)
    o, a, *_ = replay_dict["primary_batch"]
    i, E, N, A = ensemble_idx, agent.ensemble_size, agent.num_critics, agent.act_space_size
    if logits_all is None and parallel.members_sharded():
        raise NotImplementedError("member-sharded ensembles: the advantage needs every rank's actors on the batch, which "
                                  "offline_actor_update exchanges (filter_=True)")
    L, stream = _lib.lib(), _lib.stream_ptr()
    with torch.no_grad():
        s_rep = agent.encoder(o)
    X, ld = _rows(s_rep)
    B, dev = X.shape[0], X.device
    logits = _forward(agent._actor_arena, 0, E, X, ld, B) if logits_all is None else logits_all   # [E,B,A]: every actor
    q = _global_q(_forward(agent._critic_arena, i * N, N, X, ld, B), "adv_q")                      # [N,B,A]
    act = _actions(a, B)
    popart = agent.popart[i]
    adv = torch.empty(B, dtype=torch.float32, device=dev)
    mask = torch.empty(B, dtype=torch.float32, device=dev)
    prio = torch.empty(B, dtype=torch.float64, device=dev) if want_priority else None
    L.discrete_advantage(logits.data_ptr(), logits.shape[0], q.data_ptr(), q.shape[0], B, A, act.data_ptr(),
                         popart.state_ptr() if popart else None, adv.data_ptr(), mask.data_ptr(),
                         None if prio is None else prio.data_ptr(), stream)
    return adv, mask, prio


def _member_policies(rds, agent, B):
    """Members sharded over ranks: every rank's actors on every member's batch -> [E_global (actor), E_global (batch), B, A].
    The local batches' states go to every rank, each rank runs its local actors over all E_global*B rows in one grouped
    forward, and the logits come back (two exchanges)."""
    E, A = len(rds), agent.act_space_size
    with torch.no_grad():
        x_all = parallel.all_gather_members(torch.stack([_rows(agent.encoder(rd["primary_batch"][0]))[0] for rd in rds]))
    En, S = x_all.shape[0], x_all.shape[2]
    logits = _forward(agent._actor_arena, 0, E, x_all.view(En * B, S), S, En * B)   # [E, En*B, A]
    return parallel.all_gather_members(logits).view(En, En, B, A)


def offline_actor_update(buffer, agent, actor_optimizer, encoder_optimizer, batch_size, actor_clip, update_encoder,
                         encoder_clip, augmenter, actor_lambda, aug_mix, premade_replay_dicts, per, filter_):
    """learning.py:144-219 with discrete=True (learning_utils.py:241-269): advantage-filtered log-likelihood of the data
    actions under the categorical policy."""
    _check(agent)
    if actor_lambda:
        raise NotImplementedError("action invariance regulariser (lambda = 0 in every shipped config) is out of scope")
    if parallel.members_sharded() and per:
        raise NotImplementedError("member-sharded ensembles: the priority refresh needs every actor on the batch")
    lu.pipeline_barrier()
    aa = agent._actor_arena
    dev = aa.device
    L, stream = _lib.lib(), _lib.stream_ptr()
    E, B, A = agent.ensemble_size, batch_size, agent.act_space_size
    En = parallel.members_global(E)
    logs = _logs.DeviceLogs(dev)
    loss_all, loss_slot = logs.slots(E)
    opt = _arena.FlatAdam.attach(actor_optimizer, aa)
    enc_outs, adv = [], []
    rds, pols = None, None
    if filter_ and parallel.members_sharded():
        # pibar of member i's batch needs every rank's actors on it: all local batches first (the discrete filter draws
        # nothing, so the draws keep their order), then one exchange of states and one of logits
        rds = [lu._member_replay_dict(premade_replay_dicts, i, buffer, B, augmenter, aug_mix, per) for i in range(E)]
        pols = _member_policies(rds, agent, B)
        g_lo = parallel.my_range()[0]

    def member_step(i):
        rd = rds[i] if rds is not None else lu._member_replay_dict(premade_replay_dicts, i, buffer, B, augmenter, aug_mix, per)
        o, a, *_ = rd["primary_batch"]
        mask = None
        if filter_:
            _, mask, _ = _advantage(agent, rd, i, logits_all=None if pols is None else pols[:, g_lo + i].contiguous())
            adv[:] = [logs.put_tensor("losses/adv_weights_mean", mask.mean())]
        if update_encoder:
            s_rep = agent.encoder(o)
        else:
            with torch.no_grad():
                s_rep = agent.encoder(o)
        need_ds = torch.is_tensor(s_rep) and s_rep.requires_grad
        X, ld = _rows(s_rep)
        S = X.shape[1]
        logits, h1, h2 = _forward(aa, i, 1, X, ld, B, keep=True)
        act = _actions(a, B)
        dlogits = torch.empty((1, B, A), dtype=torch.float32, device=dev)
        L.discrete_bc_seed(logits.data_ptr(), act.data_ptr(), None if mask is None else mask.data_ptr(), B, A, En,
                           dlogits.data_ptr(), loss_all[i:i + 1].data_ptr(), stream)
        logs.defer(f"losses/filterd_bc_loss_{parallel.member_id(i)}", loss_slot + i)
        dxg = torch.empty((1, B, S), dtype=torch.float32, device=dev) if need_ds else None
        _ops.mlp_backward(aa, i, 1, X, B, h1, h2, dlogits, ldx=ld, want_dw=True, accumulate=False, dx=dxg, lddx=S)
        if need_ds:
            enc_outs.append((s_rep, dxg[0]))
        return rd

    replay_dicts = lu._run_members(E, dev, False, member_step)
    enc_net = lu._encoder_step(agent, encoder_optimizer, encoder_clip, enc_outs)
    if parallel.members_sharded():   # the per-member slots stay: the overall loss is summed into a slot of its own
        total, total_slot = logs.slots(1)
        torch.sum(loss_all, 0, keepdim=True, out=total)
        logs.defer("losses/filtered_bc_overall_loss", total_slot, transform=lambda v: v / En)
    else:
        total = None
        logs.defer("losses/filtered_bc_overall_loss", [loss_slot + i for i in range(E)], transform=lambda v: v / E)
    lu._actor_tail(logs, aa, opt, actor_clip, E, "gradients/actor_offline_grad_norm", total, *adv)
    lu._log_encoder_grad_norm(logs, agent, enc_net, enc_outs, "gradients/encoder_offline_actorloss_grad_norm")
    if per:
        lu.adjust_priorities(logs, replay_dicts[-1], agent, buffer)
    return logs.finalize()

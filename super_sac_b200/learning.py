"""The update entry points, drop-in for reference learning.py: critic_update (:18-141), online_actor_update
(:344-421), alpha_update (:222-263), offline_actor_update (:144-219).

Same signatures, same returned log keys, same arithmetic (fp32) -- but every member's critics run as one grouped
launch, the backward is explicit (no autograd tape on the ensemble), Adam is one fused pass over the flat parameter
arena, and the logged scalars come back with a single device->host copy.  The caller still owns the optimizer
objects, ``log_alphas`` and the target agent exactly as main.py:188-244 / :321 builds them.

This module holds the continuous member bodies and routes ``discrete=True`` to discrete.py.  The skeleton around the
bodies -- pipeline eligibility, member batches, member stream lanes, the encoder step, the logged gradient norms and
the temperature step -- is shared with discrete.py and lives in learning_utils ("shared pieces of the updates").
"""
import contextlib

import torch

from . import _arena, _encoder_opt, _lib, _logs, _ops, _rng, discrete as _discrete, graphed, parallel
from . import learning_utils as lu


def _encoder_has_grad_path(s_rep):
    return torch.is_tensor(s_rep) and s_rep.requires_grad


def _opt_sig(opt):
    pg = opt.param_groups[0]
    return (id(opt), pg["lr"], tuple(pg["betas"]), pg["eps"], pg["weight_decay"])


def _graphable(agent, random_process, per, update_priorities, encoder_optimizer=None):
    """Static shapes, device-side randomness (incl. the exploration-noise scale, GaussianExplorationNoise.scale_dev), no
    PyTorch autograd hand-off -- a parameterised encoder only if it is the native pixel encoder with its fused optimiser
    step (_encoder_opt.structurally_eligible) --, no host-side decisions."""
    return (graphed.auto_graphs_enabled() and isinstance(_rng.source(), _rng.PhiloxSource) and not per and
            not update_priorities and (random_process is None or hasattr(random_process, "scale_dev")) and
            not parallel.sharded() and
            (not lu._encoder_trainable(agent) or _encoder_opt.structurally_eligible(agent.encoder, encoder_optimizer)))


def critic_update(buffer, agent, target_agent, critic_optimizer, encoder_optimizer, log_alphas, batch_size, gamma,
                  critic_clip, encoder_clip, target_critic_ensemble_n, weighted_bellman_temp, weight_type, pop,
                  augmenter, encoder_lambda, random_process, noise_clip, aug_mix=0.75, discrete=False, per=False,
                  update_priorities=False, dr3_coeff=0.0):
    """Drop-in for reference learning.py:18-141.  With ``graphed.enable_auto_graphs()`` repeated calls with the same
    objects and hyper-parameters replay a captured CUDA graph."""
    args = (buffer, agent, target_agent, critic_optimizer, encoder_optimizer, log_alphas, batch_size, gamma, critic_clip,
            encoder_clip, target_critic_ensemble_n, weighted_bellman_temp, weight_type, pop, augmenter, encoder_lambda,
            random_process, noise_clip, aug_mix, discrete, per, update_priorities, dr3_coeff)
    # (a discrete critic update reads no random_process: the exploration process a training loop passes does not matter)
    if not encoder_lambda and _graphable(agent, None if discrete else random_process, per, update_priorities,
                                         encoder_optimizer):
        key = ("critic", id(buffer), id(agent), id(target_agent), _opt_sig(critic_optimizer), id(encoder_optimizer),
               id(random_process),
               tuple(id(l) for l in log_alphas), batch_size, gamma, critic_clip, encoder_clip, target_critic_ensemble_n,
               weighted_bellman_temp, weight_type, pop, id(augmenter), noise_clip, aug_mix, dr3_coeff, discrete,
               _lib.lib().default_mlp_impl())
        opt = _arena.FlatAdam.attach(critic_optimizer, agent._critic_arena)

        enc_trained = lu._encoder_trainable(agent)

        def on_replay():
            opt.note_replayed_step()
            if enc_trained:
                _encoder_opt.note_replayed_step(agent.encoder, encoder_optimizer)
            buffer.total_sample_calls += agent.ensemble_size

        refs = (buffer, agent, target_agent, critic_optimizer, encoder_optimizer, tuple(log_alphas), augmenter, random_process)
        # cross-call pipelining (graphed._Cross) covers what lu.pipelined_updates covers, minus PopArt (device state that
        # both sides of an update touch)
        # (discrete updates: not yet, their captures launch one after the other)
        cross_ok = (not discrete and agent.ensemble_size == 1 and weight_type is None and not any(bool(p) for p in agent.popart)
                    and lu.side_stream(agent._critic_arena.device) is not None and not enc_trained)
        return graphed.run_cached(key, lambda: _critic_update_impl(*args), on_replay, refs=refs, cross_ok=cross_ok)
    graphed.join()
    return _critic_update_impl(*args)


def _critic_update_impl(buffer, agent, target_agent, critic_optimizer, encoder_optimizer, log_alphas, batch_size, gamma,
                        critic_clip, encoder_clip, target_critic_ensemble_n, weighted_bellman_temp, weight_type, pop,
                        augmenter, encoder_lambda, random_process, noise_clip, aug_mix=0.75, discrete=False, per=False,
                        update_priorities=False, dr3_coeff=0.0):
    lu.check_batch_sharding(agent, encoder_optimizer, per, update_priorities, weight_type, weighted_bellman_temp, dr3_coeff,
                            discrete, augmenter, batch_size)
    if discrete:   # SAC-Discrete (learning.py:84-92, learning_utils.py:322-328): discrete.py
        return _discrete.critic_update(buffer, agent, target_agent, critic_optimizer, encoder_optimizer, log_alphas,
                                       batch_size, gamma, critic_clip, encoder_clip, target_critic_ensemble_n,
                                       weighted_bellman_temp, weight_type, pop, augmenter, encoder_lambda, aug_mix, per,
                                       update_priorities, dr3_coeff)
    if encoder_lambda:
        raise NotImplementedError("encoder invariance regulariser (lambda = 0 in every shipped config) is out of scope")
    ca = agent._critic_arena
    dev = ca.device
    _ops.check_cuda(ca.flat)
    L = _lib.lib()
    E, N, B_all = agent.ensemble_size, agent.num_critics, batch_size
    lo, hi = parallel.batch_range(B_all)   # batch sharded over ranks: this rank's rows of the global batch
    B = hi - lo
    S, A = lu._dims(agent)
    # Software pipelining across consecutive updates (lu.pipelined_updates): the target side of this update runs on the
    # front stream, which is NOT joined at the end of the update -- the next update's target side starts next to this
    # update's backward / Adam.
    # Critics sharded over ranks: the exchange of the target values (put + wait, parallel.all_gather_q) belongs to the target
    # side and moves to the front stream with it -- its round trip over NVLink then runs under the previous update's
    # backward.  Both halves of an exchange site stay safe: put(k+2) follows wait(k+1) on the front stream, and a peer's
    # put(k+1) follows ITS wait(k), so nobody still reads the half that put(k+2) overwrites.
    pipe = lu._critic_pipeline(agent, per, update_priorities, weight_type)
    # (the log buffer is cleared by the first member's draw kernel, i.e. on the front stream when pipelined: it then has to
    # come from that stream's allocator pool -- a block recycled from the caller's stream could still be in use by the
    # previous update's backward -- and must not be recycled before the block ends)
    if pipe is not None:
        # (first: order the front stream behind whatever it depends on -- under graph capture this is also what makes it
        # part of the capture, and an allocation on a stream outside the capture would invalidate it)
        pipe.front_wait_dep(torch.cuda.current_stream(dev))
    with (torch.cuda.stream(pipe.front) if pipe is not None else contextlib.nullcontext()):
        logs = _logs.DeviceLogs(dev, zeroed=False)
    if pipe is not None:
        pipe.keep.append(logs)
    loss_all, loss_slot = logs.slots(2 * E)   # per member: {loss contribution, mean td error of its last net}
    opt = _arena.FlatAdam.attach(critic_optimizer, ca)
    if parallel.critics_sharded() and E != 1:
        raise NotImplementedError("critic sharding covers one member (REDQ / SAC shapes); SUNRISE members shard as a whole")

    enc_outs = []
    lu._mark("start")
    En = parallel.members_global(E)   # loss normalisation: the global ensemble size when members are sharded over ranks
    presampled, q_weights = None, None

    def draw_member():
        draws = lu.draw_for_critic_member(buffer, agent, B_all, target_critic_ensemble_n, random_process, per,
                                          zero=logs.take_unzeroed())
        lu._mark("draws (indices, eps, subset)")
        return draws, lu.sample_move_and_augment(buffer=buffer, batch_size=B_all, augmenter=augmenter, aug_mix=aug_mix,
                                                 per=per, _idx=draws["idx"])

    if parallel.members_sharded() and weight_type is not None and weighted_bellman_temp is not None and En > 1:
        if weight_type != "sunrise":
            raise NotImplementedError("member-sharded ensembles exchange the sunrise weights only")
        # every local member samples first; then ONE exchange: all batches to all ranks, every rank's target critics on
        # every batch, the values back (parallel.py)
        presampled = [draw_member() for _ in range(E)]
        if any(lu._packed_of(rd) is None for _, rd in presampled):
            raise NotImplementedError("member-sharded sunrise weights need state observations (packed batches)")
        x_all = parallel.all_gather_members(torch.stack([lu._packed_of(rd)["XA"] for _, rd in presampled]))   # [En,B,S+A]
        q_loc = torch.stack([lu._critic_values(target_agent, 0, E * N, x_all[e].contiguous(), B).reshape(E * N, B)
                             for e in range(En)], dim=1)                                                    # [E*N,En,B]
        q_weights = parallel.all_gather_members(q_loc)                                                      # [En*N,En,B]
        g_lo = parallel.my_range()[0]
    # Members are independent once their batches are drawn (the draws share one device-side Philox offset and stay in
    # order): with more than one member each runs on its own stream lane, forked from / joined into the caller's stream.
    # (softmax weights draw policy samples inside the member's work: those stay serial, in the reference's draw order)
    concurrent = (E > 1 and not per and lu.side_stream(dev) is not None and not lu._encoder_trainable(agent)
                  and weight_type != "softmax")
    if concurrent and presampled is None:
        presampled = [draw_member() for _ in range(E)]

    def member_step(i, draws, rd, lane, batch_ready=None):
        loss_v = loss_all[2 * i:2 * i + 2]
        lu._mark("replay gather")
        o, a, *_ = rd["primary_batch"]
        packed = lu._packed_of(rd)
        s_rep = agent.encoder(o)
        need_ds = _encoder_has_grad_path(s_rep)
        X = lu._first_layer_input(s_rep, a, packed["XA"] if packed else None, S, A)
        h1 = torch.empty((N, B, ca.H), dtype=torch.float32, device=dev)
        h2 = torch.empty_like(h1)
        q = torch.empty((N, B, 1), dtype=torch.float32, device=dev)
        dq = torch.empty((N, B, 1), dtype=torch.float32, device=dev)
        W1, b1, W2, b2, W3, b3 = ca.ptrs(i * N)
        # The online critics' hidden layers do not depend on the TD target: run them on a second stream next to the
        # target actor -> target critics chain (their grids leave most SMs idle), join before the output layer + loss.
        side = None if need_ds else lu.side_stream(dev, lane)
        piped = pipe is not None and side is not None
        if pipe is not None and not piped:
            lu.pipeline_barrier()
        # With scalar-output critics the TD-error seed factors out of the data-gradient chain (ssac_mlp_backward_pre /
        # _post), so that chain runs on the second stream as well, before the TD target exists; after the loss only the
        # three weight-gradient reductions remain.
        split_bwd = side is not None and ca.O == 1 and ca.D <= 32 and not dr3_coeff and L.default_mlp_impl() == 2
        bws = _ops._bwd_ws(N, B, ca.H, dev) if split_bwd else None
        if side is not None:
            main = torch.cuda.current_stream(dev)
            if piped:
                # the online branch stays on the caller's stream (nothing else runs there before the loss); it needs the
                # batch, which the front stream gathered
                online = main
                main.wait_event(batch_ready)
                pipe.cross_before_online(main)
            else:
                online = side
                side.wait_stream(main)
            L.critic_forward_loss(W1, b1, W2, b2, W3, b3, N, ca.D, ca.H, X.data_ptr(), S + A, B, h1.data_ptr(),
                                  h2.data_ptr(), None, None, None, None, None, 0, En, 0, None, None, 1,
                                  None, 0, None, None, None, None, 0.0, None, None, 0, online.cuda_stream)
            if split_bwd:
                L.mlp_backward_pre(W2, W3, N, ca.H, B, h1.data_ptr(), h2.data_ptr(), bws.data_ptr(), 1, 0, online.cuda_stream)
        with (torch.cuda.stream(pipe.front) if piped else contextlib.nullcontext()):
            td_target, (s1, a1) = lu.compute_td_targets(
                logs=logs, replay_dict=rd, agent=agent, target_agent=target_agent, log_alphas=log_alphas, ensemble_idx=i,
                ensemble_n=target_critic_ensemble_n, pop=pop, gamma=gamma, random_process=random_process,
                noise_clip=noise_clip, _draws=draws,
                # (batch sharded over several ranks: the TD target kernel's statistics are pooled over the ranks)
                _fuse_into_loss=side is not None and not (parallel.batches_sharded() and parallel.world_size() > 1))
            if piped:
                target_ready = torch.cuda.Event()
                target_ready.record(pipe.front)
                pipe.keep.append((draws, rd, td_target, getattr(td_target, "_ssac_pending", None), s1, a1))
        tdp = getattr(td_target, "_ssac_pending", None)   # TD target evaluated inside the loss kernel
        w = lu.compute_backup_weights(logs=logs, replay_dict=rd, agent=agent, target_agent=target_agent,
                                      weight_type=weight_type, weight_temp=weighted_bellman_temp, batch_size=B,
                                      _q_all=None if q_weights is None else
                                      q_weights[:, g_lo + i, :].reshape(En * N, B, 1).contiguous())
        popart = agent.popart[i]
        imp = rd["imp_weights"]
        imp_ptr = imp.float().contiguous() if per else None  # per=False: ones(1), i.e. no weighting (main.py:401)
        if piped:
            main.wait_event(target_ready)
        elif side is not None:
            main.wait_stream(side)
        # N critic forwards + loss value + seed gradient dL/dq in one entry point (loss seed fused into the head kernel)
        L.critic_forward_loss(W1, b1, W2, b2, W3, b3, N, ca.D, ca.H, X.data_ptr(), S + A, B, h1.data_ptr(), h2.data_ptr(),
                              q.data_ptr(), td_target.data_ptr(), w.data_ptr() if torch.is_tensor(w) else None,
                              None if imp_ptr is None else imp_ptr.data_ptr(), popart.state_ptr() if popart else None,
                              int(bool(pop)), En, parallel.n_global(N), dq.data_ptr(), loss_v.data_ptr(), 2 if side is not None else 0,
                              *((tdp["qt"].data_ptr(), tdp["M"], _ops._p(tdp["logp"]), tdp["log_alpha"].data_ptr(),
                                 tdp["r"].data_ptr(), tdp["d"].data_ptr(), tdp["gamma"], td_target.data_ptr(),
                                 tdp["logs"].data_ptr()) if tdp else (None, 0, None, None, None, None, 0.0, None, None)),
                              0, _lib.stream_ptr())
        lu._batch_share_(B, B_all, dq, loss_v)
        lu._mark("join online hidden layers + output layer + loss seed")
        extra, extra_scale, f1 = None, 0.0, None
        if dr3_coeff > 0:
            # DR3 (learning.py:100-108): second forward on (s1, a1); both feature sets carry gradient
            X1 = packed["X1"] if packed else torch.cat((s1, a1), dim=-1).contiguous()
            _, h1b, h2b = lu._critic_values(agent, i * N, N, X1, B, keep=True)
            extra_scale = lu._dr3_term(logs, ca, i, N, B, E, h2, h2b, dr3_coeff, loss_v)
            extra, f1 = h2b, (X1, h1b, h2b)
        dxg = torch.empty((N, B, S + A), dtype=torch.float32, device=dev) if need_ds else None
        if pipe is not None:
            pipe.cross_before_grads(torch.cuda.current_stream(dev))
        if split_bwd:
            gW1, gb1, gW2, gb2, gW3, gb3 = ca.ptrs(i * N, grad=True)
            L.mlp_backward_post(W3, N, ca.D, ca.H, X.data_ptr(), S + A, 0, B, h1.data_ptr(), h2.data_ptr(), dq.data_ptr(),
                                bws.data_ptr(), gW1, gb1, gW2, gb2, gW3, gb3, 0, _lib.stream_ptr())
        else:
            _ops.mlp_backward(ca, i * N, N, X, B, h1, h2, dq, ldx=S + A, dh2_extra=extra, extra_scale=extra_scale,
                              want_dw=True, accumulate=False, dx=dxg, lddx=S + A)
        if f1 is not None:
            X1, h1b, h2b = f1
            _ops.mlp_backward(ca, i * N, N, X1, B, h1b, h2b, None, ldx=S + A, dh2_extra=h2, extra_scale=extra_scale,
                              want_dw=True, accumulate=True)
        if need_ds:
            enc_outs.append((s_rep, dxg.sum(0)[:, :S]))
        lu._mark("ensemble backward")
        return rd

    def run_member(i):
        if presampled is not None:
            draws, rd = presampled[i]
        elif pipe is not None:
            with torch.cuda.stream(pipe.front):
                draws, rd = draw_member()
                pipe.cross_after_gather()
                batch_ready = torch.cuda.Event()
                batch_ready.record(pipe.front)
            return member_step(i, draws, rd, 0, batch_ready)
        else:
            draws, rd = draw_member()
        return member_step(i, draws, rd, i % lu.MEMBER_LANES if concurrent else 0)

    replay_dicts = lu._run_members(E, dev, concurrent, run_member)
    return lu._critic_tail(logs, loss_all, loss_slot, replay_dicts, buffer, agent, opt, pipe, critic_clip, encoder_optimizer,
                           encoder_clip, enc_outs, update_priorities)


def online_actor_update(buffer, agent, pop, actor_optimizer, log_alphas, batch_size, clip, random_process, noise_clip,
                        augmenter, aug_mix, premade_replay_dicts=None, per=False, discrete=False, use_baseline=False):
    """Drop-in for reference learning.py:344-421 (graph-replayed under ``graphed.enable_auto_graphs()`` when the replay
    dicts come from a graph-replayed critic update, i.e. are the same static buffers on every call)."""
    args = (buffer, agent, pop, actor_optimizer, log_alphas, batch_size, clip, random_process, noise_clip, augmenter,
            aug_mix, premade_replay_dicts, per, discrete, use_baseline)
    # Graph the actor update only over the STATIC buffers of a graph-captured critic update: eager critic updates hand
    # out fresh replay dicts every step (whose ids CPython recycles), and a graph captured over those would replay on
    # freed memory.
    if (not use_baseline and premade_replay_dicts is not None
            and all(graphed.is_static(rd) for rd in premade_replay_dicts)
            and _graphable(agent, None if discrete else random_process, per, False)):
        key = ("actor", id(agent), _opt_sig(actor_optimizer), tuple(id(l) for l in log_alphas), batch_size, clip, pop,
               tuple(id(rd) for rd in premade_replay_dicts), _lib.lib().default_mlp_impl(), id(random_process), noise_clip,
               discrete)
        opt = _arena.FlatAdam.attach(actor_optimizer, agent._actor_arena)
        refs = (agent, actor_optimizer, tuple(log_alphas), tuple(premade_replay_dicts), random_process)
        return graphed.run_cached(key, lambda: _online_actor_update_impl(*args), opt.note_replayed_step, refs=refs)
    return _online_actor_update_impl(*args)


def _online_actor_update_impl(buffer, agent, pop, actor_optimizer, log_alphas, batch_size, clip, random_process,
                              noise_clip, augmenter, aug_mix, premade_replay_dicts=None, per=False, discrete=False,
                              use_baseline=False):
    if use_baseline:
        raise NotImplementedError("advantage baselines are out of scope")
    lu.check_batch_sharding(agent, per=per, discrete=discrete,
                            augmenter=augmenter if premade_replay_dicts is None else None, batch_size=batch_size)
    if discrete:   # learning.py:382-390
        return _discrete.online_actor_update(buffer, agent, pop, actor_optimizer, log_alphas, batch_size, clip, augmenter,
                                             aug_mix, premade_replay_dicts, per)
    lu.pipeline_barrier()
    aa, ca = agent._actor_arena, agent._critic_arena
    dev = aa.device
    _ops.check_cuda(aa.flat)
    L = _lib.lib()
    E, N, B_all = agent.ensemble_size, agent.num_critics, batch_size
    lo, hi = parallel.batch_range(B_all)   # batch sharded over ranks: this rank's rows of the global batch
    B = hi - lo
    En = parallel.members_global(E)   # loss normalisation: the global ensemble size when members are sharded over ranks
    S, A = lu._dims(agent)
    logs = _logs.DeviceLogs(dev)
    loss_all, loss_slot = logs.slots(E)   # one slot per member (members may run side by side)
    opt = _arena.FlatAdam.attach(actor_optimizer, aa)
    # members are independent given their batches and their N(0,1) draws: drawn in order on the caller's stream, then one
    # stream lane per member (as in critic_update)
    concurrent = (E > 1 and premade_replay_dicts is not None and lu.side_stream(dev) is not None
                  and not parallel.critics_sharded())

    def draw_member():   # (batch sharded: drawn for the global batch, rows [lo, hi) kept)
        eps = torch.empty((B_all, A), dtype=torch.float32, device=dev)
        _rng.source().normal(eps)
        noise = None
        if agent.deterministic and random_process is not None:
            noise = torch.empty((B_all, A), dtype=torch.float32, device=dev)
            _rng.source().normal(noise)
        return eps[lo:hi], None if noise is None else noise[lo:hi]

    predrawn = [draw_member() for _ in range(E)] if concurrent else None

    def member_step(i):
        rd = lu._member_replay_dict(premade_replay_dicts, i, buffer, B_all, augmenter, aug_mix, per)
        # batch sharded: the N(0,1) draws follow the batch's, as _policy_sample's do on one GPU (one Philox stream)
        eps, noise = predrawn[i] if concurrent else draw_member() if parallel.batches_sharded() else (None, None)
        loss_v = loss_all[i:i + 1]
        o, *_ = rd["primary_batch"]
        packed = lu._packed_of(rd)
        with torch.no_grad():  # actor gradients do not train the encoder (learning.py:378-380)
            s_rep = agent.encoder(o)
        XPI = lu._first_layer_input(s_rep, None, packed["XPI"] if packed else None, S, A)
        pol = lu._policy_sample(agent, i, XPI, B, S, A, random_process, noise_clip, rsample=True, eps=eps, noise=noise)
        q, h1c, h2c = lu._critic_values(agent, i * N, N, XPI, B, keep=True)
        popart = agent.popart[i]
        entropy_on = pol["logp"] is not None
        if parallel.critics_sharded():
            # every rank sees all N_global values, picks the arg-min net per row, and back-propagates only the rows
            # whose arg-min critic it owns; the partial dL/da are summed below
            q_all = parallel.all_gather_q(q, site="actor_q")
            Ng = q_all.shape[0]
            dq_all = torch.empty((Ng, B, 1), dtype=torch.float32, device=dev)
            L.actor_loss_seed(q_all.data_ptr(), Ng, B, pol["logp"].data_ptr() if entropy_on else None,
                              log_alphas[i].data_ptr(), popart.state_ptr() if popart else None, int(bool(pop)), En, None,
                              dq_all.data_ptr(), loss_v.data_ptr(), _lib.stream_ptr())
            lo, hi = parallel.my_range()
            dq = dq_all[lo:hi].contiguous()
        else:
            dq = torch.empty((N, B, 1), dtype=torch.float32, device=dev)
            L.actor_loss_seed(q.data_ptr(), N, B, pol["logp"].data_ptr() if entropy_on else None,
                              log_alphas[i].data_ptr(), popart.state_ptr() if popart else None, int(bool(pop)), En, None,
                              dq.data_ptr(), loss_v.data_ptr(), _lib.stream_ptr())
            lu._batch_share_(B, B_all, dq, loss_v)
        # through the critics to the action: input-gradient only (the reference's critic dW here is discarded anyway)
        da = torch.empty((B, A), dtype=torch.float32, device=dev)
        if ca.O == 1 and A <= 32:
            cW1, _, cW2, _, cW3, _ = ca.ptrs(i * N)
            bws = _ops._bwd_ws(N, B, ca.H, dev)
            L.mlp_backward_dact(cW1, cW2, cW3, N, ca.D, ca.H, S, A, B, h1c.data_ptr(), h2c.data_ptr(), dq.data_ptr(),
                                da.data_ptr(), bws.data_ptr(), 0, _lib.stream_ptr())
        else:
            dxg = torch.empty((N, B, S + A), dtype=torch.float32, device=dev)
            _ops.mlp_backward(ca, i * N, N, XPI, B, h1c, h2c, dq, ldx=S + A, want_dw=False, dx=dxg, lddx=S + A)
            L.sum_groups(dxg.data_ptr(), N, B, S + A, S, A, da.data_ptr(), _lib.stream_ptr())
        if parallel.critics_sharded():
            parallel.all_reduce_sum_(da, site="actor_da")
        O = aa.O
        dout = torch.empty((1, B, O), dtype=torch.float32, device=dev)
        if agent.deterministic:
            L.det_head_backward(pol["tanh_out"].data_ptr(), da.data_ptr(), A, B, A, dout.data_ptr(), _lib.stream_ptr())
        else:
            L.tanh_normal_backward(pol["out"].data_ptr(), pol["eps"].data_ptr(), B, A, float(agent.log_std_low),
                                   float(agent.log_std_high), da.data_ptr(), A, 1.0 / (En * B_all),
                                   log_alphas[i].data_ptr(), dout.data_ptr(), _lib.stream_ptr())
        _ops.mlp_backward(aa, i, 1, XPI, B, pol["h1"], pol["h2"], dout, ldx=S + A, want_dw=True, accumulate=False)

    lu._run_members(E, dev, concurrent, member_step)
    lu._actor_tail(logs, aa, opt, clip, E, "gradients/random_actor_online_grad", loss_all)
    logs.defer("losses/actor_pg_loss", [loss_slot + i for i in range(E)])
    return logs.finalize()


def alpha_update(buffer, agent, optimizers, batch_size, log_alphas, augmenter, aug_mix, target_entropy,
                 premade_replay_dicts, discrete):
    lu.check_batch_sharding(agent, discrete=discrete, augmenter=augmenter if premade_replay_dicts is None else None,
                            batch_size=batch_size)
    if discrete:   # learning.py:252-253
        return _discrete.alpha_update(buffer, agent, optimizers, batch_size, log_alphas, augmenter, aug_mix, target_entropy,
                                      premade_replay_dicts)
    lu.pipeline_barrier()
    dev = agent._actor_arena.device
    E, B_all = agent.ensemble_size, batch_size
    lo, hi = parallel.batch_range(B_all)   # batch sharded over ranks: this rank's rows, the mean over the global batch
    B = hi - lo
    S, A = lu._dims(agent)
    logs = _logs.DeviceLogs(dev)
    # one stream lane per member once the N(0,1) draws are made (in order, on the caller's stream), as in critic_update
    concurrent = E > 1 and premade_replay_dicts is not None and lu.side_stream(dev) is not None

    def draw_eps():   # (batch sharded: drawn for the global batch, rows [lo, hi) kept)
        eps = torch.empty((B_all, A), dtype=torch.float32, device=dev)
        _rng.source().normal(eps)
        return eps[lo:hi]

    predrawn = [draw_eps() for _ in range(E)] if concurrent and not agent.deterministic else None

    def member_step(i):
        rd = lu._member_replay_dict(premade_replay_dicts, i, buffer, B_all, augmenter, aug_mix, False)
        eps = predrawn[i] if predrawn is not None else None
        if eps is None and parallel.batches_sharded() and not agent.deterministic:
            eps = draw_eps()   # after the batch's draws, as _policy_sample's on one GPU (one Philox stream)
        o, *_ = rd["primary_batch"]
        with torch.no_grad():
            s_rep = agent.encoder(o)
        X = torch.empty((B, S + A), dtype=torch.float32, device=dev)
        X[:, :S].copy_(s_rep)
        pol = lu._policy_sample(agent, i, X, B, S, A, None, None, eps=eps)
        lu._alpha_step(logs, i, optimizers[i], log_alphas[i], pol["logp"], B_all, target_entropy)

    lu._run_members(E, dev, concurrent, member_step)
    return logs.finalize()


def offline_actor_update(buffer, agent, actor_optimizer, encoder_optimizer, batch_size, actor_clip, update_encoder,
                         encoder_clip, augmenter, actor_lambda, aug_mix, premade_replay_dicts=None, per=True,
                         discrete=False, filter_=True):
    """AFBC / behaviour cloning actor update (reference learning.py:144-219, learning_utils.py:241-269)."""
    if parallel.batches_sharded():
        raise NotImplementedError("batch sharding does not cover the offline actor update")
    if discrete:   # learning_utils.py:257-258: Categorical log-likelihood, indirect advantage filter
        return _discrete.offline_actor_update(buffer, agent, actor_optimizer, encoder_optimizer, batch_size, actor_clip,
                                              update_encoder, encoder_clip, augmenter, actor_lambda, aug_mix,
                                              premade_replay_dicts, per, filter_)
    if actor_lambda:
        raise NotImplementedError("action invariance regulariser (lambda = 0 in every shipped config) is out of scope")
    if agent.deterministic:
        raise NotImplementedError("filtered behaviour cloning needs a stochastic actor")
    lu.pipeline_barrier()
    aa = agent._actor_arena
    dev = aa.device
    _ops.check_cuda(aa.flat)
    L, stream = _lib.lib(), _lib.stream_ptr()
    E, B = agent.ensemble_size, batch_size
    En = parallel.members_global(E)   # loss normalisation: the global ensemble size when members are sharded over ranks
    S, A = lu._dims(agent)
    logs = _logs.DeviceLogs(dev)
    opt = _arena.FlatAdam.attach(actor_optimizer, aa)
    total, total_slot = logs.slots(1)
    enc_outs, adv = [], []

    def member_step(i):
        rd = lu._member_replay_dict(premade_replay_dicts, i, buffer, B, augmenter, aug_mix, per)
        o, a, *_ = rd["primary_batch"]
        if filter_:
            _, mask, _ = lu._advantage(agent, rd, i)
            adv[:] = [logs.put_tensor("losses/adv_weights_mean", mask.mean())]
        else:
            mask = torch.ones((B,), dtype=torch.float32, device=dev)
        if update_encoder:
            s_rep = agent.encoder(o)
        else:
            with torch.no_grad():
                s_rep = agent.encoder(o)
        need_ds = _encoder_has_grad_path(s_rep)
        X = torch.empty((B, S + A), dtype=torch.float32, device=dev)
        X[:, :S].copy_(s_rep.detach())
        out, h1, h2 = lu._actor_forward(agent, i, X, B, S, A)
        logp = torch.empty((B,), dtype=torch.float32, device=dev)
        dlogp = mask * (-1.0 / (B * En))
        dout = torch.empty((1, B, aa.O), dtype=torch.float32, device=dev)
        a_c = a.contiguous() if a.stride(-1) != 1 else a
        L.tanh_normal_logprob(out.data_ptr(), a_c.data_ptr(), a_c.stride(0), B, A, float(agent.log_std_low),
                              float(agent.log_std_high), logp.data_ptr(), dlogp.data_ptr(), dout.data_ptr(), stream)
        member_loss = -(logp * mask).mean()
        logs.put_tensor(f"losses/filterd_bc_loss_{parallel.member_id(i)}", member_loss)
        total.add_(member_loss / En)
        dxg = torch.empty((1, B, S + A), dtype=torch.float32, device=dev) if need_ds else None
        _ops.mlp_backward(aa, i, 1, X, B, h1, h2, dout, ldx=S + A, want_dw=True, accumulate=False, dx=dxg, lddx=S + A)
        if need_ds:
            enc_outs.append((s_rep, dxg[0, :, :S]))
        return rd

    replay_dicts = lu._run_members(E, dev, False, member_step)
    # (s_rep carries gradient only with update_encoder: the same fused clip + Adam as in critic_update)
    enc_net = lu._encoder_step(agent, encoder_optimizer, encoder_clip, enc_outs)
    logs.defer("losses/filtered_bc_overall_loss", total_slot)
    lu._actor_tail(logs, aa, opt, actor_clip, E, "gradients/actor_offline_grad_norm", total, *adv)
    lu._log_encoder_grad_norm(logs, agent, enc_net, enc_outs, "gradients/encoder_offline_actorloss_grad_norm")
    if per:
        lu.adjust_priorities(logs, replay_dicts[-1], agent, buffer)
    return logs.finalize()


def markov_state_abstraction_update(buffer, agent, optimizer, batch_size, augmenter, aug_mix, discrete, inverse_coeff,
                                    contrastive_coeff, smoothness_coeff, smoothness_max_dist, grad_clip):
    """Reference learning.py:266-341 (self-supervised Markov state abstraction).  Not part of the B200 update path
    (DESIGN 9): it trains the user's encoder and two plain nn.Module heads through autograd; refuse loudly."""
    raise NotImplementedError("markov_state_abstraction_update is out of scope of super_sac_b200 (DESIGN.md section 9); "
                              "run the reference's own function on the agent's encoder / inverse_model / contrastive_model")

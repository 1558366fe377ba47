"""Building blocks of the update step with the reference's names and signatures (reference learning_utils.py).

soft_update / hard_update (:160-167), sample_move_and_augment (:174-214), compute_td_targets (:298-354),
compute_backup_weights (:357-398), filtered_bc_loss (:241-269), adjust_priorities (:288-295), get_grad_norm
(:95-106) and GaussianExplorationNoise (:18-66).  Every tensor stays in HBM; each function enqueues a handful of
kernels from libssac_b200 on the current stream and never synchronises (logged scalars go through _logs.DeviceLogs).
"""
import contextlib
import math
import random

import numpy as np
import torch

# (discrete.py imports this module as well: the two use each other only inside functions, never at import time)
from . import _encoder_opt, _lib, _logs, _ops, _rng, augmentations, discrete as _discrete, graphed, parallel
from ._arena import MLPArena

LOG_SQRT_2PI = math.log(math.sqrt(2 * math.pi))


# ------------------------------------------------------------------------------------------------
# exploration noise (TD3 / DrQv2)
# ------------------------------------------------------------------------------------------------
class GaussianExplorationNoise:
    """sigma-annealed Gaussian action noise.  The numpy branch serves acting; inside the updates only
    ``current_scale`` is read -- noise, clipping and the straight-through clamp to the action bounds run in
    ssac_det_head_forward (reference learning_utils.py:48-59)."""

    def __init__(self, action_space, start_scale=1.0, final_scale=0.1, steps_annealed=1000, eps=1e-6):
        assert start_scale >= final_scale
        self.action_space = action_space
        self.start_scale, self.final_scale, self.steps_annealed = start_scale, final_scale, steps_annealed
        self._scale_dev = None
        self.current_scale = start_scale
        self._scale_slope = (start_scale - final_scale) / steps_annealed
        self.eps = eps
        if not (np.allclose(action_space.low, -1.0) and np.allclose(action_space.high, 1.0)):
            raise NotImplementedError("the fused noise head assumes actions normalised to [-1, 1] (NormActionSpace)")

    @property
    def current_scale(self):
        return self._current_scale

    @current_scale.setter
    def current_scale(self, v):
        self._current_scale = v
        if self._scale_dev is not None:
            self._scale_dev.fill_(float(v))

    def scale_dev(self, device):
        """The current scale as a 1-element device tensor that follows every change of ``current_scale``: the update
        kernels read sigma from it, so a CUDA graph captured over an update keeps annealing with the acting path."""
        if self._scale_dev is None or self._scale_dev.device != torch.device(device):
            self._scale_dev = torch.full((1,), float(self._current_scale), dtype=torch.float32, device=device)
        return self._scale_dev

    def sample(self, action, clip=None, update_schedule=False):
        if isinstance(action, np.ndarray):
            noise = self.current_scale * np.random.randn(*action.shape)
            if clip is not None:
                noise = np.clip(noise, -clip, clip)
            out = np.clip(action + noise, self.action_space.low + self.eps, self.action_space.high - self.eps)
        elif torch.is_tensor(action):
            B, A = action.shape
            nz = torch.empty((B, A), dtype=torch.float32, device=action.device)
            _rng.source().normal(nz)
            out = torch.empty_like(action)
            # identity "head": atanh is not needed, feed the action through the noise/clamp stage only
            noise = self.current_scale * nz
            if clip is not None:
                noise = noise.clamp(-clip, clip)
            clamped = (action + noise).clamp(-1.0 + self.eps, 1.0 - self.eps)
            out = action + (clamped - action).detach()
        else:
            raise ValueError(f"Unrecognized action array type: {type(action)}")
        if update_schedule:
            self.current_scale = max(self.current_scale - self._scale_slope, self.final_scale)
        return out


# ------------------------------------------------------------------------------------------------
# target networks
# ------------------------------------------------------------------------------------------------
_polyak_tables = {}


def _arena_of(module):
    arena = getattr(module, "_arena", None)
    return arena if isinstance(arena, MLPArena) else None


def _multi_table(target, source):
    """Device pointer table for arbitrary module pairs (user encoders); cached per pair, rebuilt if storage moved.
    (The cache keeps the parameter tensors themselves: re-validating is a data_ptr() per tensor, not a walk over the
    module tree on every Polyak step.)"""
    key = (id(target), id(source))
    cur = _polyak_tables.get(key)
    if cur is not None:
        sig, table, max_numel, tp, sp, owners = cur
        if owners[0]() is target and owners[1]() is source and all(
                t.data_ptr() == e[0] and q.data_ptr() == e[1] for t, q, e in zip(tp, sp, sig)):
            return sig, table, max_numel
    tp, sp = list(target.parameters()), list(source.parameters())
    sig = tuple((t.data_ptr(), q.data_ptr(), t.numel()) for t, q in zip(tp, sp))
    if not sig:
        table, max_numel = None, 0
    else:
        for t, q in zip(tp, sp):
            if t.dtype != torch.float32 or q.dtype != torch.float32 or not t.is_contiguous() or not q.is_contiguous():
                raise NotImplementedError("soft_update: parameters must be contiguous fp32")
        flat = [v for e in sig for v in e]
        table = torch.tensor(flat, dtype=torch.int64, device=tp[0].device)
        max_numel = max(e[2] for e in sig)
    import weakref

    _polyak_tables[key] = (sig, table, max_numel, tp, sp, (weakref.ref(target), weakref.ref(source)))
    return sig, table, max_numel


@contextlib.contextmanager
def _polyak_context():
    """Inside a pipelined_updates() block a Polyak step runs on the block's auxiliary stream (see _Pipeline)."""
    p = _pipeline
    if p is None:
        X = graphed.cross_active()
        if X is None:
            yield lambda: None
        else:   # behind the update it follows (its Adam step), on that update's stream; the next update waits for the event
            sp = X.stream_ptrs[X.last]
            with _lib.on_stream(sp):
                yield lambda: _lib.lib().event_record(X.polyak_ptr, sp)
        return
    aux = p.polyak_stream(torch.cuda.current_stream(p.device))
    with torch.cuda.stream(aux):
        yield lambda: p.note_polyak(aux)


def soft_update(target, source, tau):
    """target <- target*(1-tau) + source*tau, bit-exact with the reference (learning_utils.py:160-162)."""
    ta, sa = _arena_of(target), _arena_of(source)
    if ta is not None and sa is not None:
        _ops.check_cuda(ta.flat, sa.flat)
        g0, g1 = target._g0, target._g0 + target.num_critics
        assert (source._g0, source.num_critics) == (target._g0, target.num_critics)
        with _polyak_context() as note:
            _ops.polyak_ranges(ta.flat, sa.flat, ta.range_table(g0, g1), tau)
            note()
        return
    sig, table, max_numel = _multi_table(target, source)
    if table is None:
        return
    _ops.check_cuda(table)
    with _polyak_context() as note:
        _lib.lib().polyak_multi(table.data_ptr(), len(sig), max_numel, float(tau), _lib.stream_ptr())
        note()


def hard_update(target, source):
    """learning_utils.py:165-167 (tau = 1 is exact: t*0 + s*1)."""
    soft_update(target, source, 1.0)


def get_grad_norm(model):
    """sqrt(sum ||p.grad||^2) as a float (learning_utils.py:95-106): one reduction launch per tensor, one sync."""
    grads = [p.grad for p in model.parameters() if p.grad is not None]
    if not grads:
        return 0.0
    acc = torch.zeros(1, dtype=torch.float32, device=grads[0].device)
    L, s = _lib.lib(), _lib.stream_ptr()
    for g in grads:
        g = g.contiguous()
        L.sumsq(g.data_ptr(), g.numel(), acc.data_ptr(), 1, s)
    return float(acc.item()) ** 0.5


def _member_grad_norm_slot(logs, arena, g0, g1, stream=None):
    """Enqueue sum g^2 of nets g0..g1 into a log slot (sqrt taken at finalize)."""
    v, slot = logs.slots(1)   # slots are zero-initialised with the buffer
    L, s = _lib.lib(), (_lib.stream_ptr() if stream is None else stream.cuda_stream)
    for off, n in arena.range_table(g0, g1):
        L.sumsq(arena.grad.data_ptr() + 4 * off, n, v.data_ptr(), 1, s)
    return slot


# ---- stage marks (tools/stage_timeline.py): timing events recorded between the stages of an update, also inside a
# captured CUDA graph (external events).  Off unless a tool sets ``_marks = []``.
_marks = None


def _mark(name):
    if _marks is not None:
        ev = torch.cuda.Event(enable_timing=True, external=True)
        ev.record()
        _marks.append((name, ev))


_side_streams = {}
_member_streams = {}
MEMBER_LANES = 4


def side_stream(device, lane=0):
    """One extra stream per device (and member lane) for the independent branches of an update (online trunk next to
    the target networks, the logged gradient norm next to Adam).  None when overlap is switched off (ssac_set_overlap)
    and for a device without streams."""
    device = torch.device(device)
    if device.type != "cuda" or not _lib.lib().get_overlap():
        return None
    st = _side_streams.get((device, lane))
    if st is None:
        st = _side_streams[(device, lane)] = torch.cuda.Stream(device=device)
    return st


def member_stream(device, lane):
    """Stream of ensemble-member lane ``lane``: the members of a SUNRISE-style ensemble are independent once their
    batches are drawn, so their updates run side by side (each uses at most ~80 of the 148 SMs at a time)."""
    device = torch.device(device)
    st = _member_streams.get((device, lane))
    if st is None:
        st = _member_streams[(device, lane)] = torch.cuda.Stream(device=device)
    return st


# ---- software pipelining of consecutive critic updates ---------------------------------------------------------------
# The only true recurrence between two critic updates runs through the ONLINE critics' parameters (forward -> loss ->
# backward -> Adam -> next forward).  The target side of update k+1 -- index / noise / subset draws, replay gather,
# target actor, target critics -- reads the replay ring, the actor and the TARGET critics only, so inside a
# ``pipelined_updates()`` block it runs on its own stream ("front") next to update k's backward and Adam, ordered by
# events exactly where data flows: the batch before the online forward, the target values before the loss, a Polyak step
# before the next target-critic forward.  Same kernels, same draw order, same numbers as the sequential schedule; it is
# the UTD loop of main.py:380-414 (20 back-to-back updates for REDQ) that offers the overlap.
class _Pipeline:
    def __init__(self, device):
        self.device = device
        self.front = _front_stream(device)
        self.dep = None          # main-stream event the front has to wait for before it reads actor / ring again
        self.polyak = None       # event of the latest Polyak step (the target critics' parameters), for the front stream
        self.polyak_main = None  # the same event, for the caller's stream (its next Adam step)
        self.aux = None          # stream the Polyak steps run on
        self.cross = graphed.cross_capturing()   # (state, slot): this block is ONE update captured for cross-call pipelining
        self.keep = []           # front-allocated tensors that main-stream kernels read: alive until the block ends
        self.needs_order = False  # a barrier happened: the front's next work goes behind the caller's stream as it is then
        # the front has waited on the caller's stream once: before that it holds no work of this block, and under capture
        # waiting on it would be a dependency on work outside the graph (a block whose critic updates all run serially)
        self.forked = False

    def order_front_after_main(self, main):
        ev = torch.cuda.Event()
        ev.record(main)
        self.dep = ev

    def front_wait_dep(self, main):
        if self.needs_order:
            self.order_front_after_main(main)
            self.needs_order = False
        if self.dep is not None:
            self.front.wait_event(self.dep)
            self.dep = None
            self.forked = True
            if self.cross is not None:   # one Philox stream, one set of ring readers: behind the other capture's target side
                X, i = self.cross
                self.front.wait_event(X.gather_done[1 - i])

    def front_wait_polyak(self):
        if self.polyak is not None:
            self.front.wait_event(self.polyak)
            self.polyak = None
        if self.cross is not None:
            self.front.wait_event(self.cross[0].polyak_done)

    # ---- cross-call pipelining (graphed._Cross): external event nodes of the captured update -------------------------
    def cross_after_gather(self):
        if self.cross is not None:
            X, i = self.cross
            X.gather_done[i].record(self.front)

    def cross_before_online(self, main):
        if self.cross is not None:   # the online parameters: behind the other capture's Adam step
            X, i = self.cross
            main.wait_event(X.adam_done[1 - i])

    def cross_before_grads(self, main):
        if self.cross is not None:   # the gradient arrays / backward workspace: behind everything of the other capture
            X, i = self.cross
            main.wait_event(X.tail_done[1 - i])

    def cross_after_adam(self, main):
        if self.cross is not None:
            X, i = self.cross
            X.adam_done[i].record(main)

    def polyak_stream(self, main):
        """Polyak steps run on a stream of their own: they follow the Adam step at the caller's tail, but the caller's next
        online forward does not wait for them (only the next target-critic forward and the next Adam step do)."""
        if self.aux is None:
            self.aux = _aux_stream(self.device)
        self.aux.wait_stream(main)
        return self.aux

    def note_polyak(self, stream):
        ev = torch.cuda.Event()
        ev.record(stream)
        self.polyak = ev
        self.polyak_main = ev

    def main_wait_polyak(self, main):
        """Before the caller's stream overwrites the online parameters (Adam) a Polyak step still reads."""
        if self.polyak_main is not None:
            main.wait_event(self.polyak_main)
            self.polyak_main = None
        if self.cross is not None:
            main.wait_event(self.cross[0].polyak_done)


_pipeline = None
_front_streams = {}
_aux_streams = {}


def _aux_stream(device):
    device = torch.device(device)
    st = _aux_streams.get(device)
    if st is None:
        st = _aux_streams[device] = torch.cuda.Stream(device=device)
    return st


def _front_stream(device):
    device = torch.device(device)
    st = _front_streams.get(device)
    if st is None:
        st = _front_streams[device] = torch.cuda.Stream(device=device)
    return st


def pipeline():
    return _pipeline


@contextlib.contextmanager
def pipelined_updates(device=None):
    """Consecutive ``learning.critic_update`` (+ ``soft_update``) calls inside this block overlap as described above.
    Meant to be captured as ONE CUDA graph (graphed.GraphedCall) or run eagerly; every other update entry point joins the
    two streams first (``pipeline_barrier``).  Do not push to / re-prioritise the buffer inside the block."""
    global _pipeline
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if _pipeline is not None or not _lib.lib().get_overlap():
        yield None
        return
    p = _Pipeline(device)
    p.order_front_after_main(torch.cuda.current_stream(device))
    _pipeline = p
    try:
        yield p
    finally:
        _pipeline = None
        main = torch.cuda.current_stream(device)
        if p.forked:
            main.wait_stream(p.front)
        if p.aux is not None:
            main.wait_stream(p.aux)
        p.keep.clear()


def pipeline_barrier():
    """Join the front stream into the caller's stream and order its next work after the caller's (an entry point that
    changes what the front reads -- actor update, buffer writes -- or draws random numbers on the caller's stream)."""
    p = _pipeline
    if p is None:
        graphed.join()
    if p is not None:
        main = torch.cuda.current_stream(p.device)
        if p.forked:
            main.wait_stream(p.front)
        if p.aux is not None:
            main.wait_stream(p.aux)
            p.polyak_main = None
        p.needs_order = True


# ------------------------------------------------------------------------------------------------
# sampling
# ------------------------------------------------------------------------------------------------
class ReplayDict(dict):
    """The dict of learning_utils.py:208-214.  'augmented_obs' and 'original_obs' (only read by the invariance
    regularisers, lambda = 0 in every shipped config) are produced on first access instead of on every sample."""

    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        self._lazy = {}

    def __missing__(self, key):
        if key in self._lazy:
            val = self._lazy.pop(key)()
            self[key] = val
            return val
        raise KeyError(key)

    def __contains__(self, key):
        return dict.__contains__(self, key) or key in self._lazy


_ones_cache = {}


def _ones1(dev):
    t = _ones_cache.get(dev)
    if t is None:
        t = torch.ones(1, dtype=torch.float32, device=dev)
        _ones_cache[dev] = t
    return t


def _pixel_gather(stack, idx, shift, aug, B, aug_rows, use_aug):
    _, C, H, W = stack.shape
    out = torch.empty((B, C, H, W), dtype=torch.float32, device=stack.device)
    noise = None
    pad_mode = aug.pad_mode if use_aug else augmentations.PAD_NONE
    if use_aug and getattr(aug, "noise", False) and pad_mode != augmentations.PAD_NONE:
        noise = torch.empty((B, C, H, W), dtype=torch.float32, device=stack.device)
        _rng.source().normal(noise)
    _lib.lib().gather_aug_u8(stack.data_ptr(), out.data_ptr(), idx.data_ptr(), None if shift is None else shift.data_ptr(),
                             None if noise is None else noise.data_ptr(), B, C, H, W, int(getattr(aug, "pad", 0)),
                             pad_mode if shift is not None else 0, aug_rows, _lib.stream_ptr())
    return out


def _batch_rows(B, augmenter, per):
    """This rank's rows [lo, hi) of a batch-sharded update's batch of B; refuses what cannot be split row for row."""
    if per:
        raise NotImplementedError("batch sharding: prioritised sampling is not supported (uniform sampling only)")
    if not (isinstance(augmenter, augmentations.AugmentationSequence) and augmenter.fusable()):
        raise NotImplementedError("batch sharding needs a fusable AugmentationSequence (Identity / DrQ / DrQv2)")
    aug = augmenter.aug_list[0]
    if getattr(aug, "noise", False):
        raise NotImplementedError("batch sharding: noisy DrQ augmentation is not supported")
    if getattr(aug, "batch_size", B) != B:
        raise ValueError(f"batch sharding: the augmentation draws {aug.batch_size} shifts for a batch of {B}")
    return parallel.batch_range(B)


def _batch_share_(B, B_all, *ts):
    """Scale per-row gradient seeds and logged means normalised over this rank's B rows to the global batch's B_all (the
    ranks' shares then sum to the single-GPU values); nothing to do when the rank holds the whole batch."""
    if B == B_all:
        return
    scale = torch.full((1,), B / B_all, dtype=torch.float32, device=ts[0].device)
    for t in ts:
        _lib.lib().scale_by_dev(t.data_ptr(), t.numel(), scale.data_ptr(), _lib.stream_ptr())


def check_batch_sharding(agent, encoder_optimizer=None, per=False, update_priorities=False, weight_type=None,
                         weight_temp=None, dr3_coeff=0.0, discrete=False, augmenter=None, batch_size=None):
    """What a batch-sharded update covers (one member, uniform sampling, plain Bellman backups, no PopArt, no DR3, a
    continuous agent, an encoder without parameters or the native pixel encoder with its fused optimiser step, and --
    ``augmenter`` given: the update samples its own batch of ``batch_size`` -- an augmentation that splits row for row):
    anything else raises before the update launches anything."""
    if not parallel.batches_sharded():
        return
    if augmenter is not None:
        _batch_rows(batch_size, augmenter, per)
    why = None
    if discrete:
        why = "SAC-Discrete agents"
    elif agent.ensemble_size != 1:
        why = "ensembles of several members (E > 1)"
    elif per or update_priorities:
        why = "prioritised replay"
    elif weight_type is not None and weight_temp is not None:
        why = "weighted Bellman backups"
    elif dr3_coeff:
        why = "DR3"
    elif any(bool(p) for p in agent.popart):
        why = "PopArt"
    elif _encoder_trainable(agent):
        for net in _encoder_opt.native_nets(agent.encoder):   # (flattened lazily by the first forward otherwise)
            if net._native_params()[0].is_cuda:
                net._flatten()
        if not _encoder_opt.structurally_eligible(agent.encoder, encoder_optimizer):
            why = "trainable encoders other than the native pixel encoder with its fused optimiser step"
    if why is not None:
        raise NotImplementedError(f"batch sharding does not cover {why}")


def sample_move_and_augment(buffer, batch_size, augmenter, aug_mix, per=True, _idx=None):
    """Sample a batch on the device, cast to fp32, augment o and o1 with shared parameters and mix the first
    int(B*aug_mix) augmented rows into the batch (reference learning_utils.py:174-214)."""
    if getattr(buffer, "n_step_mode", False):   # one-step ring, n-step transitions assembled by the sampler (nstep_replay.py)
        return buffer.nstep_sample_move_and_augment(batch_size, augmenter, aug_mix, _idx=_idx, per=per)
    assert len(buffer) >= batch_size
    st, dev, B = buffer._storage, buffer.device, batch_size
    if not torch.cuda.is_current_stream_capturing():
        buffer.total_sample_calls += 1
    fused = isinstance(augmenter, augmentations.AugmentationSequence) and augmenter.fusable()
    shard = _batch_rows(B, augmenter, per) if parallel.batches_sharded() else None
    if per:
        idx, imp_weights = buffer.sample_indices_per(B)
    else:
        idx = _idx if _idx is not None else buffer.sample_indices_uniform(B)
        imp_weights = _ones1(dev)
    aug_rows = int(B * aug_mix)
    if shard is not None:   # indices drawn for the global batch: this rank gathers its rows of it
        lo, hi = shard
        idx, aug_rows, B = idx[lo:hi], parallel.local_aug_rows(B, aug_mix, lo, hi), hi - lo
    rd = ReplayDict()

    a = r = d = None
    if fused:
        aug = augmenter.aug_list[0]
        aug.change_randomization_params(dev)  # once per call; o and o1 share the shifts
        shift = getattr(aug, "shift", None)
        if shard is not None and shift is not None:   # drawn for the global batch (aug.batch_size rows)
            shift = shift[shard[0]:shard[1]]
        aug_keys = st.s_stack.keys() if augmenter.keys is None else augmenter.keys
        o, o1 = {}, {}
        srcs, dsts, rows, lds, modes = [], [], [], [], []
        keys = list(st.s_stack.keys())
        A = st.action_stack[0].numel()
        packed = None
        shifting = getattr(aug, "pad_mode", augmentations.PAD_NONE) != augmentations.PAD_NONE
        if len(keys) == 1 and st.s_stack[keys[0]].dtype == torch.float32 and st.s_stack[keys[0]].dim() == 2 \
                and st.action_stack.dim() == 2:
            if shifting and keys[0] in aug_keys:   # as the general branch below: never skip an augmentation silently
                raise NotImplementedError(f"shift augmentation of non-image key '{keys[0]}'")
            # state observations: gather s|a, s1|. and s|. straight into the [B, S+A] first-layer inputs
            k = keys[0]
            S = st.s_stack[k].shape[1]
            XA = torch.empty((B, S + A), dtype=torch.float32, device=dev)
            X1 = torch.empty((B, S + A), dtype=torch.float32, device=dev)
            XPI = torch.empty((B, S + A), dtype=torch.float32, device=dev)
            o[k], o1[k], a = XA[:, :S], X1[:, :S], XA[:, S:]
            for src, dst, n in ((st.s_stack[k], XA, S), (st.s_stack[k], XPI, S), (st.s1_stack[k], X1, S)):
                srcs.append(src); dsts.append(dst); rows.append(n); lds.append(S + A); modes.append(0)
            srcs.append(st.action_stack); dsts.append(a); rows.append(A); lds.append(S + A); modes.append(0)
            packed = dict(XA=XA, X1=X1, XPI=XPI, S=S, A=A, key=k)
        else:
            for k in keys:
                stack, stack1 = st.s_stack[k], st.s1_stack[k]
                if stack.dtype == torch.uint8 and stack.dim() == 4:
                    use = k in aug_keys
                    o[k] = _pixel_gather(stack, idx, shift, aug, B, aug_rows, use)
                    o1[k] = _pixel_gather(stack1, idx, shift, aug, B, aug_rows, use)
                elif stack.dtype in (torch.float32, torch.uint8):
                    if k in aug_keys and aug.pad_mode != augmentations.PAD_NONE:
                        raise NotImplementedError(f"shift augmentation of non-image key '{k}'")
                    n = stack[0].numel()
                    o[k] = torch.empty((B,) + tuple(stack.shape[1:]), dtype=torch.float32, device=dev)
                    o1[k] = torch.empty_like(o[k])
                    mode = 0 if stack.dtype == torch.float32 else 1
                    for src, dst in ((stack, o[k]), (stack1, o1[k])):
                        srcs.append(src); dsts.append(dst); rows.append(n); lds.append(n); modes.append(mode)
                else:
                    raise NotImplementedError(f"observation dtype {stack.dtype} (key '{k}')")
            a = torch.empty((B, A), dtype=torch.float32, device=dev)
            srcs.append(st.action_stack); dsts.append(a); rows.append(A); lds.append(A); modes.append(0)
        r = torch.empty((B, 1), dtype=torch.float32, device=dev)
        d = torch.empty((B, 1), dtype=torch.float32, device=dev)
        srcs += [st.reward_stack, st.done_stack]; dsts += [r, d]; rows += [1, 1]; lds += [1, 1]; modes += [0, 1]
        _ops.gather_rows(srcs, dsts, rows, lds, modes, idx, B)
        rd["primary_batch"] = (o, a, r, o1, d)
        if packed is not None:
            rd["_packed"] = packed

        def _orig():
            oo, oo1 = {}, {}
            for k in keys:
                stack = st.s_stack[k]
                if stack.dtype == torch.uint8 and stack.dim() == 4:
                    oo[k] = _pixel_gather(stack, idx, None, aug, B, 0, False)
                    oo1[k] = _pixel_gather(st.s1_stack[k], idx, None, aug, B, 0, False)
                else:
                    oo[k], oo1[k] = o[k], o1[k]
            return oo, oo1

        def _augd():
            ao, ao1 = {}, {}
            for k in keys:
                stack = st.s_stack[k]
                if stack.dtype == torch.uint8 and stack.dim() == 4 and k in aug_keys:
                    if getattr(aug, "noise", False):
                        raise NotImplementedError("lazy 'augmented_obs' with noisy DrqAug (noise would be re-drawn)")
                    ao[k] = _pixel_gather(stack, idx, shift, aug, B, B, True)
                    ao1[k] = _pixel_gather(st.s1_stack[k], idx, shift, aug, B, B, True)
                else:
                    ao[k], ao1[k] = o[k], o1[k]
            return ao, ao1

        rd._lazy["original_obs"] = _orig
        rd._lazy["augmented_obs"] = _augd
    else:
        # arbitrary user augmenter (callable on dicts of float tensors): gather + cast here, augment + mix in PyTorch
        s, a, r, s1, dn = st.gather(idx)
        oo = {k: v.float() for k, v in s.items()}
        oo1 = {k: v.float() for k, v in s1.items()}
        a, r, d = a.float(), r.float(), dn.float()
        ao, ao1 = augmenter(oo, oo1)
        o = {k: v.clone() for k, v in oo.items()}
        o1 = {k: v.clone() for k, v in oo1.items()}
        for k in o:
            o[k][:aug_rows] = ao[k][:aug_rows]
            o1[k][:aug_rows] = ao1[k][:aug_rows]
        rd["primary_batch"] = (o, a, r, o1, d)
        rd["augmented_obs"] = (ao, ao1)
        rd["original_obs"] = (oo, oo1)
    rd["priority_idxs"] = idx
    rd["imp_weights"] = imp_weights
    return rd


# ------------------------------------------------------------------------------------------------
# shared pieces of the updates
# ------------------------------------------------------------------------------------------------
def _first_layer_input(rep, act_cols, packed_buf, S, A):
    """[B, S+A] matrix whose first S columns hold ``rep``.  When the encoder returned the packed view itself
    (identity encoders) the gather already put the numbers there and nothing is copied."""
    B = rep.shape[0]
    if packed_buf is not None and rep.data_ptr() == packed_buf.data_ptr() and rep.stride(0) == S + A and rep.shape[1] == S:
        return packed_buf
    X = torch.empty((B, S + A), dtype=torch.float32, device=rep.device)
    X[:, :S].copy_(rep.detach())
    if act_cols is not None:
        X[:, S:].copy_(act_cols)
    return X


def _actor_forward(agent, i, X, B, S, A, keep=False):
    """Run actor i on the first S columns of X [B, S+A].  Returns (out [B,O], h1, h2)."""
    arena = agent._actor_arena
    h1 = torch.empty((1, B, arena.H), dtype=torch.float32, device=X.device)
    h2 = torch.empty_like(h1)
    out = torch.empty((1, B, arena.O), dtype=torch.float32, device=X.device)
    _ops.mlp_forward(arena, i, 1, X, B, h1, h2, out, ldx=S + A)
    return out, h1, h2


def _rows_ok(D, H, O):
    """The row-local CUDA-core kernel (ssac_mlp_rows.cu) covers this shape and is switched on."""
    return bool(_lib.lib().rows_supported(int(D), int(H), int(O)))


def _policy_sample(agent, i, X, B, S, A, random_process, noise_clip, rsample=False, eps=None, noise=None, keep=None):
    """a ~ pi_i(.|s) written into X[:, S:], with log-prob [B] (None when a noise process replaces the entropy term):
    actor MLP + policy head in one entry point (the head is fused into the output-layer kernel).  ``eps`` / ``noise``:
    pre-drawn N(0,1) tensors (drawn here otherwise).  Returns dict(out, h1, h2, eps, logp, tanh_out); h1 / h2 are only
    valid when ``keep`` (default: rsample, i.e. a backward pass follows)."""
    dev = X.device
    keep = rsample if keep is None else keep
    arena = agent._actor_arena
    det = agent.deterministic
    use_rows = (not keep and _lib.lib().default_mlp_impl() == 2 and _rows_ok(S + A, arena.H, arena.O) and A <= 8
                and B <= 64)   # the acting path (B = num_envs); large batches keep the tensor cores
    h1 = h2 = out = None
    if not use_rows:
        h1 = torch.empty((1, B, arena.H), dtype=torch.float32, device=dev)
        h2 = torch.empty_like(h1)
        out = torch.empty((1, B, arena.O), dtype=torch.float32, device=dev)
    a_dst = X[:, S:]
    res = dict(out=out, h1=h1, h2=h2, eps=None, logp=None, tanh_out=None)
    sigma, clip, tanh_out, logp = 0.0, 0.0, None, None
    if det:
        if rsample and eps is None:  # Normal(loc, 1e-4).rsample() of the reference's deterministic "distribution"
            eps = torch.empty((B, A), dtype=torch.float32, device=dev)
            _rng.source().normal(eps)
        if not rsample:
            eps = None
        if random_process is not None:
            if noise is None:
                noise = torch.empty((B, A), dtype=torch.float32, device=dev)
                _rng.source().normal(noise)
            if hasattr(random_process, "scale_dev"):
                # noise <- sigma * noise with sigma read ON THE DEVICE (bit-identical to passing it by value: one product,
                # and 1.0 * x below is exact), so the launch sequence does not depend on the annealing state
                _lib.lib().scale_by_dev(noise.data_ptr(), noise.numel(), random_process.scale_dev(dev).data_ptr(), _lib.stream_ptr())
                sigma = 1.0
            else:
                sigma = float(random_process.current_scale)
            clip = float(noise_clip) if noise_clip is not None else 0.0
        else:
            noise = None
        tanh_out = torch.empty((B, A), dtype=torch.float32, device=dev)
    else:
        if random_process is not None:
            raise NotImplementedError("an exploration-noise process on top of a stochastic actor is not supported")
        if eps is None:
            eps = torch.empty((B, A), dtype=torch.float32, device=dev)
            _rng.source().normal(eps)
        noise = None
        logp = torch.empty((B,), dtype=torch.float32, device=dev)
    W1, b1, W2, b2, W3, b3 = arena.ptrs(i)
    L = _lib.lib()
    if use_rows:
        L.policy_rows(W1, b1, W2, b2, W3, b3, arena.D, arena.H, A, int(det), X.data_ptr(), S + A, B, None, _ops._p(eps),
                      _ops._p(noise), sigma, clip, float(agent.log_std_low), float(agent.log_std_high), a_dst.data_ptr(),
                      S + A, _ops._p(logp), _ops._p(tanh_out), _lib.stream_ptr())
    else:
        L.actor_forward_sample(W1, b1, W2, b2, W3, b3, arena.D, arena.H, A, int(det), X.data_ptr(), S + A, B,
                               h1.data_ptr(), h2.data_ptr(), int(bool(keep)), out.data_ptr(), _ops._p(eps),
                               _ops._p(noise), sigma, clip,
                               float(agent.log_std_low), float(agent.log_std_high), a_dst.data_ptr(), S + A,
                               _ops._p(logp), _ops._p(tanh_out), 0, _lib.stream_ptr())
    res.update(eps=eps, logp=logp, tanh_out=tanh_out)
    if det and random_process is None:
        # Normal(loc, 1e-4).log_prob(loc) summed over A: a constant (nets/distributions.py:107-114)
        const = A * (0.0 - math.log(1e-4) - LOG_SQRT_2PI)
        if rsample and eps is not None:
            # rsample() = loc + 1e-4*eps (learning.py:392): log_prob of that sample carries -eps^2/2 per dimension
            # (no gradient: it does not depend on the parameters; the logged actor loss does)
            res["logp"] = const - 0.5 * (eps * eps).sum(1)
        else:
            res["logp"] = torch.full((B,), const, dtype=torch.float32, device=dev)
    return res


def _critic_values(agent, g0, G, X, B, net_index=None, keep=False):
    """q [G,B] of critic nets g0..g0+G (or the net_index subset relative to g0) on X [B, S+A]."""
    arena = agent._critic_arena
    h1 = torch.empty((G, B, arena.H), dtype=torch.float32, device=X.device)
    h2 = torch.empty_like(h1)
    q = torch.empty((G, B, 1), dtype=torch.float32, device=X.device)
    _ops.mlp_forward(arena, g0, G, X, B, h1, h2, q, ldx=X.shape[1], net_index=net_index, keep_hidden=keep)
    return (q, h1, h2) if keep else q


def _packed_of(replay_dict):
    return replay_dict["_packed"] if "_packed" in replay_dict else None


def _dims(agent):
    return agent._actor_arena.D, agent.act_space_size


def _encoder_trainable(agent):
    ps = agent.__dict__.get("_ssac_encoder_params")
    if ps is None:   # walking the module tree on every update call costs more than the check itself
        ps = agent.__dict__["_ssac_encoder_params"] = [p for p in agent.encoder.parameters() if p.numel() > 2]
    return any(p.requires_grad for p in ps)


def _critic_pipeline(agent, per, update_priorities, weight_type):
    """The active ``pipelined_updates()`` block if this critic update may run its target side on the block's front stream
    (one member, uniform sampling, plain Bellman backups, no trainable encoder, no PopArt), else None after joining the
    front stream.  PopArt stays serial: the next update's TD target rescales the PopArt layer this update's loss seed
    still reads.  Critics sharded over ranks pipeline only over the peer exchange (the NCCL fallback stays serial)."""
    p, dev = _pipeline, agent._critic_arena.device
    if (p is None or agent.ensemble_size != 1 or per or update_priorities or weight_type is not None
            or _encoder_trainable(agent) or any(bool(pa) for pa in agent.popart)
            or (parallel.critics_sharded() and not parallel.peer_exchange_ready()) or parallel.members_sharded()
            or parallel.batches_sharded()
            or side_stream(dev) is None or p.device != dev):
        pipeline_barrier()
        return None
    return p


def _member_replay_dict(premade_replay_dicts, i, buffer, batch_size, augmenter, aug_mix, per):
    """Member i's batch: the one the caller made (the critic update's replay dicts) or a fresh sample."""
    if premade_replay_dicts is not None:
        return premade_replay_dicts[i]
    return sample_move_and_augment(buffer=buffer, batch_size=batch_size, augmenter=augmenter, aug_mix=aug_mix, per=per)


def _run_members(E, device, concurrent, member_step):
    """[member_step(i) for every member i], in order.  ``concurrent``: member i runs on stream lane i % MEMBER_LANES,
    forked from the caller's stream, and every lane used is joined back into it afterwards."""
    if not concurrent:
        return [member_step(i) for i in range(E)]
    caller = torch.cuda.current_stream(device)
    lanes, out = [], []
    for i in range(E):
        st = member_stream(device, i % MEMBER_LANES)
        if st not in lanes:
            lanes.append(st)
            st.wait_stream(caller)
        with torch.cuda.stream(st):
            out.append(member_step(i))
    for st in lanes:
        caller.wait_stream(st)
    return out


def _encoder_step(agent, encoder_optimizer, encoder_clip, enc_outs):
    """Hand the members' input gradients ``enc_outs`` [(s_rep, ds)] to autograd and clip + step the encoder (learning.py:
    117-131).  A native pixel encoder whose gradients sit in its flat buffer takes the fused sumsq + Adam launches
    (_encoder_opt.py); that net is returned, else None."""
    encoder_optimizer.zero_grad()
    if not enc_outs:
        return None
    torch.autograd.backward([s for s, _ in enc_outs], [g for _, g in enc_outs])
    if parallel.batches_sharded():   # the native encoder's flat gradient summed over the ranks' rows
        net = _encoder_opt.eligible(agent.encoder, encoder_optimizer)
        if net is None:
            raise NotImplementedError("batch sharding trains only the native pixel encoder with its fused optimiser step")
        parallel.all_reduce_flat_(net._flat_grad, site="encoder_grad")
    net = _encoder_opt.fused_step(agent.encoder, encoder_optimizer, encoder_clip)
    if net is None:
        if encoder_clip:
            torch.nn.utils.clip_grad_norm_(agent.encoder.parameters(), encoder_clip)
        encoder_optimizer.step()
    return net


def _log_member_grad_norm(logs, arena, E, nets_per_member, key, stream=None):
    """Log the gradient norm of one member picked by ``random.choice`` (the reference's draw: it precedes the one in
    adjust_priorities)."""
    member = random.choice(range(E))
    slot = _member_grad_norm_slot(logs, arena, member * nets_per_member, (member + 1) * nets_per_member, stream=stream)
    logs.defer(key, slot, transform=lambda v: v**0.5)


def _log_encoder_grad_norm(logs, agent, enc_net, enc_outs, key):
    """Log the encoder's (post-clip) gradient norm, 0.0 when no gradient reached it."""
    if enc_net is not None:
        v, slot = logs.slots(1)
        _encoder_opt.grad_norm_sq_into(enc_net, v)
        logs.defer(key, slot, transform=lambda v: v**0.5)
    elif enc_outs:
        gn = torch.linalg.vector_norm(torch.stack([p.grad.norm() for p in agent.encoder.parameters() if p.grad is not None]))
        logs.put_tensor(key, gn)
    else:
        logs[key] = 0.0


def _dr3_term(logs, arena, i, N, B, E, h2, h2b, dr3_coeff, loss_v):
    """DR3 (learning.py:100-108) of member i's N critics from their last hidden layers on s (``h2``) and on s1 (``h2b``):
    logs the dot product, adds dr3 * dot / (E * N) to the member's loss slot ``loss_v`` (learning.py:108,112) and returns
    the scale of the gradient both feature sets carry.  Sharded ensembles normalise over the global ensemble: with the
    critics sharded this rank adds its share N / N_global to the loss (summed over the ranks with the rest of it) and
    the logged dot product is summed right here."""
    Ng, En = parallel.n_global(N), parallel.members_global(E)
    dv, dslot = logs.slots(1)
    _lib.lib().dr3_dot(h2.data_ptr(), h2b.data_ptr(), N, B, arena.H, dv.data_ptr(), _lib.stream_ptr())
    logs.defer(f"dr3_dotproduct_{parallel.member_id(i)}", dslot)
    if Ng != N:
        dv.mul_(N / Ng)
    loss_v[0:1].add_(dv, alpha=dr3_coeff / (En * Ng))
    if parallel.critics_sharded():
        parallel.all_reduce_sum_(dv, site="dr3_dot")
    return dr3_coeff / (En * Ng) / (Ng * B)


def _critic_tail(logs, loss_all, loss_slot, replay_dicts, buffer, agent, opt, pipe, critic_clip, encoder_optimizer,
                 encoder_clip, enc_outs, update_priorities):
    """The end of a critic update once every member's gradients are in: the encoder step, clip + Adam, the logged values
    and the priority refresh.  ``loss_all`` holds two slots per member: its loss contribution and the mean TD error of
    its last net.  Returns what critic_update returns."""
    ca, E, N = agent._critic_arena, agent.ensemble_size, agent.num_critics
    dev, stream = ca.device, _lib.stream_ptr()
    logs.defer("losses/last_member_critic_td_error", loss_slot + 2 * (E - 1) + 1)
    logs.defer("losses/critic_overall_loss", [loss_slot + 2 * i for i in range(E)])

    def logged_values(on=None):
        _log_member_grad_norm(logs, ca, E, N, "gradients/critic_random_grad", stream=on)
        if parallel.batches_sharded():   # each rank's share of the global-batch means: summed over the ranks
            with (torch.cuda.stream(on) if on is not None else contextlib.nullcontext()):
                parallel.all_reduce_sum_(loss_all[0:2], site="critic_loss")
        elif parallel.sharded():   # the loss summed over every rank, the TD error of the ensemble's last net
            with (torch.cuda.stream(on) if on is not None else contextlib.nullcontext()):
                parallel.reduce_logged(loss_all[0:2 * E:2], loss_all[2 * E - 1:2 * E], site="critic_loss")

    enc_net = _encoder_step(agent, encoder_optimizer, encoder_clip, enc_outs)
    if parallel.batches_sharded():   # every rank's share of the batch: clip, log and step the sum
        parallel.all_reduce_flat_(ca.grad, site="critic_grad")
    if critic_clip:
        opt.grad_norm_sq(stream)
        if parallel.sharded() and not parallel.batches_sharded():   # the global norm runs over every rank's critics (SURVEY 8e (3)): one float per rank
            parallel.all_reduce_sum_(opt.gnorm_sq, site="critic_gnorm")
    side = None if critic_clip else side_stream(dev)   # clipping rescales the gradients that get logged
    main = torch.cuda.current_stream(dev) if side is not None or pipe is not None else None
    if side is not None:   # the logged values next to Adam (which only reads the gradients)
        side.wait_stream(main)
        logged_values(side)
    if pipe is not None:
        pipe.main_wait_polyak(main)   # a Polyak step on the auxiliary stream still reads the online parameters
    opt.step(stream, max_norm=critic_clip if critic_clip else None)   # (clipping rescales the stored gradients, as the reference's does)
    if pipe is not None:
        pipe.cross_after_adam(main)
    if side is not None:
        main.wait_stream(side)
    else:
        logged_values()
    _mark("Adam (+ logged grad norm)")
    _log_encoder_grad_norm(logs, agent, enc_net, enc_outs, "gradients/encoder_criticloss_grad_norm")
    if update_priorities:
        adjust_priorities(logs, replay_dicts[-1], agent, buffer)
    return logs.finalize(), replay_dicts


def _actor_tail(logs, arena, opt, clip, E, grad_key, loss_v, last=None):
    """Clip + Adam of the actors and the logged gradient norm of a random member.  Members sharded over ranks: the clip
    norm runs over every rank's actors, the logged loss in ``loss_v`` becomes the sum over every rank's members and
    ``last``, a value of the last member, the last rank's (parallel.reduce_logged).  (With the critics sharded the
    actors are replicas: nothing to exchange.)"""
    stream = _lib.stream_ptr()
    if parallel.batches_sharded():   # every rank's share of the batch; the loss slot holds this rank's share of the mean
        parallel.all_reduce_flat_(arena.grad, site="actor_grad")
        parallel.all_reduce_sum_(loss_v, site="actor_loss")
    if clip:
        opt.grad_norm_sq(stream)
        if parallel.members_sharded():
            parallel.all_reduce_sum_(opt.gnorm_sq, site="actor_gnorm")
    opt.step(stream, max_norm=clip if clip else None)
    _log_member_grad_norm(logs, arena, E, 1, grad_key)
    if parallel.members_sharded():
        parallel.reduce_logged(loss_v, last, site="actor_loss")


class _AlphaState:
    """Adam state of one 1-element ``log_alpha`` optimiser (main.py:230-239), kept on the device."""

    def __init__(self, optimizer, log_alpha):
        self.state = torch.zeros(2, dtype=torch.float32, device=log_alpha.device)
        self.ctl = torch.zeros(2, dtype=torch.int32, device=log_alpha.device)
        st = optimizer.state[log_alpha]
        self._step_tensor = torch.zeros((), dtype=torch.float32)
        self.steps = 0
        if "exp_avg" in st:   # resuming from a loaded optimizer state (optimizer.load_state_dict)
            self.state[0:1].copy_(st["exp_avg"].reshape(1))
            self.state[1:2].copy_(st["exp_avg_sq"].reshape(1))
            self.steps = int(st["step"])
            self.ctl[0] = self.steps
            self._step_tensor.fill_(self.steps)
        st["step"], st["exp_avg"], st["exp_avg_sq"] = self._step_tensor, self.state[0:1], self.state[1:2]

    @classmethod
    def attach(cls, optimizer, log_alpha):
        cur = getattr(optimizer, "_ssac_alpha_state", None)
        st = optimizer.state.get(log_alpha)
        aliased = st is not None and "exp_avg" in st and cur is not None and st["exp_avg"].data_ptr() == cur.state.data_ptr()
        if cur is None or cur.state.device != log_alpha.device or not aliased:   # not aliased: load_state_dict replaced the state
            cur = cls(optimizer, log_alpha)
            optimizer._ssac_alpha_state = cur
        return cur


def _alpha_step(logs, i, optimizer, log_alpha, logp, B, target_entropy):
    """Member i's temperature step (learning.py:246-262) on ``logp`` [B]: loss, scalar Adam and logs (under the global
    member id) in one launch."""
    if parallel.batches_sharded():   # the temperature's mean runs over the global batch B: every rank, the same step
        logp = parallel.all_gather_batch(logp, B, site="alpha_logp")
    pg = optimizer.param_groups[0]
    st = _AlphaState.attach(optimizer, log_alpha)
    lv, slot = logs.slots(2)
    _lib.lib().alpha_step(log_alpha.data_ptr(), logp.data_ptr(), B, float(target_entropy), st.state.data_ptr(),
                          st.ctl.data_ptr(), float(pg["lr"]), float(pg["betas"][0]), float(pg["betas"][1]),
                          float(pg["eps"]), lv.data_ptr(), _lib.stream_ptr())
    st.steps += 1
    st._step_tensor.fill_(st.steps)
    logs.defer(f"losses/alpha_loss_{parallel.member_id(i)}", slot)
    logs.defer(f"alphas/alpha_{parallel.member_id(i)}", slot + 1)


def draw_for_critic_member(buffer, agent, B, ensemble_n, random_process, per, zero=None):
    """Every random draw one member's critic update consumes up front -- replay indices (replay.py:122), the policy's
    N(0,1) draw or the TD3 noise (learning_utils.py:49,330), the REDQ target subset (agent.py:29) -- in ONE launch."""
    dev = buffer.device
    S, A = _dims(agent)
    n_sub_pool = parallel.n_global(agent.num_critics)   # critics sharded over ranks: the subset of the GLOBAL ensemble
    assert 0 < ensemble_n <= n_sub_pool
    idx = None if per else torch.empty(B, dtype=torch.int64, device=dev)
    need_normal = (not agent.deterministic) or (random_process is not None)
    normal = torch.empty((B, A), dtype=torch.float32, device=dev) if need_normal else None
    subset = torch.empty(ensemble_n, dtype=torch.int32, device=dev)
    _rng.source().fill(dev, idx=idx, n_filled=len(buffer), n_filled_dev=buffer._n_filled_dev, normal=normal,
                       subset=subset, N=n_sub_pool, M=ensemble_n, zero=zero)
    if normal is not None and parallel.batches_sharded():   # drawn for the global batch: this rank's rows
        lo, hi = parallel.batch_range(B)
        normal = normal[lo:hi]
    return dict(idx=idx, normal=normal, subset=subset, batch_size=B)


def compute_td_targets(logs, replay_dict, agent, target_agent, ensemble_idx, ensemble_n, log_alphas, pop, gamma,
                       random_process, noise_clip, discrete=False, _draws=None, _fuse_into_loss=False):
    """TD target of one ensemble member (reference learning_utils.py:298-354, continuous branch).
    Returns ``td_target [B,1], (s1_rep, a_s1)``.  ``_fuse_into_loss`` (critic_update only, no PopArt): the final
    reduction is left to the critic loss kernel -- the returned tensor is filled by that launch and carries the operands
    as ``_ssac_pending``."""
    if discrete:   # learning_utils.py:322-328
        return _discrete.compute_td_targets(logs, replay_dict, agent, target_agent, ensemble_idx, ensemble_n, log_alphas, pop,
                                            gamma)
    dlogs, user_logs = _logs.as_device_logs(logs, agent._critic_arena.device)
    o, a, r, o1, d = replay_dict["primary_batch"]
    i = ensemble_idx
    S, A = _dims(agent)
    B = a.shape[0]
    packed = _packed_of(replay_dict)
    popart = agent.popart[i]
    if _pipeline is not None and any(p.numel() > 2 for p in target_agent.encoder.parameters()):
        _pipeline.front_wait_polyak()   # a target encoder with parameters is Polyak-updated as well
    with torch.no_grad():
        s1_rep = target_agent.encoder(o1)
    X1 = _first_layer_input(s1_rep, None, packed["X1"] if packed else None, S, A)
    N = agent.num_critics
    # REDQ subset: drawn over the GLOBAL ensemble when the critics are sharded over ranks (replicated Philox state)
    pool = parallel.n_global(N)
    assert 0 < ensemble_n <= pool
    if _draws is not None:   # critic_update drew indices, policy noise and the subset in ONE launch
        net_index = _draws["subset"]
        pol = _policy_sample(agent, i, X1, B, S, A, random_process, noise_clip,
                             eps=None if agent.deterministic else _draws["normal"],
                             noise=_draws["normal"] if agent.deterministic else None)
    else:
        net_index = torch.empty(ensemble_n, dtype=torch.int32, device=X1.device)
        # (the reference draws the policy sample first, the subset second: learning_utils.py:321, agent.py:29)
        pol = _policy_sample(agent, i, X1, B, S, A, random_process, noise_clip)
        _rng.source().subsets(net_index, pool, ensemble_n)
    if _pipeline is not None:
        _pipeline.front_wait_polyak()   # the target critics' parameters: the only thing this side reads that Polyak writes
    if parallel.critics_sharded():
        # every rank evaluates its own target critics and all-gathers the [N_global, B] values; the subset-min is then
        # identical on every rank
        q_t = parallel.all_gather_q(_critic_values(target_agent, i * N, N, X1, B), site="target_q", select=net_index)
    else:
        q_t = _critic_values(target_agent, i * N, ensemble_n, X1, B, net_index=net_index)
    _mark("target critics Q(s1, a1)")
    y = torch.empty((B, 1), dtype=torch.float32, device=X1.device)
    g = parallel.member_id(i)
    if _fuse_into_loss and not popart and user_logs is None:   # popart is False (reference convention) when off
        lv, slot = dlogs.slots(4)   # {sum (y-c), sum (y-c)^2, sum alpha*logp, c}: zero-initialised with the buffer
        y._ssac_pending = dict(qt=q_t, M=int(ensemble_n), logp=pol["logp"], log_alpha=log_alphas[i], r=r, d=d,
                               gamma=float(gamma), logs=lv)
        dlogs.defer_fn(f"td_targets/mean_td_target_{g}", (slot, slot + 3), lambda s1, c, n=B: c + s1 / n)
        dlogs.defer_fn(f"td_targets/std_td_target_{g}", (slot, slot + 1),
                       lambda s1, s2, n=B: max((s2 - s1 * s1 / n) / (n - 1), 0.0) ** 0.5)
        dlogs.defer_fn(f"td_targets/entropy_bonus_{g}", (slot + 2,), lambda se, n=B: se / n)
        return y, (X1[:, :S], X1[:, S:])
    lv, slot = dlogs.slots(3)
    _lib.lib().td_target(q_t.data_ptr(), ensemble_n, B, None if pol["logp"] is None else pol["logp"].data_ptr(),
                         log_alphas[i].data_ptr(), r.data_ptr(), d.data_ptr(), float(gamma),
                         popart.state_ptr() if popart else None, popart.ctl_ptr() if popart else None,
                         int(bool(pop)), float(popart.beta) if popart else 0.0, int(popart.min_steps) if popart else 0,
                         y.data_ptr(), lv.data_ptr(), _lib.stream_ptr())
    _mark("td target")
    if parallel.batches_sharded() and parallel.world_size() > 1:
        if _draws is None:
            raise NotImplementedError("batch sharding: TD targets are computed inside critic_update")
        _defer_global_td_stats(dlogs, g, lv, _draws["batch_size"])
    else:
        dlogs.defer(f"td_targets/mean_td_target_{g}", slot)
        dlogs.defer(f"td_targets/std_td_target_{g}", slot + 1)
        dlogs.defer(f"td_targets/entropy_bonus_{g}", slot + 2)
    if user_logs is not None:
        user_logs.update(dlogs.finalize())
    return y, (X1[:, :S], X1[:, S:])


def _defer_global_td_stats(dlogs, g, lv, Bg):
    """The logged TD-target statistics of the global batch of Bg rows from every rank's {mean, unbiased std, entropy
    bonus} over its rows: one gather of three floats per rank, pooled (mean, pooled variance) on the host at finalize."""
    world = parallel.world_size()
    allv, slot = dlogs.slots(3 * world)
    allv.view(world, 3).copy_(parallel.all_gather_batch(lv.view(1, 3), world, site="td_stats"))
    n = [hi - lo for lo, hi in (parallel.local_range(Bg, world, r) for r in range(world))]
    slots = tuple(range(slot, slot + 3 * world))
    for j, name in enumerate(("mean_td_target", "std_td_target", "entropy_bonus")):
        dlogs.defer_fn(f"td_targets/{name}_{g}", slots, lambda *v, j=j: pooled_stats(n, v[0::3], v[1::3], v[2::3])[j])


def pooled_stats(n, means, stds, ents):
    """(mean, unbiased std, mean entropy bonus) of a batch split into parts of n[r] rows with the given per-part mean,
    unbiased std and entropy bonus.  A part of one row has no spread of its own (its std, 0/0, is not read)."""
    total = sum(n)
    m = sum(k * x for k, x in zip(n, means)) / total
    ss = sum((k - 1) * s * s if k > 1 else 0.0 for k, s in zip(n, stds)) + sum(k * (x - m) ** 2 for k, x in zip(n, means))
    return m, max(ss / (total - 1), 0.0) ** 0.5, sum(k * e for k, e in zip(n, ents)) / total


def compute_backup_weights(logs, replay_dict, agent, target_agent, weight_type, weight_temp, batch_size, discrete=False,
                           _q_all=None):
    """SUNRISE / softmax weighted Bellman backups (reference learning_utils.py:357-398).  Returns 1.0 or w [B,1].
    ``_q_all`` [E_global*N, B, 1] ([E_global*N, B] for discrete agents): the target critics' values on this member's
    batch, already gathered over the ranks (member-sharded ensembles, parallel.enable_member_sharding)."""
    if weight_type is None or weight_temp is None or parallel.members_global(agent.ensemble_size) == 1:
        return 1.0
    if discrete:   # learning_utils.py:373-376
        return _discrete.compute_backup_weights(logs, replay_dict, agent, target_agent, weight_type, weight_temp, batch_size,
                                                _q_sel=_q_all)
    dlogs, user_logs = _logs.as_device_logs(logs, agent._critic_arena.device)
    o, a, _, o1, _ = replay_dict["primary_batch"]
    S, A = _dims(agent)
    E, N, B = agent.ensemble_size, agent.num_critics, a.shape[0]
    packed = _packed_of(replay_dict)
    dev = a.device
    if _q_all is not None:
        q, E, kind = _q_all, _q_all.shape[0] // N, 0
    elif parallel.members_sharded():
        raise NotImplementedError("member-sharded ensembles: only the sunrise weights are exchanged (through critic_update)")
    elif weight_type == "sunrise":
        with torch.no_grad():
            s_rep = target_agent.encoder(o)
        X = _first_layer_input(s_rep, a, packed["XA"] if packed else None, S, A)
        q = _critic_values(target_agent, 0, E * N, X, B)  # every target net on this member's (s, a): one launch
        kind = 0
    elif weight_type == "softmax":
        with torch.no_grad():
            s1_rep = target_agent.encoder(o1)
        q = torch.empty((E * N, B, 1), dtype=torch.float32, device=dev)
        for j in range(E):
            Xj = torch.empty((B, S + A), dtype=torch.float32, device=dev)
            Xj[:, :S].copy_(s1_rep)
            _policy_sample(agent, j, Xj, B, S, A, None, None)
            q[j * N:(j + 1) * N].copy_(_critic_values(agent, j * N, N, Xj, B))
        kind = 1
    else:
        raise ValueError(f"unknown weight_type {weight_type!r}")
    w = torch.empty((B, 1), dtype=torch.float32, device=dev)
    lv, slot = dlogs.slots(4)
    _lib.lib().backup_weights(q.data_ptr(), E, N, B, float(weight_temp), kind, w.data_ptr(), lv.data_ptr(), _lib.stream_ptr())
    for j, name in enumerate(("mean", "max", "min", "std")):
        dlogs.defer(f"bellman_weights/{name}", slot + j)
    if user_logs is not None:
        user_logs.update(dlogs.finalize())
    return w


def _advantage(agent, replay_dict, ensemble_idx, n=4, want_priority=False):
    """A(s,a) = Q(s,a) - mean_n Q(s, a'~pi) with min-over-N critics and PopArt (reference adv_estimator.py:58-79).
    Returns (adv [B], mask [B], priority float64 [B] or None)."""
    if agent.discrete:   # adv_estimator.py:45-56 ('indirect')
        return _discrete._advantage(agent, replay_dict, ensemble_idx, want_priority=want_priority)
    o, a, *_ = replay_dict["primary_batch"]
    i = ensemble_idx
    S, A = _dims(agent)
    N, B = agent.num_critics, a.shape[0]
    packed = _packed_of(replay_dict)
    dev = a.device
    popart = agent.popart[i]
    L, s = _lib.lib(), _lib.stream_ptr()
    with torch.no_grad():
        s_rep = agent.encoder(o)
    XA = _first_layer_input(s_rep, a, packed["XA"] if packed else None, S, A)
    q_pi = torch.empty((n, B), dtype=torch.float32, device=dev)
    pptr = popart.state_ptr() if popart else None
    # the n policy samples as ONE batch of n*B rows (sample-major): one actor forward, one critic forward and one
    # min-over-nets instead of n of each.  The N(0,1) draws stay n separate fills, in the reference's order.
    Xp = torch.empty((n, B, S + A), dtype=torch.float32, device=dev)
    Xp[:, :, :S].copy_(XA[:, :S].unsqueeze(0).expand(n, B, S))
    eps = None
    if not agent.deterministic:
        eps = torch.empty((n, B, A), dtype=torch.float32, device=dev)
        for j in range(n):
            _rng.source().normal(eps[j])
    Xp2 = Xp.view(n * B, S + A)
    _policy_sample(agent, i, Xp2, n * B, S, A, None, None, eps=None if eps is None else eps.view(n * B, A))
    q = _critic_values(agent, i * N, N, Xp2, n * B)
    L.min_over_nets(q.data_ptr(), N, n * B, pptr, q_pi.data_ptr(), s)
    q = _critic_values(agent, i * N, N, XA, B)
    q_data = torch.empty((B,), dtype=torch.float32, device=dev)
    L.min_over_nets(q.data_ptr(), N, B, pptr, q_data.data_ptr(), s)
    adv = torch.empty((B,), dtype=torch.float32, device=dev)
    mask = torch.empty((B,), dtype=torch.float32, device=dev)
    prio = torch.empty((B,), dtype=torch.float64, device=dev) if want_priority else None
    method = 1 if getattr(agent.adv_estimator, "cont_method", "mean") == "max" else 0
    L.advantage(q_pi.data_ptr(), n, q_data.data_ptr(), B, method, adv.data_ptr(), mask.data_ptr(),
                None if prio is None else prio.data_ptr(), s)
    return adv, mask, prio


def adjust_priorities(logs, replay_dict, agent, buffer):
    """priorities <- relu(A(s,a)) + 1e-4 on the sampled rows, without leaving the device
    (reference learning_utils.py:288-295; critics sharded over ranks with several members: one host broadcast of the
    member, parallel.same_member_choice)."""
    member = parallel.same_member_choice(agent.ensemble_size)
    _, _, prio = _advantage(agent, replay_dict, member, want_priority=True)
    buffer.update_priorities(replay_dict["priority_idxs"], prio)


# ------------------------------------------------------------------------------------------------
# caller-side helpers the reference training loop imports from learning_utils (main.py:249-275, :587)
# ------------------------------------------------------------------------------------------------
class EpsilonGreedyExplorationNoise:
    """Discrete-action counterpart of GaussianExplorationNoise (reference learning_utils.py:69-93): with probability
    ``current_scale`` the whole action array is replaced by uniform random actions; epsilon anneals linearly."""

    def __init__(self, action_space, eps_start=1.0, eps_final=1e-5, steps_annealed=1000):
        assert eps_start >= eps_final
        self.action_space = action_space
        self.eps_start, self.eps_final, self.steps_annealed = eps_start, eps_final, steps_annealed
        self.current_scale = eps_start
        self._eps_slope = (eps_start - eps_final) / steps_annealed

    def sample(self, action, clip=None, update_schedule=False):
        if random.random() < self.current_scale:
            action = np.random.randint(0, self.action_space.n, size=action.shape, dtype=action.dtype)
        if update_schedule:
            self.current_scale = max(self.current_scale - self._eps_slope, self.eps_final)
        return action


def n_step_push(buffer, window, gamma, terminate_traj):
    """Fold a full n-step window [(s, a, r, s1, d), ...] into one transition (s_0, a_0, sum_i gamma^i r_i, s1_last,
    d_last) and push it (main.py:353-365, learning_utils.py:139-151)."""
    s, a, r, s1, d = window.popleft()
    for i, (*_, r_i, s1_i, d_i) in enumerate(window):
        r = r + (gamma ** (i + 1)) * r_i
        s1, d = s1_i, d_i
    buffer.push(s, a, r, s1, d, terminate_traj=terminate_traj)
    return d


def warmup_buffer(buffer, env, warmup_steps, max_episode_steps, n_step, gamma, num_envs=1):
    """Fill the buffer with ``warmup_steps`` random-action transitions (reference learning_utils.py:108-157)."""
    from collections import deque

    state, _ = env.reset()
    done, steps_this_ep = False, 0
    window = deque([], maxlen=n_step)
    for step_num in range(warmup_steps):
        if done:
            state, _ = env.reset()
            done, steps_this_ep = False, 0
            window.clear()
        act = env.action_space.sample()
        if not isinstance(act, np.ndarray):
            act = np.array(act)
            if act.ndim == 0:
                act = np.expand_dims(act, 0)
        if num_envs > 1:
            act = np.array([act for _ in range(num_envs)])
        next_state, reward, terminated, truncated, _ = env.step(act)
        window.append((state, act, reward, next_state, terminated))   # "terminated", not "truncated", is what is stored
        if len(window) == window.maxlen:
            last_d = window[-1][4]
            over = last_d.any() if num_envs > 1 else last_d
            n_step_push(buffer, window, gamma, terminate_traj=over or step_num >= warmup_steps - 1)
        if num_envs > 1:
            done = terminated.any() or truncated.any()
        state = next_state
        steps_this_ep += 1
        if steps_this_ep >= max_episode_steps:
            done = True


def compute_filter_stats(buffer, agent, augmenter, batch_size):
    """Percentage of a uniformly sampled batch that the binary advantage filter accepts (reference
    learning_utils.py:217-238), through the kernel advantage estimator; one scalar read-back."""
    rd = sample_move_and_augment(buffer=buffer, batch_size=batch_size, augmenter=augmenter, aug_mix=0.0, per=False)
    _, mask, _ = _advantage(agent, rd, parallel.same_member_choice(agent.ensemble_size))
    return float(mask.mean().item()) * 100.0

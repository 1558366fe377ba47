"""On-the-fly n-step returns and frame-deduplicated observations (SURVEY 8f N2).

The reference builds n-step transitions on the host at collection time -- a deque of the last n one-step transitions,
``r += gamma**(i+1) * r_i`` in a Python loop, then ``buffer.push(s, a, R_n, s_{t+n}, d)`` (main.py:284,353-365,
learning_utils.py:139-151) -- and its ring stores the observation of every transition twice (``s`` and ``s1`` stacks,
replay.py:10-61); with k stacked frames per observation each frame ends up in the ring 2k times (127 KB per DrQ
transition).

``NStepReplayBuffer`` takes the ONE-step transitions instead, in time order:

* every frame is stored once, in a ring of single frames; the stack ``s_t`` is k consecutive frames of that ring and
  ``s_{t+1}`` the k frames starting one later (``ssac_gather_aug_u8_ring`` reads them in place, shift augmentation and
  uint8 -> fp32 cast fused as before).  Non-image observations are "stacks" of one frame: ``s1_t`` is simply the next
  stored observation.  At the start of an episode all k frames of the first stack are written, so the padding the frame
  stacking wrapper chose is preserved;
* the n-step transition is assembled by the sampler: a FIFO of the slots whose window [t, t+n-1] lies inside one episode
  (exactly the transitions the reference's deque logic pushes: the last n-1 steps of an episode never become a start) is
  kept next to the ring; a uniform draw over that FIFO gives the start, ``ssac_nstep_resolve`` returns
  R = r_t + gamma r_{t+1} + ... (accumulated left to right in the reference's arithmetic: float64 for Python / float64
  rewards, float32 for np.float32 rewards), and the next state / done flag are those of step t+n-1.

``len(buffer)`` is the number of n-step transitions, as in the reference.  The learner keeps using ``gamma ** n_step``
(main.py:388).  One environment (``num_envs == 1``).  ``learning_utils.sample_move_and_augment`` -- hence every update
entry point -- accepts this buffer in place of ``ReplayBuffer``.

Prioritised replay (``prioritized=True``; ``alpha`` / ``beta`` as in ``ReplayBuffer``): a transition is identified by
its slot in the FIFO of valid starts, ``v % size`` with v the running count of starts, and that slot is its leaf in
float64 sum / min trees laid out as ``ReplayBuffer``'s (root at 1, leaves at cap2 + i, cap2 = next power of two >= size).
Until the first start is evicted the v-th start is the v-th tuple the reference's deque pushes, so trees, draws, weights
and updates are bit-identical to a classic prioritised buffer fed those tuples in push order.  A push writes its leaves in
the launch of its field scatter (ssac_push_row_leaves): a completed window gets ``max_priority ** alpha``, an evicted
start (sum 0, min +inf).  After the first eviction a draw covers the whole live mass (root sum) and the weights use N =
number of live transitions (ssac_nstep_tree_sample, DESIGN 5); ``update_priorities`` drops ids whose transition was
evicted after it was sampled (ssac_tree_set_live).  ``sample`` / ``update_priorities`` /
``sample_move_and_augment(per=True)`` raise on a buffer built without ``prioritized=True``.
"""
import ctypes

import numpy as np
import torch

from . import _lib, _ops, _rng, augmentations, graphed, parallel
from .replay import PriorityMax


class NStepReplayBuffer(PriorityMax):
    _STAGE_SLOTS = 16
    n_step_mode = True

    def __init__(self, size, n_step=1, gamma=0.99, frame_stack=1, frame_capacity=None, device=None, validate=True,
                 prioritized=False, alpha=0.6, beta=1.0):
        assert n_step >= 1 and frame_stack >= 1 and size > n_step
        assert alpha >= 0
        self.prioritized, self.alpha, self.beta = bool(prioritized), alpha, beta
        self._init_max_priority()
        self._leaf_writes = []    # (leaf, sum value, min value) of the running push
        self._maxsize, self.n_step, self.gamma, self.frame_stack = int(size), int(n_step), float(gamma), int(frame_stack)
        self.device = torch.device(device if device is not None else "cuda")
        self._frame_cap = int(frame_capacity) if frame_capacity else int(size * 1.05) + 4 * frame_stack + 16
        self._validate = bool(validate)
        self.total_sample_calls = 0
        self._built = False
        # host bookkeeping (time order; slots are positions of the step ring)
        self._head = 0            # slot the next step goes to
        self._n_steps = 0
        self._ep_len = 0          # steps of the running episode stored so far
        self._frames_written = 0  # monotonically increasing frame counter
        self._next_first = 0      # frame counter of the running episode's next state stack
        self._v_head = 0          # valid-start FIFO: entries ever appended
        self._v_tail = 0          #                   entries ever evicted
        self._last_next = None

    # ---- construction on first push --------------------------------------------------------------------------------
    def _build(self, state, action):
        dev, cap, fcap, k = self.device, self._maxsize, self._frame_cap, self.frame_stack
        self.keys = list(state.keys())
        self._frame_shape, self._frame_dtype, self._stacked = {}, {}, {}
        self.frames = {}
        for key in self.keys:
            arr = np.asarray(state[key])
            stacked = arr.ndim == 3 and k > 1
            if stacked and arr.shape[0] % k != 0:
                raise ValueError(f"observation '{key}': {arr.shape[0]} channels are not {k} stacked frames")
            shape = ((arr.shape[0] // k,) + arr.shape[1:]) if stacked else arr.shape
            tdt = torch.uint8 if arr.dtype == np.uint8 else torch.float32
            self._frame_shape[key], self._frame_dtype[key], self._stacked[key] = shape, arr.dtype if tdt == torch.uint8 else np.float32, stacked
            self.frames[key] = torch.zeros((fcap,) + tuple(shape), dtype=tdt, device=dev)
        A = int(np.asarray(action).reshape(-1).shape[0])
        self.action = torch.zeros((cap, A), dtype=torch.float32, device=dev)
        self.done = torch.zeros((cap, 1), dtype=torch.uint8, device=dev)
        self.first_frame = torch.zeros(cap, dtype=torch.int64, device=dev)
        self.valid_ring = torch.zeros(cap, dtype=torch.int64, device=dev)
        self.scalars = torch.zeros(3, dtype=torch.int64, device=dev)   # {n_valid, v_tail % size, v_tail}
        self._n_filled_dev = self.scalars[0:1]   # what the index draw kernel reads (learning_utils.draw_for_critic_member)
        self.reward = None   # created by the first reward: float64 or float32 ring (see module docstring)
        self.gamma_pows = torch.tensor([self.gamma ** i for i in range(self.n_step)], dtype=torch.float64, device=dev)
        self._is_start = np.zeros(cap, dtype=bool)
        self._first_frame_host = np.zeros(cap, dtype=np.int64)
        # one pinned staging row holds every field of the largest push (an episode start: k + 1 frames per key)
        row = sum((k + 1) * ((r[0].numel() * r.element_size() + 15) // 16 * 16) for r in self.frames.values()) + 16 * 16 + A * 4
        # ... and the leaf writes of a push: at most k + 2 evicted starts (a push overwrites at most k + 1 frames, each the
        # first frame of at most one step, plus the step the full ring drops) and the completed window
        self._max_leaf_writes = k + 3
        if self.prioritized:
            cap2 = 1
            while cap2 < cap:
                cap2 *= 2
            self._capacity = cap2
            self._it_sum = torch.zeros(2 * cap2, dtype=torch.float64, device=dev)
            self._it_min = torch.full((2 * cap2,), float("inf"), dtype=torch.float64, device=dev)
            row += 24 * self._max_leaf_writes + 16
        self._stage = torch.empty((self._STAGE_SLOTS, (row + 4095) // 4096 * 4096), dtype=torch.uint8).pin_memory()
        self._stage_dev = torch.empty(self._stage.shape, dtype=torch.uint8, device=dev)
        self._stage_np = self._stage.numpy()
        self._stage_next = 0
        self._built = True

    def _make_reward_ring(self, reward):
        self._reward_f32 = isinstance(reward, np.float32) or (isinstance(reward, np.ndarray) and reward.dtype == np.float32)
        self.reward = torch.zeros(self._maxsize, dtype=torch.float32 if self._reward_f32 else torch.float64, device=self.device)

    def __len__(self):
        return self._v_head - self._v_tail

    # ---- push ------------------------------------------------------------------------------------------------------
    def _evict_oldest_step(self):
        tail = (self._head - self._n_steps) % self._maxsize
        if self._is_start[tail]:
            self._is_start[tail] = False
            if self.prioritized:
                self._leaf_writes.append((self._v_tail % self._maxsize, 0.0, float("inf")))
            self._v_tail += 1
        self._n_steps -= 1

    def push(self, state, action, reward, next_state, done, terminate_traj=None, **kwargs):
        """One ONE-step transition of the running episode (time order).  ``done`` = terminated, ``terminate_traj`` = the
        episode ends here for any reason (main.py:365 passes both; defaults to ``done``)."""
        graphed.before_push()
        action = np.asarray(action, dtype=np.float32).reshape(-1)
        if not self._built:
            self._build(state, action)
        if self.reward is None:
            self._make_reward_ring(reward)
        k, cap, fcap = self.frame_stack, self._maxsize, self._frame_cap
        fields = []   # (numpy array, destination device pointer)
        new_episode = self._ep_len == 0
        if self._validate and not new_episode:
            for key in self.keys:
                if not np.array_equal(np.asarray(state[key]), self._last_next[key]):
                    raise ValueError(f"NStepReplayBuffer.push: '{key}' of this state is not the previous next_state "
                                     "(one-step transitions must arrive in time order; pass terminate_traj=True on the last one)")
        n_new = (k if new_episode else 0) + 1
        # frames that are about to be overwritten must not belong to a live step: evict from the oldest step on
        while self._n_steps > 0 and self._first_frame_host[(self._head - self._n_steps) % cap] < self._frames_written + n_new - fcap:
            self._evict_oldest_step()
        if self._n_steps == cap:
            self._evict_oldest_step()
        if new_episode:
            self._next_first = self._frames_written
        for key in self.keys:
            st, nx = np.asarray(state[key]), np.asarray(next_state[key])
            fshape, fdt = self._frame_shape[key], self._frame_dtype[key]
            ring = self.frames[key]
            fbytes = ring[0].numel() * ring.element_size()
            cf = fshape[0] if self._stacked[key] else None
            if self._validate and self._stacked[key] and not np.array_equal(nx[:-cf], st[cf:]):
                raise ValueError(f"NStepReplayBuffer.push: next_state['{key}'] is not state['{key}'] shifted by one frame")
            c = self._frames_written
            if new_episode:
                parts = [st[j * cf:(j + 1) * cf] for j in range(k)] if self._stacked[key] else [st] * 1
                if not self._stacked[key] and k > 1:
                    parts = [st] * k   # a non-stacked key keeps the common frame counter: k copies at the episode start
                for part in parts:
                    fields.append((np.ascontiguousarray(part, dtype=fdt), ring.data_ptr() + (c % fcap) * fbytes))
                    c += 1
            newest = nx[-cf:] if self._stacked[key] else nx
            fields.append((np.ascontiguousarray(newest, dtype=fdt), ring.data_ptr() + (c % fcap) * fbytes))
        self._frames_written += n_new
        p = self._head
        # the state stack of this step starts k-1 frames before its newest frame
        first = self._next_first
        self._next_first += 1
        self._first_frame_host[p] = first
        rdt = np.float32 if self._reward_f32 else np.float64
        fields.append((action, self.action.data_ptr() + p * self.action.shape[1] * 4))
        fields.append((np.asarray([reward], dtype=rdt), self.reward.data_ptr() + p * self.reward.element_size()))
        fields.append((np.asarray([bool(done)], dtype=np.uint8), self.done.data_ptr() + p))
        fields.append((np.asarray([first], dtype=np.int64), self.first_frame.data_ptr() + 8 * p))
        self._ep_len += 1
        self._n_steps += 1
        self._head = (p + 1) % cap
        if self._ep_len >= self.n_step:   # the window that ends at this step is complete: its first step becomes a start
            start = (p - self.n_step + 1) % cap
            self._is_start[start] = True
            fields.append((np.asarray([start], dtype=np.int64), self.valid_ring.data_ptr() + 8 * (self._v_head % cap)))
            if self.prioritized:   # replay.py:129 (push with priorities=None)
                v = self._max_priority ** self.alpha
                self._leaf_writes.append((self._v_head % cap, v, v))
            self._v_head += 1
        fields.append((np.asarray([self._v_head - self._v_tail, self._v_tail % cap, self._v_tail], dtype=np.int64),
                       self.scalars.data_ptr()))
        end = bool(done) if terminate_traj is None else bool(terminate_traj)
        if end:
            self._ep_len = 0
            self._last_next = None
        elif self._validate:
            self._last_next = {key: np.array(next_state[key], copy=True) for key in self.keys}
        leaves, self._leaf_writes = self._leaf_writes, []
        self._flush(fields, leaves)

    def _flush(self, fields, leaves=()):
        """All fields of one push through ONE pinned staging row per <= 15 fields (ssac_push_row: one H2D copy + one
        scatter kernel).  The leaf writes ride in the last row and its launch (ssac_push_row_leaves)."""
        L = _lib.lib()
        assert len(leaves) <= self._max_leaf_writes
        last = (len(fields) - 1) // 15 * 15
        for i in range(0, len(fields), 15):
            chunk = fields[i:i + 15]
            slot = self._stage_next
            self._stage_next = (slot + 1) % self._STAGE_SLOTS
            row, off = self._stage_np[slot], 0
            n = len(chunk)
            dsts, nbytes, offs = (ctypes.c_void_p * n)(), (ctypes.c_int64 * n)(), (ctypes.c_int64 * n)()
            for j, (arr, dst) in enumerate(chunk):
                nb = arr.nbytes
                row[off:off + nb] = arr.reshape(-1).view(np.uint8)
                dsts[j], nbytes[j], offs[j] = dst, nb, off
                off += (nb + 15) // 16 * 16
            rb = self._stage.shape[1]
            if leaves and i == last:
                m = len(leaves)
                ids, sums, mins = zip(*leaves)
                row[off:off + 8 * m].view(np.int64)[:] = ids
                row[off + 8 * m:off + 16 * m].view(np.float64)[:] = sums
                row[off + 16 * m:off + 24 * m].view(np.float64)[:] = mins
                L.push_row_leaves(self._stage.data_ptr() + slot * rb, self._stage_dev.data_ptr() + slot * rb, off + 24 * m, slot,
                                  dsts, nbytes, offs, n, self._it_sum.data_ptr(), self._it_min.data_ptr(), self._capacity, off, m,
                                  self._stage_next, None, _lib.stream_ptr())
                continue
            L.push_row(self._stage.data_ptr() + slot * rb, self._stage_dev.data_ptr() + slot * rb, off, slot, dsts, nbytes, offs, n,
                       None, None, 0, 0, 0, self._stage_next, None, _lib.stream_ptr())

    # ---- sampling ----------------------------------------------------------------------------------------------------
    def sample_indices_uniform(self, batch_size, out=None):
        if out is None:
            out = torch.empty(batch_size, dtype=torch.int64, device=self.device)
        return _rng.source().indices(out, len(self), self._n_filled_dev)

    def _resolve_out(self, B):
        dev = self.device
        return dict(start=torch.empty(B, dtype=torch.int64, device=dev), last=torch.empty(B, dtype=torch.int64, device=dev),
                    R=torch.empty((B, 1), dtype=torch.float32, device=dev), frame_s=torch.empty(B, dtype=torch.int64, device=dev),
                    frame_s1=torch.empty(B, dtype=torch.int64, device=dev))

    def _resolve(self, j):
        """Positions j [B] in the FIFO of valid starts -> dict(start, last, R [B,1], frame_s, frame_s1)."""
        B = j.shape[0]
        out = self._resolve_out(B)
        _lib.lib().nstep_resolve(j.data_ptr(), B, self.valid_ring.data_ptr(), self.scalars.data_ptr(), self._maxsize, self.n_step,
                                 None if self._reward_f32 else self.reward.data_ptr(),
                                 self.reward.data_ptr() if self._reward_f32 else None, self.gamma_pows.data_ptr(),
                                 self.first_frame.data_ptr(), out["start"].data_ptr(), out["last"].data_ptr(), out["R"].data_ptr(),
                                 out["frame_s"].data_ptr(), out["frame_s1"].data_ptr(), _lib.stream_ptr())
        return out

    def _require_prioritized(self, what):
        if not self.prioritized:
            raise NotImplementedError(f"{what} needs NStepReplayBuffer(..., prioritized=True): this buffer samples uniformly")

    def sample_per(self, batch_size):
        """Proportional draw (float64 u from the draw source, replay.py:163-177) + resolve in one launch
        (ssac_nstep_tree_sample) -> (dict of _resolve plus ``slot`` = leaf ids, ``j`` = FIFO positions; weights float64 [B])."""
        self._require_prioritized("prioritised sampling")
        B, dev = batch_size, self.device
        n = len(self)
        if n < (2 if self._v_tail == 0 else 1):
            raise ValueError(f"NStepReplayBuffer: {n} transitions are too few to sample from")
        u = torch.empty(B, dtype=torch.float64, device=dev)
        _rng.source().uniform01(u)
        out = self._resolve_out(B)
        out["slot"] = torch.empty(B, dtype=torch.int64, device=dev)
        out["j"] = torch.empty(B, dtype=torch.int64, device=dev)
        w = torch.empty(B, dtype=torch.float64, device=dev)
        _lib.lib().nstep_tree_sample(self._it_sum.data_ptr(), self._it_min.data_ptr(), self._capacity, self._maxsize,
                                     self.scalars.data_ptr(), u.data_ptr(), B, float(self.beta), out["slot"].data_ptr(),
                                     out["j"].data_ptr(), w.data_ptr(), self.valid_ring.data_ptr(), self.n_step,
                                     None if self._reward_f32 else self.reward.data_ptr(),
                                     self.reward.data_ptr() if self._reward_f32 else None, self.gamma_pows.data_ptr(),
                                     self.first_frame.data_ptr(), out["start"].data_ptr(), out["last"].data_ptr(),
                                     out["R"].data_ptr(), out["frame_s"].data_ptr(), out["frame_s1"].data_ptr(), _lib.stream_ptr())
        return out, w

    def _gather_obs(self, key, frame_idx, shift, aug, B, aug_rows, use_aug):
        """fp32 observation batch of key ``key`` whose stacks start at frame counters ``frame_idx``."""
        ring, k, fcap = self.frames[key], self.frame_stack, self._frame_cap
        if ring.dtype == torch.uint8 and ring.dim() == 4:
            cf, H, W = ring.shape[1:]
            C = cf * (k if self._stacked[key] else 1)
            out = torch.empty((B, C, H, W), dtype=torch.float32, device=self.device)
            pad_mode = getattr(aug, "pad_mode", augmentations.PAD_NONE) if use_aug else augmentations.PAD_NONE
            if pad_mode == augmentations.PAD_RAD:
                raise NotImplementedError("RAD crop over the frame-deduplicated ring")
            noise = None
            if use_aug and getattr(aug, "noise", False):
                noise = torch.empty_like(out)
                _rng.source().normal(noise)
            fi = frame_idx if self._stacked[key] or k == 1 else frame_idx + (k - 1)   # non-stacked key: the newest copy
            _lib.lib().gather_aug_u8_ring(ring.data_ptr(), out.data_ptr(), fi.data_ptr(), cf, fcap,
                                          None if shift is None or pad_mode == augmentations.PAD_NONE else shift.data_ptr(),
                                          None if noise is None else noise.data_ptr(), B, C, H, W, int(getattr(aug, "pad", 0)),
                                          int(pad_mode), int(aug_rows if use_aug else 0), _lib.stream_ptr())
            return out
        n = ring[0].numel()
        out = torch.empty((B,) + tuple(ring.shape[1:]), dtype=torch.float32, device=self.device)
        fi = (frame_idx + (k - 1)) % fcap
        _ops.gather_rows([ring], [out], [n], [n], [0 if ring.dtype == torch.float32 else 1], fi, B)
        return out

    def nstep_sample_move_and_augment(self, batch_size, augmenter, aug_mix, _idx=None, per=False):
        """What learning_utils.sample_move_and_augment returns, for this buffer (fusable augmentations only).  per=True:
        prioritised draw, ``imp_weights`` float64 [B] and ``priority_idxs`` = leaf ids (what update_priorities takes)."""
        from . import learning_utils as lu

        if per:
            self._require_prioritized("sample_move_and_augment(per=True)")
        assert len(self) >= batch_size
        B, dev = batch_size, self.device
        if not torch.cuda.is_current_stream_capturing():
            self.total_sample_calls += 1
        if not (isinstance(augmenter, augmentations.AugmentationSequence) and augmenter.fusable()):
            raise NotImplementedError("NStepReplayBuffer needs a fusable AugmentationSequence (Identity / DrQ / DrQv2)")
        rows = lu._batch_rows(B, augmenter, per) if parallel.batches_sharded() else None
        aug_rows = int(B * aug_mix)
        if per:
            res, imp_weights = self.sample_per(B)
        else:
            idx = _idx if _idx is not None else self.sample_indices_uniform(B)
            if rows is not None:   # indices drawn for the global batch: this rank gathers its rows of it
                idx, aug_rows, B = idx[rows[0]:rows[1]], parallel.local_aug_rows(B, aug_mix, *rows), rows[1] - rows[0]
            res = self._resolve(idx)
        aug = augmenter.aug_list[0]
        aug.change_randomization_params(dev)   # once per call; o and o1 share the shifts
        shift = getattr(aug, "shift", None)
        if rows is not None and shift is not None:   # drawn for the global batch (aug.batch_size rows)
            shift = shift[rows[0]:rows[1]]
        aug_keys = self.keys if augmenter.keys is None else augmenter.keys
        rd = lu.ReplayDict()
        A = self.action.shape[1]
        o, o1 = {}, {}
        packed = None
        flat = len(self.keys) == 1 and self.frames[self.keys[0]].dtype == torch.float32 and self.frames[self.keys[0]].dim() == 2
        fs, fs1 = (res["frame_s"] + (self.frame_stack - 1)) % self._frame_cap, (res["frame_s1"] + (self.frame_stack - 1)) % self._frame_cap
        if flat:
            # state observations: straight into the [B, S+A] first-layer inputs, as the classic buffer does
            key = self.keys[0]
            ring = self.frames[key]
            S = ring.shape[1]
            XA = torch.empty((B, S + A), dtype=torch.float32, device=dev)
            X1 = torch.empty((B, S + A), dtype=torch.float32, device=dev)
            XPI = torch.empty((B, S + A), dtype=torch.float32, device=dev)
            o[key], o1[key], a = XA[:, :S], X1[:, :S], XA[:, S:]
            _ops.gather_rows([ring, ring], [XA, XPI], [S, S], [S + A, S + A], [0, 0], fs, B)
            _ops.gather_rows([ring], [X1], [S], [S + A], [0], fs1, B)
            _ops.gather_rows([self.action], [a], [A], [S + A], [0], res["start"], B)
            packed = dict(XA=XA, X1=X1, XPI=XPI, S=S, A=A, key=key)
        else:
            for key in self.keys:
                use = key in aug_keys
                if use and getattr(aug, "pad_mode", augmentations.PAD_NONE) != augmentations.PAD_NONE and self.frames[key].dim() != 4:
                    raise NotImplementedError(f"shift augmentation of non-image key '{key}'")
                o[key] = self._gather_obs(key, res["frame_s"], shift, aug, B, aug_rows, use)
                o1[key] = self._gather_obs(key, res["frame_s1"], shift, aug, B, aug_rows, use)
            a = torch.empty((B, A), dtype=torch.float32, device=dev)
            _ops.gather_rows([self.action], [a], [A], [A], [0], res["start"], B)
        d = torch.empty((B, 1), dtype=torch.float32, device=dev)
        _ops.gather_rows([self.done], [d], [1], [1], [1], res["last"], B)
        rd["primary_batch"] = (o, a, res["R"], o1, d)
        if packed is not None:
            rd["_packed"] = packed
        rd["priority_idxs"] = res["slot"] if per else res["start"]
        rd["imp_weights"] = imp_weights if per else lu._ones1(dev)
        return rd

    # ---- reference API ---------------------------------------------------------------------------------------------
    def sample_uniform(self, batch_size):
        """((s, a, r, s1, d), idxs) in the storage dtypes, like replay.py:179-181 (idxs = start slots)."""
        graphed.join()
        self.total_sample_calls += 1
        return self._tuples(self.sample_indices_uniform(batch_size))

    def _tuples(self, j):
        res = self._resolve(j)
        return self._batch_of(res, j.shape[0]), res["start"].cpu().numpy()

    def _batch_of(self, res, B):
        s, s1 = {}, {}
        ident = augmentations.IdentityAug(B)
        for key in self.keys:
            ring = self.frames[key]
            a_, b_ = (self._gather_obs(key, res[f], None, ident, B, 0, False) for f in ("frame_s", "frame_s1"))
            s[key], s1[key] = (a_.to(ring.dtype), b_.to(ring.dtype)) if ring.dtype == torch.uint8 else (a_, b_)
        return s, self.action[res["start"]], res["R"], s1, self.done[res["last"]]

    def get_all_transitions(self):
        """Every n-step transition currently in the buffer, oldest first."""
        graphed.join()
        return self._tuples(torch.arange(len(self), dtype=torch.int64, device=self.device))[0]

    def sample(self, batch_size):
        """((s, a, R, s1, d), weights float64 [B], idxs) like ReplayBuffer.sample (idxs = leaf ids)."""
        self._require_prioritized("NStepReplayBuffer.sample")
        graphed.join()
        self.total_sample_calls += 1
        res, w = self.sample_per(batch_size)
        return self._batch_of(res, batch_size), w, res["slot"].cpu().numpy()

    def _tree_set_live(self, idx_dev, val_dev):
        L = _lib.lib()
        for i in range(0, idx_dev.numel(), 1024):   # in order: the last write of a leaf still wins
            ii, vv = idx_dev[i:i + 1024], val_dev[i:i + 1024]
            L.tree_set_live(self._it_sum.data_ptr(), self._it_min.data_ptr(), self._capacity, self._maxsize,
                            self.scalars.data_ptr(), ii.data_ptr(), vv.data_ptr(), ii.numel(), _lib.stream_ptr())

    def update_priorities(self, idxes, priorities):
        """idxes (leaf ids from sample / priority_idxs) / priorities: numpy arrays or device tensors, like
        ReplayBuffer.update_priorities.  Ids whose transition has been evicted since it was drawn (and whose slot no newer
        transition has taken) are dropped on the device."""
        self._require_prioritized("NStepReplayBuffer.update_priorities")
        assert len(idxes) == len(priorities)
        if not torch.cuda.is_current_stream_capturing():
            graphed.join()
        if torch.is_tensor(priorities):
            idx_dev = idxes if torch.is_tensor(idxes) else torch.from_numpy(np.asarray(idxes, dtype=np.int64)).to(self.device)
            pr = priorities.to(torch.float64)
            self._tree_set_live(idx_dev.to(torch.int64).contiguous(), (pr**self.alpha).contiguous())
            self._note_priorities_dev(pr)
            return
        idxes, priorities = np.asarray(idxes), np.asarray(priorities, dtype=np.float64)
        assert np.min(priorities) > 0
        assert np.min(idxes) >= 0
        assert np.max(idxes) < self._maxsize
        self._tree_set_live(torch.from_numpy(idxes.astype(np.int64)).to(self.device),
                            torch.from_numpy(priorities**self.alpha).to(self.device))
        self._max_priority = max(self._max_priority, float(np.max(priorities)))

    def bytes_per_transition(self):
        """Device bytes per stored step (frames once + bookkeeping) -- the reference layout stores 2k frames."""
        per = sum(r[0].numel() * r.element_size() for r in self.frames.values()) * self._frame_cap / self._maxsize
        return per + self.action.shape[1] * 4 + self.reward.element_size() + 1 + 16

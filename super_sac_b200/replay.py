"""Device-resident replay buffer with the reference's API (reference replay.py:10-190, :207-353).

``ReplayBuffer(size, alpha, beta)``: ``push / load_experience / sample / sample_uniform / update_priorities /
get_all_transitions / len() / total_sample_calls`` behave like the reference's, but the ring storage lives in HBM
in its native dtype (uint8 pixels stay uint8: 63.5 KB per 9x84x84 frame), transitions cross PCIe once at ``push``
time instead of once per sampled batch, and sampling is an index kernel + a coalesced gather (ssac_rng_fill,
ssac_gather_rows, ssac_gather_aug_u8).  The prioritised path keeps the reference's float64 sum / min segment
trees (same layout: root at 1, leaves at capacity + i) on the device (ssac_tree_set / ssac_tree_sample).

Memory: like the reference, ``s`` and ``s1`` are stored separately, so a pixel buffer costs 2 x 63.5 KB per
transition -- size the capacity for the 180 GB of a B200 (1.4 M pixel transitions at most; 100 k = 12.7 GB).
"""
import numpy as np
import torch

from . import _lib, _ops, _rng, graphed


def _default_device():
    from . import device

    return device


class ReplayBufferStorage:
    """Ring storage (reference replay.py:10-95), tensors on the device."""

    def __init__(self, size, state_example, act_example, device):
        self.size = size
        self.device = device
        self.action_stack = torch.zeros((size,) + tuple(act_example.shape), dtype=torch.float32, device=device)
        self.reward_stack = torch.zeros((size, 1), dtype=torch.float32, device=device)
        self.done_stack = torch.zeros((size, 1), dtype=torch.uint8, device=device)
        self.s_stack, self.s1_stack, self.s_dtypes = {}, {}, {}
        for label, array in state_example.items():
            array = np.asarray(array)
            tdtype = torch.from_numpy(np.zeros(1, dtype=array.dtype)).dtype
            self.s_dtypes[label] = array.dtype
            self.s_stack[label] = torch.zeros((size,) + array.shape, dtype=tdtype, device=device)
            self.s1_stack[label] = torch.zeros((size,) + array.shape, dtype=tdtype, device=device)
        self._next_idx = 0
        self._max_filled = 0

    def __len__(self):
        return self._max_filled

    def _put(self, stack, start, n, host):
        """Write n rows at ring positions start.. (with wrap) from a host array: one or two H2D copies."""
        t = torch.from_numpy(np.ascontiguousarray(host)).reshape((n,) + tuple(stack.shape[1:]))
        first = min(n, self.size - start)
        stack[start:start + first].copy_(t[:first], non_blocking=True)
        if first < n:
            stack[: n - first].copy_(t[first:], non_blocking=True)

    def add(self, s, a, r, s1, d):
        a = np.asarray(a)
        if a.ndim > 1:
            n = len(a)
        else:
            n = 1
            r, d = np.array(r), np.array(d)
        if n > self.size:
            raise ValueError("more transitions pushed at once than the buffer holds")
        start = self._next_idx
        for label in s:
            self._put(self.s_stack[label], start, n, np.asarray(s[label]).astype(self.s_dtypes[label]))
        for label in s1:
            self._put(self.s1_stack[label], start, n, np.asarray(s1[label]).astype(self.s_dtypes[label]))
        self._put(self.action_stack, start, n, a.astype(np.float32))
        self._put(self.reward_stack, start, n, np.asarray(r).astype(np.float32))
        self._put(self.done_stack, start, n, np.asarray(d).astype(np.uint8))
        R = np.arange(start, start + n) % self.size
        self._max_filled = min(max(start + n, self._max_filled), self.size)
        self._next_idx = (start + n) % self.size
        return R

    def gather(self, idx):
        """Plain gather in storage dtypes (reference replay.py:66-84): the public, un-fused path."""
        B = idx.numel()
        srcs, dsts, rows, lds, modes = [], [], [], [], []
        state, next_state = {}, {}

        def add(stack, out):
            srcs.append(stack); dsts.append(out)
            nbytes = stack[0].numel() * stack.element_size()
            if stack.dtype == torch.float32:
                rows.append(stack[0].numel()); lds.append(stack[0].numel()); modes.append(0)
            else:
                rows.append(nbytes); lds.append(nbytes); modes.append(2)

        for label in self.s_stack:
            state[label] = torch.empty((B,) + tuple(self.s_stack[label].shape[1:]), dtype=self.s_stack[label].dtype, device=self.device)
            next_state[label] = torch.empty_like(state[label])
            add(self.s_stack[label], state[label])
            add(self.s1_stack[label], next_state[label])
        action = torch.empty((B,) + tuple(self.action_stack.shape[1:]), dtype=torch.float32, device=self.device)
        reward = torch.empty((B, 1), dtype=torch.float32, device=self.device)
        done = torch.empty((B, 1), dtype=torch.uint8, device=self.device)
        add(self.action_stack, action); add(self.reward_stack, reward); add(self.done_stack, done)
        for k0 in range(0, len(srcs), 16):
            _ops.gather_rows(srcs[k0:k0 + 16], dsts[k0:k0 + 16], rows[k0:k0 + 16], lds[k0:k0 + 16], modes[k0:k0 + 16], idx, B)
        if action.dim() < 2:
            action = action.unsqueeze(1)
        return state, action, reward, next_state, done

    def get_all_transitions(self):
        n = self._max_filled
        s = {k: v[:n].cpu().numpy() for k, v in self.s_stack.items()}
        s1 = {k: v[:n].cpu().numpy() for k, v in self.s1_stack.items()}
        return s, self.action_stack[:n].cpu().numpy(), self.reward_stack[:n].cpu().numpy(), s1, self.done_stack[:n].cpu().numpy()


class PriorityMax:
    """Running maximum of the priorities given to ``update_priorities`` (replay.py:190), the priority a new transition
    gets.  Device-tensor updates only record a pending device-side maximum; it is folded into the host value (one sync)
    when the next push reads it."""

    def _init_max_priority(self):
        self._max_priority_host = 1.0
        self._max_priority_dev = None  # pending device-side maximum (folded in lazily: no sync per update)

    @property
    def _max_priority(self):
        if self._max_priority_dev is not None:
            self._max_priority_host = max(self._max_priority_host, float(self._max_priority_dev))
            self._max_priority_dev = None
        return self._max_priority_host

    @_max_priority.setter
    def _max_priority(self, v):
        self._max_priority_host, self._max_priority_dev = float(v), None

    def _note_priorities_dev(self, pr):
        """pr: float64 device tensor of new priorities."""
        m = pr.max()
        self._max_priority_dev = m if self._max_priority_dev is None else torch.maximum(self._max_priority_dev, m)


class ReplayBuffer(PriorityMax):
    """Uniform + prioritised replay (reference replay.py:98-190)."""

    def __init__(self, size, alpha=0.6, beta=1.0, device=None):
        assert alpha >= 0
        self._maxsize = size
        self._storage = None
        self.alpha, self.beta = alpha, beta
        self.device = torch.device(device) if device is not None else None
        cap = 1
        while cap < size:
            cap *= 2
        self._capacity = cap
        self._it_sum = self._it_min = None  # float64 [2*cap] device trees, created with the storage
        self._init_max_priority()
        self.total_sample_calls = 0

    def __len__(self):
        return len(self._storage) if self._storage is not None else 0

    def _ensure_storage(self, state, action):
        if self._storage is not None:
            return
        if self.device is None:
            self.device = torch.device(_default_device())
        if self.device.type != "cuda":
            raise _lib.SsacError("the replay buffer is device-resident: a CUDA (sm_100) device is required")
        _lib.require_device(self.device.index if self.device.index is not None else torch.cuda.current_device())
        action = np.asarray(action)
        if action.ndim > 1:
            act_example, state_example = action[0], {k: np.asarray(v)[0] for k, v in state.items()}
        else:
            act_example, state_example = action, {k: np.asarray(v) for k, v in state.items()}
        self._storage = ReplayBufferStorage(self._maxsize, state_example, act_example, self.device)
        self._it_sum = torch.zeros(2 * self._capacity, dtype=torch.float64, device=self.device)
        self._it_min = torch.full((2 * self._capacity,), float("inf"), dtype=torch.float64, device=self.device)
        self._n_filled_dev = torch.zeros(1, dtype=torch.int64, device=self.device)  # read by captured graphs

    def _tree_set(self, idx_dev, val_dev):
        _lib.lib().tree_set(self._it_sum.data_ptr(), self._it_min.data_ptr(), self._capacity, idx_dev.data_ptr(),
                            val_dev.data_ptr(), idx_dev.numel(), _lib.stream_ptr())

    # --- single-transition fast path: one pinned staging buffer, one H2D copy, one scatter kernel ----------------
    _STAGE_SLOTS = 64

    def _push_one(self, state, action, reward, next_state, done, priority, wait_event=None):
        import ctypes

        st = self._storage
        if not hasattr(self, "_stage"):
            # layout of one staging row: [s, s1 per obs key] action reward done fill | tree idx, priority (not scattered)
            lay, dst_base, dst_stride, kinds, off = [], [], [], [], 0

            def add(nb, tensor, kind):
                nonlocal off
                lay.append((off, nb))
                dst_base.append(tensor.data_ptr() if tensor is not None else 0)
                dst_stride.append(tensor.stride(0) * tensor.element_size() if tensor is not None and kind != "fixed" else 0)
                kinds.append(kind)
                off = (off + nb + 15) // 16 * 16

            for label in st.s_stack:
                for stack in (st.s_stack[label], st.s1_stack[label]):
                    add(stack[0].numel() * stack.element_size(), stack, "ring")
            add(st.action_stack[0].numel() * 4, st.action_stack, "ring")
            add(4, st.reward_stack, "ring")
            add(1, st.done_stack, "ring")
            add(8, self._n_filled_dev, "fixed")
            self._n_scatter = len(lay)
            add(8, None, "tree")
            add(8, None, "tree")
            self._stage_layout, self._stage_bytes = lay, off
            self._stage = torch.empty((self._STAGE_SLOTS, off), dtype=torch.uint8).pin_memory()
            self._stage_dev = torch.empty((self._STAGE_SLOTS, off), dtype=torch.uint8, device=self.device)
            self._stage_next = 0
            self._dst_base, self._dst_stride = dst_base, dst_stride
            n = self._n_scatter
            self._c_dsts = (ctypes.c_void_p * n)()
            self._c_nbytes = (ctypes.c_int64 * n)(*[nb for _, nb in lay[:n]])
            self._c_offs = (ctypes.c_int64 * n)(*[o for o, _ in lay[:n]])
            # typed numpy views of every field of every pinned row: one assignment per field and push
            host = self._stage.numpy()
            views = []
            for slot in range(self._STAGE_SLOTS):
                row, k, v = host[slot], 0, []
                for label in st.s_stack:
                    for _ in range(2):
                        o, nb = lay[k]; k += 1
                        v.append(row[o:o + nb].view(st.s_dtypes[label]).reshape(st.s_stack[label].shape[1:]))
                for dt in (np.float32, np.float32, np.uint8, np.int64, np.int64, np.float64):
                    o, nb = lay[k]; k += 1
                    v.append(row[o:o + nb].view(dt))
                views.append(v)
            self._stage_views = views
            self._stage_host_ptr = self._stage.data_ptr()
            self._stage_dev_ptr = self._stage_dev.data_ptr()
        L = _lib.lib()
        slot = self._stage_next
        self._stage_next = (slot + 1) % self._STAGE_SLOTS
        # (the H2D copy that last used this pinned row has finished: the previous push waited for it on its way out)
        v = self._stage_views[slot]
        pos = st._next_idx
        k = 0
        for label in st.s_stack:
            v[k][...] = state[label]; v[k + 1][...] = next_state[label]
            k += 2
        v[k][...] = action
        v[k + 1][0] = reward
        v[k + 2][0] = bool(done)
        filled = min(max(pos + 1, st._max_filled), st.size)
        v[k + 3][0] = filled
        v[k + 4][0] = pos
        v[k + 5][0] = priority
        dsts, base, stride = self._c_dsts, self._dst_base, self._dst_stride
        for i in range(self._n_scatter):
            dsts[i] = base[i] + pos * stride[i]
        lay = self._stage_layout
        nb = self._stage_bytes
        L.push_row(self._stage_host_ptr + slot * nb, self._stage_dev_ptr + slot * nb, nb, slot, dsts, self._c_nbytes,
                   self._c_offs, self._n_scatter, self._it_sum.data_ptr(), self._it_min.data_ptr(), self._capacity,
                   lay[-2][0], lay[-1][0], self._stage_next, wait_event, _lib.stream_ptr())
        st._max_filled = filled
        st._next_idx = (pos + 1) % st.size
        return np.array([pos])

    def push(self, state, action, reward, next_state, done, priorities=None, **kwargs):
        self._ensure_storage(state, action)
        if np.asarray(action).ndim == 1 and (priorities is None or np.ndim(priorities) == 0):
            p = self._max_priority if priorities is None else float(priorities)
            # (cross-call pipelined updates: the latest gather may still read the slot this overwrites -- the push's own
            # launch waits for it, one C call instead of two)
            return self._push_one(state, action, reward, next_state, done, p**self.alpha, graphed.push_wait_event())
        graphed.before_push()
        R = self._storage.add(state, action, reward, next_state, done)
        self._n_filled_dev.fill_(len(self._storage))
        if priorities is None:
            priorities = self._max_priority
        vals = np.broadcast_to(np.asarray(priorities, dtype=np.float64) ** self.alpha, R.shape)
        self._tree_set(torch.from_numpy(R.astype(np.int64)).to(self.device),
                       torch.from_numpy(np.array(vals, dtype=np.float64, copy=True)).to(self.device))
        return R

    def load_experience(self, s, a, r, s1, d):
        assert len(a) <= self._maxsize, "Experience dataset is larger than the buffer."
        r, d = np.asarray(r), np.asarray(d)
        if r.ndim < 2:
            r = np.expand_dims(r, 1)
        if d.ndim < 2:
            d = np.expand_dims(d, 1)
        self.push(s, a, r, s1, d)

    def get_all_transitions(self):
        return self._storage.get_all_transitions()

    # --- device-side sampling used by learning_utils.sample_move_and_augment ------------------------
    def sample_indices_uniform(self, batch_size, out=None):
        if out is None:
            out = torch.empty(batch_size, dtype=torch.int64, device=self.device)
        return _rng.source().indices(out, len(self._storage), self._n_filled_dev)

    def sample_indices_per(self, batch_size):
        """Proportional sampling + importance weights on the device (reference replay.py:163-177)."""
        u = torch.empty(batch_size, dtype=torch.float64, device=self.device)
        _rng.source().uniform01(u)
        idx = torch.empty(batch_size, dtype=torch.int64, device=self.device)
        w = torch.empty(batch_size, dtype=torch.float64, device=self.device)
        _lib.lib().tree_sample(self._it_sum.data_ptr(), self._it_min.data_ptr(), self._capacity, len(self._storage),
                               u.data_ptr(), batch_size, float(self.beta), idx.data_ptr(), w.data_ptr(), _lib.stream_ptr())
        return idx, w

    # --- reference API ---------------------------------------------------------------------------------
    def sample(self, batch_size):
        graphed.join()
        self.total_sample_calls += 1
        idx, w = self.sample_indices_per(batch_size)
        return self._storage.gather(idx), w, idx.cpu().numpy()

    def sample_uniform(self, batch_size):
        graphed.join()
        self.total_sample_calls += 1
        idx = self.sample_indices_uniform(batch_size)
        return self._storage.gather(idx), idx.cpu().numpy()

    def update_priorities(self, idxes, priorities):
        """idxes / priorities: numpy arrays (reference signature) or device tensors (no host round trip)."""
        assert len(idxes) == len(priorities)
        if not torch.cuda.is_current_stream_capturing():
            graphed.join()
        if torch.is_tensor(priorities):
            idx_dev = idxes if torch.is_tensor(idxes) else torch.from_numpy(np.asarray(idxes, dtype=np.int64)).to(self.device)
            pr = priorities.to(torch.float64)
            self._tree_set(idx_dev, pr**self.alpha)
            self._note_priorities_dev(pr)
            return
        idxes, priorities = np.asarray(idxes), np.asarray(priorities, dtype=np.float64)
        assert np.min(priorities) > 0
        assert np.min(idxes) >= 0
        assert np.max(idxes) < len(self._storage)
        self._tree_set(torch.from_numpy(idxes.astype(np.int64)).to(self.device),
                       torch.from_numpy(priorities**self.alpha).to(self.device))
        self._max_priority = max(self._max_priority, float(np.max(priorities)))


from .nstep_replay import NStepReplayBuffer  # noqa: E402,F401  (on-the-fly n-step + frame-deduplicated layout)

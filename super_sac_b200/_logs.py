"""Logged scalars without a host sync per value.

The reference calls ``.item()`` ~70 times per REDQ update (learning_utils.py:351-353, :394-397, :95-106,
learning.py:132-137).  Here kernels write their scalars into slots of one small device buffer; ``finalize()`` does
ONE device->host copy and fills the dict with plain floats under the reference's key names.
"""
import contextlib

import torch

_defer_depth = 0
_embed_readback = False   # capture the D2H copy of the logged scalars as the last node of the graph (auto-graph path)


@contextlib.contextmanager
def deferred(embed_readback=False):
    """Inside this context ``finalize()`` does not synchronise (used while a CUDA graph is being captured);
    call ``fetch()`` on the returned logs after the work has run.  embed_readback: the device->host copy of the logged
    scalars becomes the last node of the captured graph (for callers that read the logs after every replay)."""
    global _defer_depth, _embed_readback
    _defer_depth += 1
    prev, _embed_readback = _embed_readback, embed_readback
    try:
        yield
    finally:
        _defer_depth -= 1
        _embed_readback = prev


# Pinned host buffers for the read-back.  They are allocated outside stream capture (a captured update takes one from
# the pool and owns it for the life of its graph: the D2H copy becomes a node of the graph).
_pin_pool = []
_pin_shared = {}
_PIN_RESERVE = 8


def _capturing():
    return torch.cuda.is_available() and torch.cuda.is_current_stream_capturing()


def _reserve_pinned(capacity):
    if not _capturing():
        while len(_pin_pool) < _PIN_RESERVE:
            _pin_pool.append(torch.empty(capacity, dtype=torch.float32).pin_memory())


class _Multi:
    __slots__ = ("fn",)

    def __init__(self, fn):
        self.fn = fn


class DeviceLogs(dict):
    def __init__(self, device, capacity=256, zeroed=True):
        """zeroed=False: the caller clears ``take_unzeroed()`` inside its first kernel (saves the memset launch)."""
        super().__init__()
        self._buf = (torch.zeros if zeroed else torch.empty)(capacity, dtype=torch.float32, device=device)
        self._needs_zero = not zeroed
        self._host = None   # pinned buffer written by a D2H node of the captured graph (set in finalize under capture)
        self._n = 0
        self._pending = []  # (key, slot, transform)

    def take_unzeroed(self):
        """The buffer if it still has to be cleared (once), else None."""
        if self._needs_zero:
            self._needs_zero = False
            return self._buf
        return None

    def slots(self, n):
        """Reserve n consecutive float slots; returns (tensor view, first slot index)."""
        if self._n + n > self._buf.numel():
            raise RuntimeError("DeviceLogs: out of slots")
        v = self._buf[self._n:self._n + n]
        first = self._n
        self._n += n
        return v, first

    def defer(self, key, slot, transform=None):
        """``slot`` may be a list of slots: their sum is reported."""
        self._pending.append((key, slot, transform))

    def defer_fn(self, key, slots, fn):
        """``fn(*values_of_slots)`` is reported (statistics a kernel leaves as partial sums)."""
        self._pending.append((key, tuple(slots), _Multi(fn)))

    def put_tensor(self, key, scalar_tensor, transform=None):
        """Copy a 0-d / 1-element device tensor into a slot (no sync) and register it under ``key``; returns the slot."""
        v, s = self.slots(1)
        v.copy_(scalar_tensor.reshape(1))
        self.defer(key, s, transform)
        return v

    def finalize(self):
        if _defer_depth > 0:
            if _embed_readback and self._pending and self._host is None and _capturing() and _pin_pool \
                    and _pin_pool[-1].numel() >= self._buf.numel():
                self._host = _pin_pool.pop()
                self._host[: self._n].copy_(self._buf[: self._n], non_blocking=True)   # captured: replays with the graph
            return self
        return self.fetch()

    def fetch(self, keep=False, synced=False):
        """Resolve pending entries with one device->host copy.  keep=True leaves them registered so the same
        buffer can be read again after the next graph replay.  synced: the caller already waited for the replay whose
        embedded copy filled the pinned buffer (an event recorded behind it)."""
        if self._pending:
            if self._host is not None:
                if not synced:
                    torch.cuda.current_stream(self._buf.device).synchronize()   # the copy is part of the replayed graph
                host = self._host[: self._n].tolist()
            else:
                _reserve_pinned(self._buf.numel())
                pin = _pin_shared.get(self._buf.numel())
                if pin is None:
                    pin = _pin_shared[self._buf.numel()] = torch.empty(self._buf.numel(), dtype=torch.float32).pin_memory()
                pin[: self._n].copy_(self._buf[: self._n], non_blocking=True)
                torch.cuda.current_stream(self._buf.device).synchronize()   # the one sync
                host = pin[: self._n].tolist()
            for key, slot, transform in self._pending:
                if isinstance(transform, _Multi):
                    self[key] = transform.fn(*[host[s_] for s_ in slot])
                    continue
                val = sum(host[s_] for s_ in slot) if isinstance(slot, (list, tuple)) else host[slot]
                self[key] = transform(val) if transform is not None else val
            if not keep:
                self._pending = []
        return self


def as_device_logs(logs, device):
    """Update functions accept a plain dict too (reference signature); values are then synced on finalize into it."""
    if isinstance(logs, DeviceLogs):
        return logs, None
    return DeviceLogs(device), logs


class LazyLogs(dict):
    """The logged scalars of a graph-replayed update whose device->host copy is still in flight.

    ``graphed.enable_auto_graphs(lazy_logs=True)``: ``learning.critic_update`` returns right after ``cudaGraphLaunch``; the
    values (plain floats under the reference's keys) materialise on first access -- one event wait -- or, at the latest,
    when the same update is launched again (its pinned read-back buffer is about to be overwritten).  A training loop that
    only looks at its logs every few hundred steps (main.py:552-572) never stalls on them, and the host prepares the
    next transition (``buffer.push``) while the GPU is still inside the update."""

    def __init__(self, logs, event):
        super().__init__()
        self._src, self._event = logs, event

    def resolve(self):
        if self._src is not None:
            src, self._src = self._src, None
            self._event.synchronize()
            dict.update(self, src.fetch(keep=True, synced=True))
        return self

    def __getitem__(self, k):
        return dict.__getitem__(self.resolve(), k)

    def __iter__(self):
        return dict.__iter__(self.resolve())

    def __len__(self):
        return dict.__len__(self.resolve())

    def __contains__(self, k):
        return dict.__contains__(self.resolve(), k)

    def __repr__(self):
        return dict.__repr__(self.resolve())

    def __eq__(self, other):
        return dict.__eq__(self.resolve(), other)

    __hash__ = None

    def get(self, k, default=None):
        return dict.get(self.resolve(), k, default)

    def keys(self):
        return dict.keys(self.resolve())

    def values(self):
        return dict.values(self.resolve())

    def items(self):
        return dict.items(self.resolve())

    def copy(self):
        return dict(self.resolve())

    def update(self, *a, **k):
        return dict.update(self.resolve(), *a, **k)

    def __setitem__(self, k, v):
        return dict.__setitem__(self.resolve(), k, v)

    def pop(self, *a):
        return dict.pop(self.resolve(), *a)

    def setdefault(self, *a):
        return dict.setdefault(self.resolve(), *a)

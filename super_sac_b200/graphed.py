"""CUDA-graph replay of the update entry points.

One REDQ-10 critic update is ~25 short kernels; launched one by one from Python the step is bound by launch and
interpreter latency, not by the GPU (SURVEY F13).  ``GraphedCall`` runs any of the update functions once under
``torch.cuda.graph`` -- every kernel of libssac_b200 is capturable: no allocation, no sync, and everything that
changes between replays (Adam step, PopArt state, Philox offset, log_alpha, buffer fill level) lives in device
memory -- and afterwards replays the whole step with a single ``cudaGraphLaunch``.

    step = GraphedCall(lambda: learning.critic_update(buffer=..., agent=..., ...))
    step.replay()            # one update, no host sync
    logs = step.logs()       # one device->host copy, reference log keys

Restrictions (checked by the caller): static shapes and hyper-parameters, the default Philox randomness source, and
no host-side decisions inside the captured function (``random.choice`` for the logged member is frozen at capture).
"""
import torch

from . import _lib, _logs


class GraphedCall:
    def __init__(self, fn, warmup=2):
        self.graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):  # allocator / lazy state (Adam moments, rng state) settles before capture
                fn()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        with _logs.deferred():
            with torch.cuda.graph(self.graph):
                self.result = fn()
        self.n_replays = 0

    def replay(self):
        self.graph.replay()
        self.n_replays += 1

    def _logs_obj(self):
        r = self.result
        if isinstance(r, tuple):
            r = r[0]
        return r

    def logs(self):
        """Logged scalars of the most recent replay (one D2H copy + sync)."""
        return dict(self._logs_obj().fetch(keep=True))


# ------------------------------------------------------------------------------------------------
# transparent graph replay behind the drop-in entry points
# ------------------------------------------------------------------------------------------------
_auto = {"on": False, "cache": {}, "min_calls": 2, "lazy": False, "pipeline": False, "cross": None}


def enable_auto_graphs(on=True, lazy_logs=False, pipeline=False):
    """After ``enable_auto_graphs()``, ``learning.critic_update`` / ``online_actor_update`` (continuous or discrete) replay a
    captured CUDA graph from the third call with identical arguments on (same objects, same hyper-parameters): the call
    a user makes stays ``learning.critic_update(...)``, the ~20 launches and their Python marshalling collapse into one
    ``cudaGraphLaunch`` + one device->host copy of the logged scalars.  ``lazy_logs``: the returned dict materialises its
    values on first access instead of synchronising inside the call (``_logs.LazyLogs``).  ``pipeline`` (implies
    ``lazy_logs``): consecutive ``critic_update`` calls overlap on the device, see ``_Cross``."""
    join()
    _auto["on"] = bool(on)
    _auto["pipeline"] = bool(pipeline) and bool(on)
    _auto["lazy"] = (bool(lazy_logs) or bool(pipeline)) and bool(on)
    if not on:
        _auto["cache"].clear()
        _auto["cross"] = None


class _Cross:
    """Cross-call software pipelining of graph-replayed critic updates (``enable_auto_graphs(pipeline=True)``).

    The two alternating captures of the update (see ``run_cached``) are launched on two private streams, so update k+1
    does not queue behind update k as a whole; what orders them is what the data flow requires, expressed as external
    event nodes inside the graphs: the target side of k+1 (draws, gather, target actor, target critics) only follows the
    target side of k (one Philox stream, one replay ring), the online forward of k+1 follows the Adam step of k, the
    weight-gradient kernels of k+1 follow everything of k that still reads the gradients, a Polyak step (issued between
    the calls, behind update k) precedes the target critics and the Adam step of k+1.  The caller's own stream -- where
    ``buffer.push`` runs -- stays free: each launch waits for it, it waits for nothing except the gather that could still
    be reading the ring slot a push overwrites.  Same kernels, same draw order: bit-identical to the serial schedule
    (tests/test_cuda_update_parity.py).  Every other entry point of the package joins the two streams first (``join``);
    code that touches parameters or batches with its OWN kernels must call ``graphed.join()`` itself."""

    def __init__(self, device, owner_key):
        self.device, self.owner = device, owner_key
        self.streams = [torch.cuda.Stream(device=device) for _ in range(2)]
        ev = lambda: torch.cuda.Event(external=True)   # noqa: E731
        self.gather_done, self.adam_done, self.tail_done = [ev(), ev()], [ev(), ev()], [ev(), ev()]
        self.polyak_done = ev()
        self.caller_ready = torch.cuda.Event()
        self.last = None         # slot of the most recent launch
        self.capturing = None    # slot being captured
        cur = torch.cuda.current_stream(device)
        for e in self.gather_done + self.adam_done + self.tail_done + [self.polyak_done]:
            e.record(cur)        # created now: a wait on a never-recorded event would be dropped from the capture
        self.caller_ready.record(cur)
        # raw handles: the per-update host path goes through single C calls (csrc/ssac_host.cu)
        self.stream_ptrs = [st.cuda_stream for st in self.streams]
        self.gather_ptrs = [e.cuda_event for e in self.gather_done]
        self.polyak_ptr = self.polyak_done.cuda_event
        self.caller_ready_ptr = self.caller_ready.cuda_event


def cross_capturing():
    """(state, slot) while a cross-call pipelined capture is under way, else None."""
    X = _auto["cross"]
    return (X, X.capturing) if X is not None and X.capturing is not None else None


def cross_active():
    """The cross-call pipeline state once a pipelined update has been launched (and outside a capture), else None."""
    X = _auto["cross"]
    return X if X is not None and X.last is not None and X.capturing is None else None


def join():
    """Make the caller's current stream wait for every pipelined update in flight."""
    X = _auto["cross"]
    if X is not None and X.last is not None and X.capturing is None:
        cur = torch.cuda.current_stream(X.device)
        for st in X.streams:
            cur.wait_stream(st)


def before_push():
    """A push overwrites one ring slot: the most recent gather may still be reading it."""
    X = _auto["cross"]
    if X is not None and X.last is not None and X.capturing is None:
        _lib.lib().stream_wait_event(_lib.stream_ptr(), X.gather_ptrs[X.last])


def push_wait_event():
    """The same as ``before_push`` for callers that can hand the event to their own launch (ssac_push_row): the raw handle
    of the event the caller's stream has to wait for, or None."""
    X = _auto["cross"]
    if X is not None and X.last is not None and X.capturing is None:
        return X.gather_ptrs[X.last]
    return None


def auto_graphs_enabled():
    return _auto["on"]


class _Slot:
    __slots__ = ("graph", "result", "pending", "event", "exec_ptr", "event_ptr")

    def __init__(self):
        self.graph, self.result, self.pending, self.event = None, None, None, None
        self.exec_ptr, self.event_ptr = None, None


class _Entry:
    __slots__ = ("calls", "slots", "turn", "on_replay", "refs")

    def __init__(self):
        self.calls, self.on_replay, self.refs = 0, None, None
        self.slots, self.turn = [_Slot()], 0


def is_static(obj):
    """True for objects (replay dicts) returned by a captured graph: the same buffers on every call."""
    return getattr(obj, "_ssac_static", False)


def run_cached(key, fn, on_replay=None, refs=None, cross_ok=False):
    """Eager for the first ``min_calls`` calls with this key (allocator and lazy state settle), then capture once
    (capturing does not execute) and replay.  ``on_replay`` updates host-side mirrors (step counters).  ``refs``: the
    objects whose ``id()`` went into ``key`` -- the entry keeps them alive, so that CPython cannot hand one of those ids
    to a new object while the entry exists (a key built from the ids of dead objects could otherwise match by accident).
    The replay dicts a captured call returns are tagged static (``is_static``): they are the graph's own buffers.

    With ``lazy_logs`` the entry holds TWO captures of the same call (own static buffers, own pinned read-back buffer)
    and alternates between them: a replay only has to wait for the logs of the replay before last, so the host runs up to
    two updates ahead of the GPU and the graphs follow each other without a host round trip in between."""
    e = _auto["cache"].get(key)
    if e is None:
        e = _auto["cache"][key] = _Entry()
        e.refs = refs
    X = None
    if cross_ok and _auto["pipeline"]:
        X = _auto["cross"]
        if X is None:
            X = _auto["cross"] = _Cross(torch.device("cuda", torch.cuda.current_device()), key)
        if X.owner != key:   # one pipelined update stream per process: anything else runs behind it
            X = None
    if X is None:
        join()
    if e.calls < _auto["min_calls"]:
        e.calls += 1
        join()
        return fn()
    if _auto["lazy"] and len(e.slots) == 1:
        e.slots.append(_Slot())
    idx = e.turn % len(e.slots)
    sl = e.slots[idx]
    e.turn += 1
    if sl.graph is None:
        join()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with _logs.deferred(embed_readback=True):   # this path fetches the logs after every replay
            if X is not None:
                from . import learning_utils as lu

                with torch.cuda.graph(g, stream=X.streams[idx]):
                    X.capturing = idx
                    try:
                        with lu.pipelined_updates(X.device):
                            sl.result = fn()
                        X.tail_done[idx].record(torch.cuda.current_stream(X.device))
                    finally:
                        X.capturing = None
            else:
                with torch.cuda.graph(g):
                    sl.result = fn()
        sl.graph, e.on_replay = g, on_replay
        sl.exec_ptr = g.raw_cuda_graph_exec() if hasattr(g, "raw_cuda_graph_exec") else None
        sl.event = torch.cuda.Event()
        sl.event.record()   # created
        sl.event_ptr = sl.event.cuda_event
        if isinstance(sl.result, tuple):
            for part in sl.result[1:]:
                for rd in (part if isinstance(part, (list, tuple)) else [part]):
                    try:
                        rd._ssac_static = True
                    except AttributeError:
                        pass
    if sl.pending is not None:    # this capture's previous logs live in the pinned buffer this replay overwrites
        sl.pending.resolve()
        sl.pending = None
    res = sl.result
    logs = res[0] if isinstance(res, tuple) else res
    lazy = _auto["lazy"] and logs._host is not None
    if X is not None:
        # behind everything the caller has issued so far (pushes, actor updates, ...), on this capture's own stream
        if sl.exec_ptr is not None:
            _lib.lib().pipelined_launch(sl.exec_ptr, X.stream_ptrs[idx], _lib.stream_ptr(), X.caller_ready_ptr, sl.event_ptr)
        else:
            st = X.streams[idx]
            X.caller_ready.record(torch.cuda.current_stream(X.device))
            st.wait_event(X.caller_ready)
            with torch.cuda.stream(st):
                sl.graph.replay()
                sl.event.record(st)
        X.last = idx
    elif sl.exec_ptr is not None:
        _lib.lib().graph_launch(sl.exec_ptr, _lib.stream_ptr(), sl.event_ptr if lazy else None)
    else:
        sl.graph.replay()
        if lazy:
            sl.event.record()
    if e.on_replay is not None:
        e.on_replay()
    if lazy:
        out = sl.pending = _logs.LazyLogs(logs, sl.event)
    else:
        out = dict(logs.fetch(keep=True))
    return (out,) + tuple(res[1:]) if isinstance(res, tuple) else out

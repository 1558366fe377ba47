"""Ensemble sharding across the GPUs of one node (SURVEY §8e): one process per GPU, `torch.distributed` plumbing.

One ensemble is partitioned over the ranks in one of two ways, never both at once:

- critics (``enable_critic_sharding``): rank r builds its ``Agent`` with only its ``n_local`` critics (``local_range``) of
  one member; every rank keeps a replica of the actor, the temperature and the batch (identical Philox seed =>
  identical indices, eps and subset on every rank, no broadcast).  REDQ-style critics shard naturally: each critic's
  forward / backward / Adam / Polyak is independent given the TD target, so the updates exchange only small tensors:

    critic update : gather of the target critics' Q(s1, a1)  [N, B]  -> subset-min on every rank (same TD target)
    actor update  : gather of Q(s, pi(s))                     [N, B]  -> arg-min routing;
                    sum of dL/da                              [B, A]  -> replicated actor backward + Adam

- members (``enable_member_sharding``): rank r builds its ``Agent`` with only its block of whole SUNRISE members and
  seeds its own Philox stream.  Members are independent learners (own actor, critics, batch); the single coupling is the
  SUNRISE weight, a statistic over ALL members' target critics on each member's batch: one gather of the local batches
  and one of the local target critics' values on every batch per update (``all_gather_members``).

- batch (``enable_batch_sharding``): ONE learner whose batch rows are split over the ranks (``batch_range``).  Every rank
  keeps full replicas of the agent, the target agent, the optimisers, the temperatures and the replay ring; every draw
  is made for the global batch on every rank (identical Philox state) and each rank keeps its rows, so rank r's batch is
  rows [lo, hi) of the single-GPU batch.  Losses are normalised by the global batch, and the flat gradient arenas
  (critics, native pixel encoder, actor) are summed over the ranks before clipping and Adam (``all_reduce_flat_``: a
  two-shot all-reduce over NVLink, ssac_peer_allreduce) -- every rank then steps identical data and the replicas stay
  bitwise identical.  This is the axis on which a shared, trainable encoder splits: its gradient is a sum over rows.

Any of these sharded updates equals the single-GPU one: the losses are normalised by the global ensemble
(``n_global``, ``members_global``), per-member log keys carry the global member id (``member_id``) and the logged sums
and last-net values are the whole ensemble's (``reduce_logged``).

Payloads are <= 10 KB, so every exchange is pure latency.  On CUDA devices with peer access the exchanges do not go
through NCCL at all: every rank stores its rows straight into all peers' symmetric buffers over NVLink and raises a
signal, the consumer spins on its signals (ssac_peer_put / ssac_peer_wait, csrc/ssac_peer.cu; the buffers' peer mappings
come from torch.distributed._symmetric_memory).  ``torch.distributed`` collectives (all-gather, all-reduce) remain as
the fallback (CPU / gloo tests, boxes without peer access) -- ``exchange_name()`` says which one is live.  Each call
site has an exchange site of its own (a name): a site is used from one stream only, as its two halves alternate
between consecutive exchanges.
"""
import os
import random

import torch
import torch.distributed as dist

# kind: None, "critics", "members" or "batch"; n: the global number of the sharded units (critics of the member, or
# members; None for the batch, whose size each call names)
_state = {"kind": None, "group": None, "world": 1, "rank": 0, "n": None}


# ---- peer-memory exchange sites ---------------------------------------------------------------------------------------
_peer = {"sites": {}, "why_not": None, "disabled": os.environ.get("SSAC_PEER_EXCHANGE", "1") == "0"}


class _PeerSite:
    """One exchange site: a symmetric buffer of two halves (epoch parity), a symmetric signal row and a device epoch."""

    def __init__(self, half_bytes, group, device):
        import torch.distributed._symmetric_memory as symm

        from . import _lib

        self.lib = _lib
        self.group = group if group is not None else dist.group.WORLD
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.half = (int(half_bytes) + 15) // 16 * 16
        name = self.group.group_name
        try:
            symm.enable_symm_mem_for_group(name)
        except Exception:  # noqa: BLE001  (newer torch enables groups lazily)
            pass
        self.buf = symm.empty(2 * self.half, dtype=torch.uint8, device=device)
        self.sig = symm.empty(64, dtype=torch.int32, device=device)
        self.buf.zero_()
        self.sig.zero_()
        self._hb = symm.rendezvous(self.buf, name)
        self._hs = symm.rendezvous(self.sig, name)
        self.buf_ptrs = torch.tensor([int(p) for p in self._hb.buffer_ptrs], dtype=torch.int64, device=device)
        self.sig_ptrs = torch.tensor([int(p) for p in self._hs.buffer_ptrs], dtype=torch.int64, device=device)
        self.epoch = torch.zeros(1, dtype=torch.int32, device=device)
        torch.cuda.synchronize(device)
        dist.barrier(group=group)   # every rank's buffers are zeroed and mapped before the first put

    def put(self, src, dst_off):
        src = src.contiguous()
        self.lib.lib().peer_put(src.data_ptr(), src.numel() * src.element_size(), int(dst_off), self.half, self.buf_ptrs.data_ptr(),
                                self.sig_ptrs.data_ptr(), self.rank, self.world, self.epoch.data_ptr(), self.lib.stream_ptr())

    def wait(self, out, row_index=None, total_bytes=None):
        """Gather the exchanged buffer into ``out`` -- all of it, or (``row_index``: device int32) only those rows."""
        nbytes = out.numel() * out.element_size() if row_index is None else int(total_bytes)
        n_rows = 0 if row_index is None else row_index.numel()
        self.lib.lib().peer_wait(self.buf.data_ptr(), self.half, nbytes, self.sig.data_ptr(), self.world, self.epoch.data_ptr(),
                                 out.data_ptr(), None if row_index is None else row_index.data_ptr(), n_rows,
                                 0 if row_index is None else out[0].numel() * out.element_size(), self.lib.stream_ptr())


def _site(name, nbytes, group, device):
    """The peer-exchange site ``name`` (created on first use, outside any stream capture), or None when peer exchange is
    not available -- the reason is kept for ``exchange_name()``."""
    if _peer["disabled"] or _peer["why_not"] is not None or device.type != "cuda":
        return None
    key = (name, int(nbytes), id(group))
    site = _peer["sites"].get(key)
    if site is None:
        if torch.cuda.is_current_stream_capturing():
            return None
        try:
            site = _peer["sites"][key] = _PeerSite(nbytes, group, device)
        except Exception as e:  # noqa: BLE001
            _peer["why_not"] = f"{type(e).__name__}: {str(e)[:120]}"
            return None
    return site


def peer_exchange_ready():
    """True when the exchanges run over peer memory (kernels on the caller's current stream), not NCCL collectives."""
    return bool(_peer["sites"]) and _peer["why_not"] is None and not _peer["disabled"]


def exchange_name():
    if _peer["sites"] and _peer["why_not"] is None:
        return "NVLink peer stores + signals (ssac_peer_put / ssac_peer_wait / ssac_peer_allreduce over symmetric memory)"
    why = "disabled" if _peer["disabled"] else (_peer["why_not"] or "not used yet / CPU tensors")
    return f"torch.distributed collectives (peer exchange unavailable: {why})"


def local_range(n_global, world, rank):
    """Contiguous block of nets owned by ``rank``: sizes differ by at most one, the first ``n % world`` ranks get the
    extra net (10 nets over 8 ranks -> 2,2,1,1,1,1,1,1)."""
    base, extra = divmod(n_global, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def _enable(kind, n, group):
    if _state["kind"] not in (None, kind):
        raise NotImplementedError(f"the {_state['kind']} are sharded already: critic, member and batch sharding "
                                  "cannot be combined")
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    if n is None:
        _state.update(kind=kind, group=group, world=world, rank=rank, n=None)
        return None
    if n < world:
        raise ValueError(f"{n} {kind} cannot be sharded over {world} ranks")
    _state.update(kind=kind, group=group, world=world, rank=rank, n=int(n))
    return local_range(n, world, rank)


def enable_critic_sharding(num_critics_global, group=None):
    """Call after ``dist.init_process_group``; returns (lo, hi), the global ids of this rank's critics.  Build the Agent
    with ``num_critics = hi - lo``."""
    return _enable("critics", num_critics_global, group)


def enable_member_sharding(ensemble_size_global, group=None):
    """Call after ``dist.init_process_group``; returns (lo, hi), the global ids of this rank's members.  Build the Agent
    with ``ensemble_size = hi - lo``."""
    return _enable("members", ensemble_size_global, group)


def enable_batch_sharding(group=None):
    """Call after ``dist.init_process_group``: every update splits its batch over the ranks (``batch_range``).  Build the
    same Agent, target agent, optimisers and replay buffer on every rank and push the same transitions on every rank."""
    _enable("batch", None, group)


def batch_range(batch_size):
    """Rows [lo, hi) of a batch of ``batch_size`` that this rank computes (all of them unless the batch is sharded)."""
    if not batches_sharded():
        return 0, int(batch_size)
    if batch_size < _state["world"]:
        raise ValueError(f"a batch of {batch_size} rows cannot be sharded over {_state['world']} ranks")
    return local_range(int(batch_size), _state["world"], _state["rank"])


def local_aug_rows(batch_size, aug_mix, lo, hi):
    """How many of rows [lo, hi) are augmented: the batch's first int(B * aug_mix) rows, counted in global row numbers."""
    return min(max(int(batch_size * aug_mix) - lo, 0), hi - lo)


def disable():
    _state.update(kind=None, group=None, world=1, rank=0, n=None)


def sharded():
    return _state["kind"] is not None


def critics_sharded():
    return _state["kind"] == "critics"


def members_sharded():
    return _state["kind"] == "members"


def batches_sharded():
    return _state["kind"] == "batch"


def world_size():
    """The number of ranks the active sharding spans (1 when nothing is sharded)."""
    return _state["world"]


def n_global(n_local):
    """The number of critics per member the losses are normalised with: every rank's when the critics are sharded."""
    return _state["n"] if critics_sharded() else n_local


def members_global(e_local):
    """The ensemble size the losses are normalised with: every rank's members when the members are sharded."""
    return _state["n"] if members_sharded() else e_local


def my_range():
    """Global ids [lo, hi) of this rank's critics or members."""
    return local_range(_state["n"], _state["world"], _state["rank"])


def my_members():
    """Global ids [lo, hi) of this rank's members (members sharded)."""
    return my_range()


def member_id(i):
    """Global id of local member i, for per-member log keys."""
    return i + my_range()[0] if members_sharded() else i


def same_member_choice(e):
    """``random.choice(range(e))`` -- the reference's host draw of the member whose critics rate a batch (priority refresh,
    filter statistics) -- made the same on every rank when the critics are sharded: the ranks then exchange that
    member's critic rows, so they must all evaluate the same member, and Python's ``random`` state is not kept in step
    across ranks.  Every rank draws (its RNG stream advances as unsharded) and rank 0's pick is broadcast: one host round
    trip, on those eager paths only."""
    member = random.choice(range(e))
    if e > 1 and critics_sharded():
        box = [member]
        dist.broadcast_object_list(box, group=_state["group"], group_src=0)
        member = int(box[0])
    return member


def all_gather_q(q_local, site="q", select=None):
    """q_local [n_local, B, ...] -> [N_global, B, ...] in global net order (or only the rows ``select``).  ``site`` names
    the call site: every site has its own symmetric buffer and signals."""
    return _all_gather_rows(q_local, site, select=select)


def _all_gather_rows(q_local, site_name, select=None, n=None):
    """``select`` (device int32 [m]): return only those global rows (cheaper than gathering everything and indexing).
    ``n``: the global number of rows (default: the sharded units)."""
    world, rank, group = _state["world"], _state["rank"], _state["group"]
    n = _state["n"] if n is None else int(n)
    row = q_local[0].numel() * q_local.element_size() if q_local.shape[0] else 0
    site = _site(site_name, n * row, group, q_local.device) if row else None
    if site is not None:
        site.put(q_local, local_range(n, world, rank)[0] * row)
        if select is not None:
            out = torch.empty((select.numel(),) + tuple(q_local.shape[1:]), dtype=q_local.dtype, device=q_local.device)
            site.wait(out, row_index=select, total_bytes=n * row)
        else:
            out = torch.empty((n,) + tuple(q_local.shape[1:]), dtype=q_local.dtype, device=q_local.device)
            site.wait(out)
        return out
    n_max = -(-n // world)
    pad = torch.zeros((n_max,) + tuple(q_local.shape[1:]), dtype=q_local.dtype, device=q_local.device)
    pad[: q_local.shape[0]].copy_(q_local)
    out = torch.empty((world * n_max,) + tuple(q_local.shape[1:]), dtype=q_local.dtype, device=q_local.device)
    dist.all_gather_into_tensor(out, pad, group=group)
    if n == world * n_max:
        return out if select is None else out.index_select(0, select.long())
    rows = []
    for r in range(world):
        lo, hi = local_range(n, world, r)
        rows.append(out[r * n_max: r * n_max + (hi - lo)])
    out = torch.cat(rows, dim=0)
    return out if select is None else out.index_select(0, select.long())


def all_reduce_sum_(t, site="sum"):
    world, group = _state["world"], _state["group"]
    peer = _site(site, world * t.numel() * t.element_size(), group, t.device)
    if peer is not None:
        # every rank lands its partial in slot `rank` of every peer, then sums the slots in rank order: the same
        # arithmetic on every rank (replicas stay bit-identical), no ring order to depend on
        parts = torch.empty((world,) + tuple(t.shape), dtype=t.dtype, device=t.device)
        peer.put(t, _state["rank"] * t.numel() * t.element_size())
        peer.wait(parts)
        t.copy_(parts.sum(0))
        return t
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t


def all_reduce_members_(t):
    """Sum ``t`` over the ranks of a member-sharded ensemble."""
    return all_reduce_sum_(t, site="members_sum")


def reduce_logged(loss_v, last=None, site="logged"):
    """The logged values of a sharded update made the single-GPU ones, in one exchange of one or two floats: the sum of
    this rank's loss slots ``loss_v`` over every rank is left in loss_v[0] (the other slots are cleared), and ``last``, a
    value of this rank's last net or member, becomes that of the rank that owns the ensemble's last one."""
    red = torch.empty(1 if last is None else 2, dtype=torch.float32, device=loss_v.device)
    torch.sum(loss_v, 0, keepdim=True, out=red[0:1])
    if last is not None:
        if my_range()[1] == _state["n"]:
            red[1:2].copy_(last)
        else:
            red[1:2].zero_()
    all_reduce_sum_(red, site)
    loss_v.zero_()
    loss_v[0:1].copy_(red[0:1])
    if last is not None:
        last.copy_(red[1:2])


def all_gather_members(x_local):
    """x_local [E_local * k, ...] (k rows per member, member-major) -> [E_global * k, ...] in global member order."""
    lo, hi = my_range()
    k = x_local.shape[0] // (hi - lo)
    x = x_local.reshape((hi - lo, k) + tuple(x_local.shape[1:]))
    out = _all_gather_rows(x.contiguous(), "members%d" % (x[0].numel() if x.shape[0] else 0))
    return out.reshape((_state["n"] * k,) + tuple(x_local.shape[1:]))


def all_gather_batch(x_local, batch_size, site):
    """x_local [hi - lo, ...] (this rank's rows of a batch-sharded update) -> [batch_size, ...] in global row order: the
    per-row values whose statistics are logged (TD targets, log-probs) then go through the unchanged single-GPU kernels."""
    return _all_gather_rows(x_local.contiguous(), site, n=batch_size)


class _AllreduceSite:
    """Symmetric buffer of ssac_peer_allreduce: two epoch halves of {in, out} regions of ``cap`` bytes, a symmetric
    signal row of 128 uint32 (staged / reduced), a device epoch and the local ticket counters of the kernels' last block."""

    def __init__(self, n, group, device):
        import torch.distributed._symmetric_memory as symm

        from . import _lib

        self.lib = _lib
        self.group = group if group is not None else dist.group.WORLD
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.n = int(n)
        self.cap = (4 * self.n + 15) // 16 * 16
        name = self.group.group_name
        try:
            symm.enable_symm_mem_for_group(name)
        except Exception:  # noqa: BLE001  (newer torch enables groups lazily)
            pass
        self.buf = symm.empty(4 * self.cap, dtype=torch.uint8, device=device)
        self.sig = symm.empty(128, dtype=torch.int32, device=device)
        self.sig.zero_()
        self._hb = symm.rendezvous(self.buf, name)
        self._hs = symm.rendezvous(self.sig, name)
        self.buf_ptrs = torch.tensor([int(p) for p in self._hb.buffer_ptrs], dtype=torch.int64, device=device)
        self.sig_ptrs = torch.tensor([int(p) for p in self._hs.buffer_ptrs], dtype=torch.int64, device=device)
        self.epoch = torch.zeros(1, dtype=torch.int32, device=device)
        self.ticket = torch.zeros(2, dtype=torch.int32, device=device)
        torch.cuda.synchronize(device)
        dist.barrier(group=group)   # every rank's signals are zeroed and mapped before the first stage

    def __call__(self, src, dst):
        self.lib.lib().peer_allreduce(src.data_ptr(), dst.data_ptr(), self.n, self.buf.data_ptr(), self.cap,
                                      self.buf_ptrs.data_ptr(), self.sig.data_ptr(), self.sig_ptrs.data_ptr(), self.rank,
                                      self.world, self.epoch.data_ptr(), self.ticket.data_ptr(), self.lib.stream_ptr())


def _allreduce_site(name, n, group, device):
    """The all-reduce site ``name`` for n floats (created on first use, outside any stream capture), or None when peer
    memory is not available (the reason is kept for ``exchange_name()``), as ``_site``."""
    if _peer["disabled"] or _peer["why_not"] is not None or device.type != "cuda":
        return None
    key = ("allreduce", name, int(n), id(group))
    site = _peer["sites"].get(key)
    if site is None:
        if torch.cuda.is_current_stream_capturing():
            return None
        try:
            site = _peer["sites"][key] = _AllreduceSite(n, group, device)
        except Exception as e:  # noqa: BLE001
            _peer["why_not"] = f"{type(e).__name__}: {str(e)[:120]}"
            return None
    return site


def all_reduce_flat_(t, site):
    """Sum the contiguous fp32 tensor ``t`` (a flat gradient arena) over the ranks in place, with the same bits on every
    rank: ssac_peer_allreduce over NVLink peer memory, else ``torch.distributed.all_reduce``.  ``site`` names the call
    site (one symmetric buffer each, used from one stream)."""
    if not t.is_contiguous() or t.dtype != torch.float32:
        raise ValueError("all_reduce_flat_: a contiguous fp32 tensor")
    if t.numel() == 0:
        return t
    peer = _allreduce_site(site, t.numel(), _state["group"], t.device)
    if peer is not None:
        peer(t, t)
        return t
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=_state["group"])
    return t

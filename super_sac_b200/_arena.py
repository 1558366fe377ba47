"""Flat HBM layout of the ensemble parameters, the fused Adam adapter and the workspace cache.

All E*N critic nets (and all E actors) of an Agent live in ONE contiguous fp32 arena, net-major per array:

    [ W1: G x H x D | b1: G x H | W2: G x H x H | b2: G x H | W3: G x O x H | b3: G x O ]   (G = E*N or E)

so that (a) one grouped launch walks every net with uniform strides (ssac_mlp_forward/backward), (b) Adam and
Polyak are single coalesced passes over the arena (ssac_adam_step / ssac_polyak), and (c) the nn.Parameters the
reference API exposes (``critics[i].nets[k].fc1.weight`` ...) are views into it -- ``parameters()``,
``state_dict()``, ``Agent.save/load`` and the caller's ``torch.optim.Adam(...)`` construction (main.py:188-227)
keep working.  Gradients live in a twin arena and are exposed as the ``.grad`` of the same Parameters.
Each array starts on a 128-byte boundary (vector loads now, TMA tiles later); pad elements stay zero.
"""
import torch

from . import _lib

NAMES = ("W1", "b1", "W2", "b2", "W3", "b3")
_ALIGN = 32  # floats (128 B)


def _last_linear(module):
    if hasattr(module, "out"):
        return module.out
    return module.act_p if hasattr(module, "act_p") else module.fc3   # act_p: DiscreteActor (nets/mlps.py:137)


def supported_mlp(module):
    """True for modules with the fc1 / fc2 / (out|fc3) nn.Linear structure the grouped kernels implement."""
    try:
        lins = (module.fc1, module.fc2, _last_linear(module))
    except AttributeError:
        return False
    if not all(isinstance(l, torch.nn.Linear) and l.bias is not None for l in lins):
        return False
    n_params = sum(1 for _ in module.parameters())
    return n_params == 6 and lins[0].out_features == lins[1].in_features == lins[1].out_features == lins[2].in_features


class MLPArena:
    def __init__(self, G, D, H, O, device="cpu"):
        self.G, self.D, self.H, self.O = G, D, H, O
        per_net = {"W1": H * D, "b1": H, "W2": H * H, "b2": H, "W3": O * H, "b3": O}
        self.shapes = {"W1": (G, H, D), "b1": (G, H), "W2": (G, H, H), "b2": (G, H), "W3": (G, O, H), "b3": (G, O)}
        self.net_stride = per_net
        self.offsets = {}
        off = 0
        for n in NAMES:
            self.offsets[n] = off
            off += G * per_net[n]
            off = (off + _ALIGN - 1) // _ALIGN * _ALIGN
        self.numel = off
        # Tail padding (never part of `numel`): keeps the TMA boxes of the last net's matrices inside the allocation even
        # when the arena is the last thing in its cudaMalloc block (csrc/ssac_mlp_tc.cu make_map explains what was
        # measured: a tensor map must not declare an extent that leaves mapped memory).
        self._pad = 128 * max(H, D) + 1024
        self.flat = self._alloc(device)
        self.grad = self._alloc(device)
        self.modules = []
        self._make_views()

    def _alloc(self, device, like=None):
        store = torch.zeros(self.numel + self._pad, dtype=torch.float32, device=device)
        if like is not None:
            store[: self.numel].copy_(like)
        return store[: self.numel]

    def _make_views(self):
        self.p = {}
        self.g = {}
        for n in NAMES:
            o, shape = self.offsets[n], self.shapes[n]
            cnt = 1
            for s in shape:
                cnt *= s
            self.p[n] = self.flat[o:o + cnt].view(shape)
            self.g[n] = self.grad[o:o + cnt].view(shape)

    @property
    def device(self):
        return self.flat.device

    def _module_params(self, m):
        last = _last_linear(m)
        return {"W1": m.fc1.weight, "b1": m.fc1.bias, "W2": m.fc2.weight, "b2": m.fc2.bias, "W3": last.weight, "b3": last.bias}

    def bind(self, modules):
        """Adopt the current values of ``modules`` (len G) and re-point their Parameters at the arena."""
        assert len(modules) == self.G
        self.modules = list(modules)
        with torch.no_grad():
            for g, m in enumerate(modules):
                for n, prm in self._module_params(m).items():
                    self.p[n][g].copy_(prm.data.to(self.device))
        self._rebind()

    def _rebind(self):
        for g, m in enumerate(self.modules):
            for n, prm in self._module_params(m).items():
                prm.data = self.p[n][g]
                prm.grad = self.g[n][g]

    def to(self, device):
        if torch.device(device) != self.flat.device:
            self.flat = self._alloc(device, like=self.flat)
            self.grad = self._alloc(device, like=self.grad)
            self._make_views()
            self._rebind()
        return self

    def parameters(self):
        for m in self.modules:
            yield from self._module_params(m).values()

    # raw pointers for the C ABI -------------------------------------------------------------
    def ptr(self, name, g0=0, grad=False):
        t = (self.g if grad else self.p)[name]
        return t.data_ptr() + 4 * g0 * self.net_stride[name]

    def ptrs(self, g0=0, grad=False):
        return tuple(self.ptr(n, g0, grad) for n in NAMES)

    def range_table(self, g0, g1):
        """[(offset, numel)] of nets g0..g1-1 inside the flat arena (6 ranges; one if g0..g1 is everything)."""
        if g0 == 0 and g1 == self.G:
            return [(0, self.numel)]
        return [(self.offsets[n] + g0 * self.net_stride[n], (g1 - g0) * self.net_stride[n]) for n in NAMES]


class FlatAdam:
    """Routes a caller-built ``torch.optim.Adam`` over arena parameters to ssac_adam_step.

    The reference training loop constructs stock Adam objects itself (main.py:188-239) and hands them to the
    update functions, so the drop-in recognises them: hyper-parameters are read from ``param_groups[0]`` on every
    step, the moments live in flat buffers next to the arena and are exposed through ``optimizer.state`` with the
    usual keys, and the step counter lives in device memory (graph replays advance it).
    """

    def __init__(self, optimizer, arena):
        if not isinstance(optimizer, torch.optim.Adam) or len(optimizer.param_groups) != 1:
            raise NotImplementedError("the fused path needs a single-group torch.optim.Adam (as built by main.py:188-239)")
        pg = optimizer.param_groups[0]
        if pg.get("amsgrad", False) or pg.get("maximize", False):
            raise NotImplementedError("amsgrad / maximize are not supported by ssac_adam_step")
        want = {id(p) for p in arena.parameters()}
        have = {id(p) for p in pg["params"]}
        if want != have:
            raise NotImplementedError("optimizer parameters do not coincide with the agent's ensemble parameters")
        self.optimizer, self.arena = optimizer, arena
        dev = arena.device
        self.m = torch.zeros_like(arena.flat)
        self.v = torch.zeros_like(arena.flat)
        self.ctl = torch.zeros(2, dtype=torch.int32, device=dev)   # [0] step, [1] blocks done
        self.gnorm_sq = torch.zeros(1, dtype=torch.float32, device=dev)
        self.steps = 0
        self._step_tensor = torch.zeros((), dtype=torch.float32)
        mviews, vviews = {}, {}
        for n in NAMES:
            o, shape = arena.offsets[n], arena.shapes[n]
            cnt = 1
            for s in shape:
                cnt *= s
            mviews[n] = self.m[o:o + cnt].view(shape)
            vviews[n] = self.v[o:o + cnt].view(shape)
        for g, mod in enumerate(arena.modules):
            for n, prm in arena._module_params(mod).items():
                st = optimizer.state[prm]
                if "exp_avg" in st:  # resuming from a loaded optimizer state
                    mviews[n][g].copy_(st["exp_avg"])
                    vviews[n][g].copy_(st["exp_avg_sq"])
                    self.steps = int(st["step"])
                st["step"] = self._step_tensor
                st["exp_avg"] = mviews[n][g]
                st["exp_avg_sq"] = vviews[n][g]
        if self.steps:
            self.ctl[0] = self.steps
            self._step_tensor.fill_(self.steps)

    @classmethod
    def attach(cls, optimizer, arena):
        cur = getattr(optimizer, "_ssac_flat_adam", None)
        if cur is not None and cur.arena is arena and cur.m.device == arena.device:
            # optimizer.load_state_dict() replaces optimizer.state with fresh tensors: the fused step would keep using its
            # private moments and silently ignore the loaded ones.  Probe one parameter: if its exp_avg no longer aliases
            # the flat buffer, re-import the state (the constructor copies exp_avg / exp_avg_sq / step back in).
            p0 = cur.__dict__.get("_probe")
            if p0 is None:   # (walking the module tree on every update call costs more than the probe itself)
                p0 = cur._probe = next(iter(arena.parameters()), None)
            st = optimizer.state.get(p0) if p0 is not None else None
            if st is None or "exp_avg" not in st or st["exp_avg"].data_ptr() != cur.m.data_ptr() + 4 * arena.offsets["W1"]:
                cur = None
        else:
            cur = None
        if cur is None:
            cur = cls(optimizer, arena)
            optimizer._ssac_flat_adam = cur
        return cur

    def hyper(self):
        pg = self.optimizer.param_groups[0]
        return float(pg["lr"]), float(pg["betas"][0]), float(pg["betas"][1]), float(pg["eps"]), float(pg["weight_decay"])

    def grad_norm_sq(self, stream):
        """sum g^2 over the arena into self.gnorm_sq (device)."""
        _lib.lib().sumsq(self.arena.grad.data_ptr(), self.arena.numel, self.gnorm_sq.data_ptr(), 0, stream)
        return self.gnorm_sq

    def step(self, stream, max_norm=None, target_arena=None, tau=0.0):
        lr, b1, b2, eps, wd = self.hyper()
        a = self.arena
        clip = max_norm is not None and max_norm > 0
        gptr = self.gnorm_sq.data_ptr() if clip else None
        if target_arena is not None:
            _lib.lib().adam_polyak_step(a.flat.data_ptr(), a.grad.data_ptr(), self.m.data_ptr(), self.v.data_ptr(),
                                        target_arena.flat.data_ptr(), a.numel, self.ctl.data_ptr(), lr, b1, b2, eps, wd,
                                        gptr, float(max_norm or 0.0), 1, float(tau), stream)
        else:
            _lib.lib().adam_step(a.flat.data_ptr(), a.grad.data_ptr(), self.m.data_ptr(), self.v.data_ptr(), a.numel,
                                 self.ctl.data_ptr(), lr, b1, b2, eps, wd, gptr, float(max_norm or 0.0), 1, stream)
        if not torch.cuda.is_current_stream_capturing():   # a captured step executes (and is counted) at replay time
            self.steps += 1
            self._step_tensor.fill_(self.steps)

    def note_replayed_step(self):
        """A captured graph containing this optimiser's step was replayed: the device counter advanced by itself."""
        self.steps += 1
        self._step_tensor.fill_(self.steps)


class Workspace:
    """Pointer-stable scratch tensors keyed by name (CUDA-graph friendly, no allocator traffic per update)."""

    def __init__(self):
        self._bufs = {}

    def get(self, key, shape, dtype=torch.float32, device=None, zero=False):
        shape = tuple(int(s) for s in shape)
        t = self._bufs.get(key)
        if t is None or t.shape != shape or t.dtype != dtype or (device is not None and t.device != torch.device(device)):
            t = torch.zeros(shape, dtype=dtype, device=device)
            self._bufs[key] = t
        elif zero:
            t.zero_()
        return t

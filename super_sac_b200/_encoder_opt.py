"""Optimiser step of a native pixel encoder (nets.cnns.BigPixelEncoder) as ONE fused launch.

The caller owns a plain ``torch.optim.Adam(agent.encoder.parameters())`` (main.py:203-209).  When every gradient it would
consume lives in the encoder's flat gradient buffer (``BigPixelEncoder._flatten``), ``clip_grad_norm_`` + ``step()``
(learning.py:122-131) become ``ssac_sumsq`` + ``ssac_adam_step`` over that buffer -- same arithmetic as torch's
``_single_tensor_adam`` (csrc/ssac_common.cuh adam1) -- and the optimiser's ``state`` keeps aliasing the fused moments, so
``state_dict()`` / checkpoints see what torch would have produced.  Anything else (a user encoder with further trainable
parameters, accumulated or copied gradients, several parameter groups, amsgrad ...) returns None and the caller runs the
torch path.
"""
import os

import torch

from . import _lib


def native_nets(encoder):
    nets = encoder.__dict__.get("_ssac_native_nets")
    if nets is None:
        from .nets import cnns

        nets = encoder.__dict__["_ssac_native_nets"] = [m for m in encoder.modules() if isinstance(m, cnns.BigPixelEncoder)]
    return nets


class FlatParamAdam:
    def __init__(self, optimizer, net):
        self.optimizer, self.net = optimizer, net
        self.flat, self.grad = net._flat, net._flat_grad
        self.m, self.v = torch.zeros_like(self.flat), torch.zeros_like(self.flat)
        self.ctl = torch.zeros(2, dtype=torch.int32, device=self.flat.device)
        self.gnorm_sq = torch.zeros(1, dtype=torch.float32, device=self.flat.device)
        self.steps = 0
        self._step_tensor = torch.zeros((), dtype=torch.float32)
        for p, o in zip(net._native_params(), net._flat_off):
            st = optimizer.state[p]
            mv, vv = self.m[o:o + p.numel()].view(p.shape), self.v[o:o + p.numel()].view(p.shape)
            if "exp_avg" in st:   # resuming from a loaded / torch-stepped optimizer state
                mv.copy_(st["exp_avg"])
                vv.copy_(st["exp_avg_sq"])
                self.steps = int(st["step"])
            st["step"], st["exp_avg"], st["exp_avg_sq"] = self._step_tensor, mv, vv
        if self.steps:
            self.ctl[0] = self.steps
            self._step_tensor.fill_(self.steps)

    @classmethod
    def attach(cls, optimizer, net):
        cur = getattr(optimizer, "_ssac_flat_param_adam", None)
        if cur is not None and cur.net is net and cur.flat is net._flat:
            p0 = net.conv1.weight
            st = optimizer.state.get(p0)
            if st is not None and "exp_avg" in st and st["exp_avg"].data_ptr() == cur.m.data_ptr():
                return cur
        cur = optimizer._ssac_flat_param_adam = cls(optimizer, net)
        return cur

    def step(self, stream, max_norm):
        pg = self.optimizer.param_groups[0]
        L = _lib.lib()
        clip = max_norm is not None and max_norm > 0
        if clip:
            L.sumsq(self.grad.data_ptr(), self.grad.numel(), self.gnorm_sq.data_ptr(), 0, stream)
        L.adam_step(self.flat.data_ptr(), self.grad.data_ptr(), self.m.data_ptr(), self.v.data_ptr(), self.flat.numel(),
                    self.ctl.data_ptr(), float(pg["lr"]), float(pg["betas"][0]), float(pg["betas"][1]), float(pg["eps"]),
                    float(pg["weight_decay"]), self.gnorm_sq.data_ptr() if clip else None, float(max_norm or 0.0), 1, stream)
        if not torch.cuda.is_current_stream_capturing():
            self.steps += 1
            self._step_tensor.fill_(self.steps)


def structurally_eligible(encoder, optimizer=None):
    """What can be known BEFORE an update runs: the encoder's only trainable parameters of any size are those of one native
    net that has already been flattened (and, given the optimiser, that it is a plain single-group Adam over them).  Such
    an update hands nothing to torch.autograd that a CUDA graph could not replay."""
    nets = native_nets(encoder)
    if len(nets) != 1 or nets[0].__dict__.get("_flat") is None:
        return False
    own = {id(p) for p in nets[0]._native_params()}
    if any(p.numel() > 2 and p.requires_grad and id(p) not in own for p in encoder.parameters()):
        return False
    if optimizer is not None:
        if not isinstance(optimizer, torch.optim.Adam) or len(optimizer.param_groups) != 1:
            return False
        pg = optimizer.param_groups[0]
        if pg.get("amsgrad") or pg.get("maximize") or pg.get("capturable") or pg.get("differentiable"):
            return False
    return os.environ.get("SSAC_ENCODER_OPT") != "torch"


def note_replayed_step(encoder, optimizer):
    """A captured graph containing the fused encoder step was replayed: the device counter advanced by itself."""
    st = getattr(optimizer, "_ssac_flat_param_adam", None)
    if st is not None:
        st.steps += 1
        st._step_tensor.fill_(st.steps)


def eligible(encoder, optimizer):
    """The native net whose flat gradient buffer holds every gradient `optimizer` would consume, or None."""
    nets = native_nets(encoder)
    if len(nets) != 1 or len(optimizer.param_groups) != 1 or not isinstance(optimizer, torch.optim.Adam):
        return None
    net, pg = nets[0], optimizer.param_groups[0]
    flat = net.__dict__.get("_flat")
    if flat is None or pg.get("amsgrad") or pg.get("maximize") or pg.get("capturable") or pg.get("differentiable"):
        return None
    g0 = net._flat_grad.data_ptr()
    own = {id(p): o for p, o in zip(net._native_params(), net._flat_off)}
    adopt = []
    for p in pg["params"]:
        o = own.get(id(p))
        if o is None:
            if p.grad is not None:
                return None
        elif p.grad is None or p.data_ptr() != flat.data_ptr() + 4 * o:
            return None
        elif p.grad.data_ptr() != g0 + 4 * o:
            adopt.append((p, o))
    # autograd normally adopts the views the backward wrote as `.grad`; where it chose to copy instead (it may, e.g. when
    # something else still references the gradient), move the copy into the flat buffer and alias it
    for p, o in adopt:
        if p.grad.dtype != torch.float32 or not p.grad.is_contiguous():
            return None
        view = net._flat_grad[o:o + p.numel()].view(p.shape)
        with torch.no_grad():
            view.copy_(p.grad)
        p.grad = view
    return net


def fused_step(encoder, optimizer, max_norm):
    """clip_grad_norm_(encoder.parameters(), max_norm) + optimizer.step() as sumsq + one Adam launch.  Returns the net whose
    flat gradient was consumed (its post-clip norm can then be logged with one more ssac_sumsq), or None if not eligible."""
    if os.environ.get("SSAC_ENCODER_OPT") == "torch":   # A/B switch for tests: always the torch calls
        return None
    net = eligible(encoder, optimizer)
    if net is None:
        return None
    FlatParamAdam.attach(optimizer, net).step(_lib.stream_ptr(), max_norm)
    return net


def grad_norm_sq_into(net, out_slot_tensor):
    """sum g^2 of the flat gradient into a 1-element device tensor (a log slot)."""
    _lib.lib().sumsq(net._flat_grad.data_ptr(), net._flat_grad.numel(), out_slot_tensor.data_ptr(), 0, _lib.stream_ptr())

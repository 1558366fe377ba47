"""Pixel encoders (reference nets/cnns.py:37-103).

``BigPixelEncoder`` -- the DrQ / DrQv2 encoder of the pixel configs -- keeps the reference's ``nn.Module`` shell
(parameter names and shapes, so ``state_dict`` / optimisers / ``deepcopy`` / Polyak keep working) but on a CUDA tensor its
forward and backward are the library's tcgen05 implicit-GEMM kernels (``ssac_conv_encoder_forward / _backward``,
csrc/ssac_conv.cu; SURVEY 8f row N3), handed to autograd as one ``torch.autograd.Function``.  There is no cuDNN or ATen
fallback on the GPU: a missing library raises.  On CPU tensors the module is the plain PyTorch definition (state-dict
round trips and host-side tests).
"""
import ctypes
import os

import torch
import torch.nn.functional as F
from torch import nn

from . import weight_init


def _conv_out(size, kernel, stride):
    return (size - (kernel - 1) - 1) // stride + 1


class _Workspace:
    """Zero-initialised device workspaces of the native encoder, one per (batch, save) and recycled once the backward
    that needs the saved activations has run."""

    def __init__(self):
        self.free = {}

    def take(self, key, n_floats, device):
        pool = self.free.setdefault(key, [])
        if pool:
            return pool.pop()
        return torch.zeros(n_floats, dtype=torch.float32, device=device)

    def give(self, key, ws):
        self.free.setdefault(key, []).append(ws)


class _EncoderFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, module, obs, *params):
        from .. import _lib

        lib = _lib.lib()
        B, C, H, W = obs.shape
        O = module.embedding_dim
        save = 1 if any(ctx.needs_input_grad[2:]) else 0
        # (one workspace per shape: every update path that may run encoders on several streams at once -- member lanes,
        # pipelined blocks -- excludes agents with a parameterised encoder, learning_utils._encoder_trainable)
        key = (B, C, H, W, save, obs.device)
        n = ctypes.c_int64()
        lib.conv_encoder_ws_floats(B, C, H, W, O, save, ctypes.byref(n))
        ws = module._ws.take(key, n.value, obs.device)
        out = torch.empty(B, O, dtype=torch.float32, device=obs.device)
        pp = _lib.host_array(ctypes.c_void_p, [p.data_ptr() for p in params])
        lib.conv_encoder_forward(obs.data_ptr(), B, C, H, W, O, pp, ws.data_ptr(), save, out.data_ptr(), _lib.stream_ptr())
        if save:
            ctx.module, ctx.key, ctx.ws, ctx.dims = module, key, ws, (B, C, H, W, O)
            ctx.save_for_backward(out, obs, *params)
        else:
            module._ws.give(key, ws)
        return out

    @staticmethod
    def backward(ctx, dout):
        from .. import _lib

        lib = _lib.lib()
        out, obs, *params = ctx.saved_tensors
        B, C, H, W, O = ctx.dims
        dout = dout.contiguous()
        grads = ctx.module._grad_targets(params)
        pp = _lib.host_array(ctypes.c_void_p, [p.data_ptr() for p in params])
        gp = _lib.host_array(ctypes.c_void_p, [g.data_ptr() for g in grads])
        lib.conv_encoder_backward(dout.data_ptr(), out.data_ptr(), obs.data_ptr(), B, C, H, W, O, pp, ctx.ws.data_ptr(), gp, _lib.stream_ptr())
        ctx.module._ws.give(ctx.key, ctx.ws)
        ctx.ws = None
        return (None, None, *grads)


class BigPixelEncoder(nn.Module):
    """DrQ encoder: conv3x3(32) s2,1,1,1 -> FC -> LayerNorm -> tanh on obs/255 - 0.5 (nets/cnns.py:37-69)."""

    def __init__(self, obs_shape, out_dim=50):
        super().__init__()
        c, h, w = obs_shape
        self.conv1 = nn.Conv2d(c, 32, kernel_size=3, stride=2)
        self.conv2 = nn.Conv2d(32, 32, kernel_size=3, stride=1)
        self.conv3 = nn.Conv2d(32, 32, kernel_size=3, stride=1)
        self.conv4 = nn.Conv2d(32, 32, kernel_size=3, stride=1)
        h, w = _conv_out(h, 3, 2), _conv_out(w, 3, 2)
        for _ in range(3):
            h, w = _conv_out(h, 3, 1), _conv_out(w, 3, 1)
        self.fc = nn.Linear(h * w * 32, out_dim)
        self.ln = nn.LayerNorm(out_dim)
        self.apply(weight_init)
        self.embedding_dim = out_dim
        self._ws = _Workspace()

    def __deepcopy__(self, memo):
        # target_agent = deepcopy(agent) (main.py:321): parameters are copied, workspaces are not shared
        import copy

        cls = self.__class__
        new = cls.__new__(cls)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            if k in ("_flat", "_flat_off", "_flat_grad"):
                continue
            new.__dict__[k] = _Workspace() if k == "_ws" else copy.deepcopy(v, memo)
        return new

    def __getstate__(self):
        # pickling (torch.save(agent)): parameters travel, device workspaces and the flat-buffer bookkeeping do not
        state = dict(self.__dict__)
        for k in ("_ws", "_flat", "_flat_off", "_flat_grad"):
            state.pop(k, None)
        return state

    def __setstate__(self, state):
        self.__dict__.update(state)
        self.__dict__["_ws"] = _Workspace()

    def _flatten(self):
        """Parameters as views of ONE contiguous buffer (and a twin gradient buffer), so that Adam, gradient clipping and
        the logged gradient norm are one launch each (_encoder_opt.py) instead of a dozen per tensor.  Lazy: `.to()` /
        deepcopy / load_state_dict(assign=True) give the parameters fresh storage, noticed here by address."""
        ps = self._native_params()
        flat = self.__dict__.get("_flat")
        if flat is not None and flat.device == ps[0].device and all(
                p.data_ptr() == flat.data_ptr() + 4 * o for p, o in zip(ps, self._flat_off)):
            return
        offs, n = [], 0
        for p in ps:
            offs.append(n)
            n += (p.numel() + 3) & ~3
        flat = torch.zeros(n, dtype=torch.float32, device=ps[0].device)
        with torch.no_grad():
            for p, o in zip(ps, offs):
                view = flat[o:o + p.numel()].view(p.shape)
                view.copy_(p)
                p.data = view
        self.__dict__["_flat"], self.__dict__["_flat_off"] = flat, offs
        self.__dict__["_flat_grad"] = torch.zeros_like(flat)

    def _grad_targets(self, params):
        """Where a backward writes its gradients: the views of the flat gradient buffer when nothing lives there yet (autograd
        then adopts them as `.grad` without a copy), else fresh tensors that autograd accumulates as usual."""
        flat = self.__dict__.get("_flat")
        own = self._native_params()
        if (flat is None or any(p.grad is not None for p in own)
                or any(q.data_ptr() != flat.data_ptr() + 4 * o for q, o in zip(params, self._flat_off))):
            return [torch.empty_like(p) for p in params]
        g = self._flat_grad
        return [g[o:o + p.numel()].view(p.shape) for p, o in zip(params, self._flat_off)]

    def _native_params(self):
        return (self.conv1.weight, self.conv1.bias, self.conv2.weight, self.conv2.bias, self.conv3.weight, self.conv3.bias,
                self.conv4.weight, self.conv4.bias, self.fc.weight, self.fc.bias, self.ln.weight, self.ln.bias)

    def native_supported(self, obs):
        return (obs.dim() == 4 and obs.shape[1] <= 16 and obs.shape[2] % 2 == 0 and obs.shape[3] % 2 == 0
                and min(obs.shape[2], obs.shape[3]) >= 16 and self.embedding_dim <= 64)

    def _check_geometry(self, obs):
        """The kernels size everything from the observation's shape: it has to be the shape the module was built for."""
        c, h, w = obs.shape[1:]
        vh, vw = h // 2 - 7, w // 2 - 7
        if c != self.conv1.in_channels or vh <= 0 or vw <= 0 or 32 * vh * vw != self.fc.in_features:
            raise ValueError(f"BigPixelEncoder built for {self.conv1.in_channels} channels / {self.fc.in_features} features "
                             f"got observations of shape {tuple(obs.shape[1:])}")

    def forward(self, obs):
        if obs.is_cuda and os.environ.get("SSAC_ENCODER_IMPL", "native") != "torch":
            if not self.native_supported(obs):
                raise NotImplementedError("BigPixelEncoder on CUDA: <= 16 channels, even sides >= 16, out_dim <= 64")
            self._check_geometry(obs)
            x = obs if obs.dtype == torch.float32 else obs.float()
            self._flatten()
            params = self._native_params()
            if not torch.is_grad_enabled():
                params = tuple(p.detach() for p in params)
            return _EncoderFn.apply(self, x.contiguous(), *params)
        x = (obs / 255.0) - 0.5
        x = F.relu(self.conv1(x))
        x = F.relu(self.conv2(x))
        x = F.relu(self.conv3(x))
        x = F.relu(self.conv4(x))
        x = self.fc(x.view(x.size(0), -1))
        return torch.tanh(self.ln(x))

"""TSCNet generator: the reference's nn.Module interface over the hand-written CUDA path.

``TSCNet(num_channel=64, num_features=201)`` keeps the reference's constructor, ``forward`` signature
(x: (B, 2, T, F), any strides -> (final_real, final_imag), each (B, 1, T, F)) and the 359-key state dict
(ref: generator.py:159-196), so ``load_state_dict(torch.load("best_ckpt/ckpt"))`` and the call sites in
train.py:100 / evaluation.py:40 work unchanged.  Nothing in ``forward``/``backward`` is a PyTorch compute
op: activations live channel-last as rows (b, t, f) x channels, every contraction is a ``cmgan_gemm_*``
call and everything else one of the HBM-bound kernels in csrc/.  PyTorch provides memory, streams and the
autograd graph node (one ``torch.autograd.Function`` for the whole network).
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional

import torch
import torch.nn as nn

from . import ops
from .conformer_block import C
from .network import tscnet_bwd, tscnet_fwd


# ====================================================================================== parameters / module
def _param_specs(num_channel: int, num_features: int):
    """[(key, shape, kind, fan_in)] in the reference's state-dict order (ref: generator.py:159-172)."""
    c = num_channel
    specs = []

    def conv(key, cout, cin, kh, kw, bias=True):
        specs.append((key + ".weight", (cout, cin, kh, kw), "kaiming", cin * kh * kw))
        if bias:
            specs.append((key + ".bias", (cout,), "bias", cin * kh * kw))

    def affine(key, n):
        specs.append((key + ".weight", (n,), "ones", 0))
        specs.append((key + ".bias", (n,), "zeros", 0))

    def prelu(key, n, init=0.25):
        specs.append((key + ".weight", (n,), ("const", init), 0))

    def dense(p):
        for i in range(1, 5):
            conv(f"{p}.conv{i}", c, c * i, 2, 3)
            affine(f"{p}.norm{i}", c)
            prelu(f"{p}.prelu{i}", c)

    def linear(key, nout, nin, bias=True):
        specs.append((key + ".weight", (nout, nin), "kaiming", nin))
        if bias:
            specs.append((key + ".bias", (nout,), "bias", nin))

    conv("dense_encoder.conv_1.0", c, 3, 1, 1)
    affine("dense_encoder.conv_1.1", c)
    prelu("dense_encoder.conv_1.2", c)
    dense("dense_encoder.dilated_dense")
    conv("dense_encoder.conv_2.0", c, c, 1, 3)
    affine("dense_encoder.conv_2.1", c)
    prelu("dense_encoder.conv_2.2", c)
    for i in range(1, 5):
        for name in ("time_conformer", "freq_conformer"):
            p = f"TSCB_{i}.{name}"
            for ff in ("ff1",):
                linear(f"{p}.{ff}.fn.fn.net.0", 4 * c, c)
                linear(f"{p}.{ff}.fn.fn.net.3", c, 4 * c)
                affine(f"{p}.{ff}.fn.norm", c)
            linear(f"{p}.attn.fn.to_q", c, c, bias=False)
            linear(f"{p}.attn.fn.to_kv", 2 * c, c, bias=False)
            linear(f"{p}.attn.fn.to_out", c, c)
            specs.append((f"{p}.attn.fn.rel_pos_emb.weight", (1025, c // 4), "normal", 0))
            affine(f"{p}.attn.norm", c)
            affine(f"{p}.conv.net.0", c)
            specs.append((f"{p}.conv.net.2.weight", (4 * c, c, 1), "kaiming", c))
            specs.append((f"{p}.conv.net.2.bias", (4 * c,), "bias", c))
            specs.append((f"{p}.conv.net.4.conv.weight", (2 * c, 1, 31), "kaiming", 31))
            specs.append((f"{p}.conv.net.4.conv.bias", (2 * c,), "bias", 31))
            affine(f"{p}.conv.net.5", 2 * c)
            specs.append((f"{p}.conv.net.5.running_mean", (2 * c,), "buf_zeros", 0))
            specs.append((f"{p}.conv.net.5.running_var", (2 * c,), "buf_ones", 0))
            specs.append((f"{p}.conv.net.5.num_batches_tracked", (), "buf_long", 0))
            specs.append((f"{p}.conv.net.7.weight", (c, 2 * c, 1), "kaiming", 2 * c))
            specs.append((f"{p}.conv.net.7.bias", (c,), "bias", 2 * c))
            linear(f"{p}.ff2.fn.fn.net.0", 4 * c, c)
            linear(f"{p}.ff2.fn.fn.net.3", c, 4 * c)
            affine(f"{p}.ff2.fn.norm", c)
            affine(f"{p}.post_norm", c)
    dense("mask_decoder.dense_block")
    conv("mask_decoder.sub_pixel.conv", 2 * c, c, 1, 3)
    conv("mask_decoder.conv_1", 1, c, 1, 2)
    affine("mask_decoder.norm", 1)
    prelu("mask_decoder.prelu", 1)
    conv("mask_decoder.final_conv", 1, 1, 1, 1)
    prelu("mask_decoder.prelu_out", num_features, -0.25)
    dense("complex_decoder.dense_block")
    conv("complex_decoder.sub_pixel.conv", 2 * c, c, 1, 3)
    prelu("complex_decoder.prelu", c)
    affine("complex_decoder.norm", c)
    conv("complex_decoder.conv", 2, c, 1, 2)
    return specs


def _init_tensor(shape, kind, fan_in):
    if kind == "kaiming":       # nn.Conv*/nn.Linear default: kaiming_uniform_(a=sqrt(5)) == U(-1/sqrt(fan_in), 1/sqrt(fan_in))
        b = 1.0 / math.sqrt(fan_in)
        return torch.empty(shape).uniform_(-b, b)
    if kind == "bias":
        b = 1.0 / math.sqrt(fan_in)
        return torch.empty(shape).uniform_(-b, b)
    if kind == "ones" or kind == "buf_ones":
        return torch.ones(shape)
    if kind == "zeros" or kind == "buf_zeros":
        return torch.zeros(shape)
    if kind == "normal":
        return torch.randn(shape)
    if kind == "buf_long":
        return torch.zeros(shape, dtype=torch.long)
    if isinstance(kind, tuple) and kind[0] == "const":
        return torch.full(shape, float(kind[1]))
    raise ValueError(kind)


class _Holder(nn.Module):
    """Name-space node of the parameter tree (no compute)."""


def _register(root: nn.Module, key: str, tensor: torch.Tensor, is_buffer: bool):
    parts = key.split(".")
    mod = root
    for part in parts[:-1]:
        if not hasattr(mod, part):
            mod.add_module(part, _Holder())
        mod = getattr(mod, part)
    if is_buffer:
        mod.register_buffer(parts[-1], tensor)
    else:
        mod.register_parameter(parts[-1], nn.Parameter(tensor))


class _TSCNetFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, module, training, seed, *params):
        P = module._tensor_dict()
        save = {} if any(ctx.needs_input_grad) else None
        fr, fi = tscnet_fwd(x, P, training, seed, save)
        ctx.module = module
        ctx.saved = save
        return fr, fi

    @staticmethod
    def backward(ctx, dfr, dfi):
        module = ctx.module
        S = ctx.saved
        if S is None:
            raise RuntimeError("TSCNet backward called but the forward pass did not record state")
        P = module._tensor_dict()
        G, ret = module._grad_targets()
        tscnet_bwd(S, dfr, dfi, P, G)
        ctx.saved = None
        return (None, None, None, None, *ret)


class TSCNet(nn.Module):
    """Drop-in for reference ``models.generator.TSCNet`` (generator.py:159-196)."""

    def __init__(self, num_channel: int = 64, num_features: int = 201):
        super().__init__()
        if num_channel != C:
            raise ValueError("the sm_100a kernels are specialised for num_channel=64 (the reference's only configuration)")
        self.num_channel, self.num_features = num_channel, num_features
        self._keys: List[str] = []
        for key, shape, kind, fan_in in _param_specs(num_channel, num_features):
            is_buf = isinstance(kind, str) and kind.startswith("buf_")
            _register(self, key, _init_tensor(shape, kind, fan_in), is_buf)
            self._keys.append(key)
        self._param_keys = [k for k, _ in self.named_parameters()]
        self.seed = 0
        self._step = 0
        self.flat_grad: Optional[torch.Tensor] = None    # set by enable_flat_grads()
        self._flat_views: Optional[Dict[str, torch.Tensor]] = None
        self._pack, self._pack_sig = ops.PackCache(), None
        self._weights_epoch = 0          # bumped by FusedTrainer whenever its kernels update the parameters behind PyTorch's back

    # -- plumbing ---------------------------------------------------------------------------------
    def _tensor_dict(self) -> Dict[str, torch.Tensor]:
        d = dict(self.named_parameters())
        d.update(dict(self.named_buffers()))
        return d

    def enable_flat_grads(self) -> torch.Tensor:
        """Allocate one flat fp32 gradient buffer, make every ``param.grad`` a view of it, and let the backward kernels accumulate
        straight into it (one NCCL all-reduce per step, no per-parameter copies).  Returns the flat buffer; zero it once per step."""
        params = list(self.named_parameters())
        sizes = [((p.numel() + 3) // 4) * 4 for _, p in params]      # 16-byte aligned segments
        flat = torch.zeros(sum(sizes), device=params[0][1].device)
        views, off = {}, 0
        for (k, p), n in zip(params, sizes):
            v = flat[off:off + p.numel()].view_as(p)
            p.grad = v
            views[k] = v
            off += n
        self.flat_grad, self._flat_views = flat, views
        return flat

    def _grad_targets(self):
        """(name -> tensor the kernels accumulate into, tuple returned to autograd for *params)"""
        if self._flat_views is not None:
            # ``optimizer.zero_grad()`` (set_to_none=True by default) detaches p.grad from the flat buffer: re-attach the views and give
            # the call its meaning (gradients start from zero) instead of silently accumulating into a buffer the optimiser no longer sees
            named = dict(self.named_parameters())
            if any(named[k].grad is None for k in self._param_keys):
                from .ops import call
                call("cmgan_fill", self.flat_grad, self.flat_grad.numel(), 0.0)
                for k in self._param_keys:
                    named[k].grad = self._flat_views[k]
            return self._flat_views, tuple(None for _ in self._param_keys)
        named = dict(self.named_parameters())
        G = {k: torch.zeros_like(named[k]) for k in self._param_keys}
        return G, tuple(G[k] if named[k].requires_grad else None for k in self._param_keys)

    def forward(self, x: torch.Tensor, frames=None):
        """``frames`` (optional): ragged batch for inference -- item b of the padded input holds frames[b] valid frames (host-side
        sequence or tensor of B ints, 1 <= frames[b] <= T).  Output frames t < frames[b] equal ``forward(x[b:b+1, :, :frames[b]])``; the
        rest are unspecified (the padded input frames may hold anything and are never read by a valid frame)."""
        if not x.is_cuda:
            raise RuntimeError("cmgan_b200.TSCNet runs on CUDA only (no CPU fallback)")
        if x.dtype != torch.float32:
            raise RuntimeError("cmgan_b200.TSCNet expects float32 input")
        if frames is not None:
            frames = self._ragged_frames(x, frames)
        if self.training:
            self._step += 1
            torch._foreach_add_([b for k, b in self.named_buffers() if k.endswith("num_batches_tracked")], 1)   # bookkeeping only
        params = [p for _, p in self.named_parameters()]
        if not self.training and not torch.is_grad_enabled() and ops.PACK_CACHE is None:
            # inference with frozen weights: keep the re-tiled tensor-core copies of the weights between calls; any in-place change of a
            # parameter through PyTorch (load_state_dict, an optimiser) bumps its version counter and drops the cache
            sig = (params[0].data_ptr(), sum(p._version for p in params), self._weights_epoch)
            if sig != self._pack_sig:
                self._pack.clear()
                self._pack_sig = sig
            ops.PACK_CACHE = self._pack
            try:
                return self._run(x, params, frames)
            finally:
                ops.PACK_CACHE = None
        return self._run(x, params, frames)

    def _run(self, x, params, frames):
        if frames is None:
            return _TSCNetFn.apply(x, self, self.training, self.seed * 7919 + self._step, *params)
        return tscnet_fwd(x, self._tensor_dict(), False, 0, None, frames)

    def _ragged_frames(self, x: torch.Tensor, frames) -> torch.Tensor:
        """validate host-side frame counts of a ragged batch, then upload them (device int32 (B,))"""
        if self.training or torch.is_grad_enabled():
            raise ValueError("TSCNet.forward(x, frames): ragged batches are inference only (model.eval() under torch.no_grad())")
        if ops.PRECISION == 1 and ops.ATTN_TC:
            raise ValueError("TSCNet.forward(x, frames): the tcgen05 attention forward (CMGAN_ATTN_TC=1) has no ragged-batch variant")
        B, T = x.shape[0], x.shape[2]
        n = torch.as_tensor(frames).detach().to("cpu", torch.int64).reshape(-1)
        if n.numel() != B:
            raise ValueError(f"TSCNet.forward(x, frames): expected {B} frame counts, got {n.numel()}")
        if B and (int(n.min()) < 1 or int(n.max()) > T):
            raise ValueError(f"TSCNet.forward(x, frames): frame counts must lie in [1, {T}], got [{int(n.min())}, {int(n.max())}]")
        return n.to(torch.int32).to(x.device)

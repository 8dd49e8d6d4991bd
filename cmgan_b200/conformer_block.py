"""Conformer block (macaron FFN - MHSA with Shaw relative positions - convolution module - FFN - LayerNorm) over the CUDA
kernels: forward and hand-written backward orchestration (ref: conformer.py:182-222, generator.py:92-99).

Rows are channel-last (b, t, f) x 64; a block processes either all time sequences (axis 0) or all frequency sequences
(axis 1) of the (B, T, F2) grid without ever transposing: only the attention and depthwise-convolution kernels look at
the sequence axis.  Every GEMM operand that needs a non-linearity in front of it is materialised once by the kernel that
produces it (LayerNorm output, Swish(+dropout) of the feed-forward hidden layer via the dual-output GEMM epilogue,
BatchNorm+Swish of the depthwise output), so the tensor-core GEMMs stream their A operand with plain async copies.
Helper classes for normalisation tables / statistics scratch live here too.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from . import ops
from ._lib import lib
from .ops import EPI_ACC, EPI_DBNSWISH, EPI_DROP_RES, EPI_DSWISH_DROP, EPI_SWISH_DUAL, call, gemm

C = 64          # num_channel (the kernels are specialised for 64 channels = 4 heads x 16)
CAT = 5 * C     # width of a dense-block concat buffer: [out4 | out3 | out2 | out1 | x]
FF_DROP = 0.2   # ref: generator.py:82,89
ATT_DROP = 0.2  # ref: generator.py:81,88


def _empty(*shape, dev, dtype=torch.float32):
    return torch.empty(*shape, dtype=dtype, device=dev)


def _adjacent(a: torch.Tensor, b: torch.Tensor) -> bool:
    """b starts exactly where the contiguous tensor a ends (consecutive segments of a flat parameter / gradient buffer)"""
    return a.is_contiguous() and b.is_contiguous() and b.data_ptr() == a.data_ptr() + a.numel() * a.element_size()


class _Tabs:
    """scale/shift/mean/rstd per (group, channel) and PReLU slope per channel of a normalisation site"""

    def __init__(self, G, width, dev, identity=False):
        self.scale = _empty(G, width, dev=dev)
        self.shift = _empty(G, width, dev=dev)
        self.mean = _empty(G, width, dev=dev)
        self.rstd = _empty(G, width, dev=dev)
        self.slope = _empty(width, dev=dev)
        self.width = width
        if identity:
            call("cmgan_fill", self.scale, G * width, 1.0)
            call("cmgan_fill", self.shift, G * width, 0.0)
            call("cmgan_fill", self.slope, width, 1.0)


class _Sums:
    """One zero-initialised double scratch per pass, sliced per statistics site (a single memset)."""

    def __init__(self, n, dev):
        self.buf = torch.zeros(n, dtype=torch.float64, device=dev)
        self.off = 0

    def take(self, n):
        assert self.off + n <= self.buf.numel(), "statistics scratch exhausted"
        o = self.off
        self.off += n
        return (self.buf, o)


def _inst_norm_site(x, ldx, G, rows, Cn, gamma, beta, tabs: _Tabs, c0, slope_w, sums: _Sums, frames=None, T=None):
    """InstanceNorm2d statistics (ref: generator.py:35) -> tables at channel offset c0 of ``tabs``.
    ``frames`` (ragged batch, device int32 (G,)): group g spans its first frames[g] of T frames (rows / T rows each)"""
    s = sums.take(G * Cn * 2)
    tabs_out = ((tabs.scale, c0), (tabs.shift, c0), (tabs.mean, c0), (tabs.rstd, c0), tabs.width)
    if frames is not None:
        call("cmgan_norm_stats_varlen", x, ldx, G, rows, Cn, frames, rows // T, s)
        call("cmgan_norm_finalize_varlen", s, frames, rows // T, T, G, Cn, gamma, beta, *tabs_out)
    else:
        call("cmgan_norm_stats", x, ldx, G, rows, Cn, s)
        call("cmgan_norm_finalize", s, rows, G, Cn, 0, gamma, beta, None, None, 0.0, *tabs_out)
    if slope_w is not None:
        call("cmgan_copy_rows", slope_w, Cn, (tabs.slope, c0), Cn, 1, Cn)


def _norm_bwd(x, ldx, dact, ldd, G, rows, Cn, act, batch_stats, tabs: _Tabs, c0, slope, dx, lddx, dgamma, dbeta, dslope, sums: _Sums,
              operand: bool = False):
    """``operand``: dx is read by tensor-core contractions (data + weight gradient of a convolution): rounded to tf32 on store in tf32 mode"""
    s = sums.take(G * Cn * 2)
    args = ((tabs.scale, c0), (tabs.shift, c0), (tabs.mean, c0), (tabs.rstd, c0), tabs.width, slope)
    call("cmgan_norm_bwd_reduce", x, ldx, dact, ldd, G, rows, Cn, act, *args, s, dslope)
    call("cmgan_norm_bwd_apply", x, ldx, dact, ldd, G, rows, Cn, act | (16 if operand and ops.PRECISION == 1 else 0), 1 if batch_stats else 0, *args, s,
         dx, lddx, dgamma, dbeta)


def _site_seed(seed: int, block_id: int, site: int) -> int:
    return (seed * 1000003 + block_id * 16 + site + 1) & 0xFFFFFFFFFFFFFFFF


def _rnd() -> int:
    """1 when the GEMM consumers run on the tf32 tensor cores (round materialised operands once, to nearest)"""
    return 1 if ops.PRECISION == 1 else 0


# ====================================================================================== conformer block
def conformer_fwd(x, P, p, B, T, F2, axis, training, seed, block_id, sums: _Sums, save: Optional[dict], frames=None):
    """ConformerBlock + the outer TSCB residual (ref: conformer.py:216-222, generator.py:95,97).
    x: (M, 64) rows of the (B, T, F2) grid; axis 0 = sequences along T, 1 = along F2.  Returns LN(x4) + x.
    ``frames`` (inference only, device int32 (B,)): ragged batch -- item b has frames[b] valid frames; attention and the depthwise
    convolution never read the rows of padded frames, every other operation works row by row."""
    if frames is not None and (training or save is not None):
        raise ValueError("conformer_fwd: ragged batches (frames) are inference only")
    dev = x.device
    M = x.shape[0]
    dp = FF_DROP if training else 0.0
    da = ATT_DROP if training else 0.0
    sd = [_site_seed(seed, block_id, i) for i in range(5)]
    keep = save is not None

    def layer_norm(xin, wkey, bkey):
        st = _empty(M, 2, dev=dev)
        xn = _empty(M, C, dev=dev)
        call("cmgan_ln_apply", xin, C, M, P[wkey], P[bkey], None, 0, xn, C, st, _rnd())
        return xn, st

    def ff(xin, name, s1, s2):
        """0.5 * FF(LN(x)) + x  (ref: conformer.py:54-72,136-148,211-212)"""
        if ops.PRECISION == 1 and ops.FUSED_FFN:
            # one kernel: the (M, 256) hidden activation lives in TMEM / shared memory only (csrc/ffn_fused.cu); the backward pass
            # recomputes it from the module input, so nothing but that input is kept
            W1, W2 = P[f"{p}.{name}.fn.fn.net.0.weight"], P[f"{p}.{name}.fn.fn.net.3.weight"]
            out = _empty(M, C, dev=dev)
            thr, inv = ops.drop_params(dp)
            call("cmgan_ffn_fwd", xin, C, M, P[f"{p}.{name}.fn.norm.weight"], P[f"{p}.{name}.fn.norm.bias"],
                 ops.packed_weight(W1, 0, 1, C, C, 1, 4 * C), P[f"{p}.{name}.fn.fn.net.0.bias"],
                 ops.packed_weight(W2, 0, 1, 4 * C, 4 * C, 1, C), P[f"{p}.{name}.fn.fn.net.3.bias"], 0.5,
                 s1 & 0xFFFFFFFFFFFFFFFF, s2 & 0xFFFFFFFFFFFFFFFF, thr, inv, ops.SEED_DEV, out, C)
            return (dict(fused=True) if keep else None), out
        xn, st = layer_norm(xin, f"{p}.{name}.fn.norm.weight", f"{p}.{name}.fn.norm.bias")
        h = _empty(M, 4 * C, dev=dev) if keep else None          # pre-activation: only the backward pass needs it
        a = _empty(M, 4 * C, dev=dev)                            # swish(h) * dropout: operand of the second Linear
        gemm(A=xn, lda=C, W=P[f"{p}.{name}.fn.fn.net.0.weight"], sb_k=1, sb_n=C, bias=P[f"{p}.{name}.fn.fn.net.0.bias"], C=h, ldc=4 * C, M=M,
             N=4 * C, Cin=C, epi=EPI_SWISH_DUAL, C2=a, ldc2=4 * C, seed=s1, drop_p=dp)
        out = _empty(M, C, dev=dev)
        gemm(A=a, lda=4 * C, W=P[f"{p}.{name}.fn.fn.net.3.weight"], sb_k=1, sb_n=4 * C, bias=P[f"{p}.{name}.fn.fn.net.3.bias"], C=out, ldc=C, M=M,
             N=C, Cin=4 * C, epi=EPI_DROP_RES, alpha=0.5, R=xin, ldr=C, seed=s2, drop_p=dp)
        return dict(xn=xn, st=st, h=h, a=a), out

    f1, x1 = ff(x, "ff1", sd[0], sd[1])
    # ---- attention (ref: conformer.py:90-133)
    xn2, st2 = layer_norm(x1, f"{p}.attn.norm.weight", f"{p}.attn.norm.bias")
    qkv = _empty(M, 3 * C, dev=dev)
    Wq, Wkv = P[f"{p}.attn.fn.to_q.weight"], P[f"{p}.attn.fn.to_kv.weight"]
    if _adjacent(Wq, Wkv):      # flat parameter buffer: [Wq; Wkv] is one (192, 64) matrix -> one projection instead of two
        gemm(A=xn2, lda=C, W=Wq, sb_k=1, sb_n=C, C=qkv, ldc=3 * C, M=M, N=3 * C, Cin=C)
    else:
        gemm(A=xn2, lda=C, W=Wq, sb_k=1, sb_n=C, C=qkv, ldc=3 * C, M=M, N=C, Cin=C)
        gemm(A=xn2, lda=C, W=Wkv, sb_k=1, sb_n=C, C=(qkv, C), ldc=3 * C, M=M, N=2 * C, Cin=C)
    ctx = _empty(M, C, dev=dev)
    lse = _empty(M, 4, dev=dev)
    if frames is not None:
        if ops.PRECISION == 1 and ops.ATTN_TC:
            raise ValueError("the tcgen05 attention forward (CMGAN_ATTN_TC=1) has no ragged-batch variant; unset it to pass frames")
        call("cmgan_attention_fwd_tf32_varlen" if ops.PRECISION == 1 else "cmgan_attention_fwd_varlen", qkv, P[f"{p}.attn.fn.rel_pos_emb.weight"],
             B, T, F2, axis, frames, ctx, lse)
    else:
        call(("cmgan_attention_fwd_tc" if ops.ATTN_TC else "cmgan_attention_fwd_tf32") if ops.PRECISION == 1 else "cmgan_attention_fwd", qkv, P[f"{p}.attn.fn.rel_pos_emb.weight"], B, T, F2, axis,
             ctx, lse)
    x2 = _empty(M, C, dev=dev)
    gemm(A=ctx, lda=C, W=P[f"{p}.attn.fn.to_out.weight"], sb_k=1, sb_n=C, bias=P[f"{p}.attn.fn.to_out.bias"], C=x2, ldc=C, M=M, N=C, Cin=C,
         epi=EPI_DROP_RES, alpha=1.0, R=x1, ldr=C, seed=sd[2], drop_p=da)
    # ---- convolution module (ref: conformer.py:160-173)
    xn3, st3 = layer_norm(x2, f"{p}.conv.net.0.weight", f"{p}.conv.net.0.bias")
    g = _empty(M, 4 * C, dev=dev)
    gemm(A=xn3, lda=C, W=P[f"{p}.conv.net.2.weight"], sb_k=1, sb_n=C, bias=P[f"{p}.conv.net.2.bias"], C=g, ldc=4 * C, M=M, N=4 * C, Cin=C)
    d = _empty(M, 2 * C, dev=dev)
    # training: the BatchNorm batch statistics (sum, sum of squares per channel) come out of the depthwise kernel's epilogue
    s = sums.take(2 * C * 2) if training else None
    if frames is not None:
        call("cmgan_glu_dwconv_fwd_varlen", g, P[f"{p}.conv.net.4.conv.weight"], P[f"{p}.conv.net.4.conv.bias"], B, T, F2, axis, frames, d)
    else:
        call("cmgan_glu_dwconv_fwd", g, P[f"{p}.conv.net.4.conv.weight"], P[f"{p}.conv.net.4.conv.bias"], B, T, F2, axis, d, s)
    bn = _Tabs(1, 2 * C, dev)
    bnp = (P[f"{p}.conv.net.5.weight"], P[f"{p}.conv.net.5.bias"], P[f"{p}.conv.net.5.running_mean"], P[f"{p}.conv.net.5.running_var"])
    if training:
        call("cmgan_norm_finalize", s, M, 1, 2 * C, 0, *bnp, 0.1, bn.scale, bn.shift, bn.mean, bn.rstd, 2 * C)
    else:
        call("cmgan_norm_finalize", None, M, 1, 2 * C, 1, *bnp, 0.1, bn.scale, bn.shift, bn.mean, bn.rstd, 2 * C)
    dsw = _empty(M, 2 * C, dev=dev)           # swish(bn(d)): operand of the second pointwise conv
    call("cmgan_norm_apply", d, 2 * C, 1, M, 2 * C, 2 | (16 * _rnd()), bn.scale, bn.shift, 2 * C, None, dsw, 2 * C)
    x3 = _empty(M, C, dev=dev)
    gemm(A=dsw, lda=2 * C, W=P[f"{p}.conv.net.7.weight"], sb_k=1, sb_n=2 * C, bias=P[f"{p}.conv.net.7.bias"], C=x3, ldc=C, M=M, N=C, Cin=2 * C,
         epi=EPI_DROP_RES, alpha=1.0, R=x2, ldr=C)
    # ---- second feed-forward, post norm, outer residual
    f2, x4 = ff(x3, "ff2", sd[3], sd[4])
    st5 = _empty(M, 2, dev=dev)
    y = _empty(M, C, dev=dev)
    call("cmgan_ln_apply", x4, C, M, P[f"{p}.post_norm.weight"], P[f"{p}.post_norm.bias"], x, C, y, C, st5, 0)
    if save is not None:
        save.update(x=x, f1=f1, x1=x1, xn2=xn2, st2=st2, qkv=qkv, ctx=ctx, lse=lse, x2=x2, xn3=xn3, st3=st3, g=g, d=d, dsw=dsw, bn=bn, x3=x3,
                    f2=f2, x4=x4, st5=st5, sd=sd, dp=dp, da=da, axis=axis, training=training, p=p)
    return y


def conformer_bwd(dy, S: dict, P, G: Dict[str, torch.Tensor], B, T, F2, sums: _Sums):
    """Gradient of conformer_fwd: dy (M, 64) -> dx (M, 64); parameter gradients accumulate into G[name]."""
    dev = dy.device
    M = dy.shape[0]
    p, axis, dp, da, sd = S["p"], S["axis"], S["dp"], S["da"], S["sd"]

    def ln_bwd(dyv, xv, st, name, res, res2, zalpha=None, zseed=0, zp=0.0):
        """LayerNorm backward (+ residual gradients); with ``zalpha`` also the dropout-scaled copy that enters the next residual
        branch (dz = zalpha * mask(zseed) * dx), so that branch's GEMMs read a plain operand"""
        dxv = _empty(M, C, dev=dev)
        args = (dyv, C, xv, C, st, P[f"{name}.weight"], M, res, C if res is not None else 0, res2, C if res2 is not None else 0, dxv, C,
                G[f"{name}.weight"], G[f"{name}.bias"])
        if zalpha is None:
            call("cmgan_ln_bwd", *args)
            return dxv, None
        dzv = _empty(M, C, dev=dev)
        thr, inv = ops.drop_params(zp)
        call("cmgan_ln_bwd_drop", *args, dzv, C, float(zalpha), zseed & 0xFFFFFFFFFFFFFFFF, thr, inv, ops.SEED_DEV)
        return dxv, dzv

    def ff_bwd(dout, dz, xin, f, name, s1, res2=None, **znext):
        # out = xin + 0.5 * drop2(W2 a + b2),  a = swish(h) * drop1,  h = W1 LN(xin) + b1;   dz = 0.5 * drop2-mask * dout
        W1, W2 = P[f"{p}.{name}.fn.fn.net.0.weight"], P[f"{p}.{name}.fn.fn.net.3.weight"]
        if f.get("fused"):
            # one kernel for the data gradients (hidden activation recomputed, LayerNorm backward in its epilogue); it leaves the operands
            # of the two weight-gradient GEMMs behind: a = swish(h) * drop, dh, xn
            a, dh, xn, dxv = _empty(M, 4 * C, dev=dev), _empty(M, 4 * C, dev=dev), _empty(M, C, dev=dev), _empty(M, C, dev=dev)
            thr, inv = ops.drop_params(dp)
            call("cmgan_ffn_bwd", xin, C, dz, C, dout, C, res2, C if res2 is not None else 0, M, P[f"{p}.{name}.fn.norm.weight"],
                 P[f"{p}.{name}.fn.norm.bias"], ops.packed_weight(W1, 0, 1, C, C, 1, 4 * C), P[f"{p}.{name}.fn.fn.net.0.bias"],
                 ops.packed_weight(W2, 0, 4 * C, 1, C, 1, 4 * C), ops.packed_weight(W1, 0, C, 1, 4 * C, 1, C), s1 & 0xFFFFFFFFFFFFFFFF, thr, inv,
                 ops.SEED_DEV, dxv, C, a, dh, xn, G[f"{p}.{name}.fn.norm.weight"], G[f"{p}.{name}.fn.norm.bias"])
            gemm(wgrad=True, A=a, lda=4 * C, Cin=4 * C, D=dz, ldd=C, N=C, W=None, C=G[f"{p}.{name}.fn.fn.net.3.weight"], sb_k=1, sb_n=4 * C, ldc=0,
                 M=M, dbias=G[f"{p}.{name}.fn.fn.net.3.bias"])
            gemm(wgrad=True, A=xn, lda=C, Cin=C, D=dh, ldd=4 * C, N=4 * C, W=None, C=G[f"{p}.{name}.fn.fn.net.0.weight"], sb_k=1, sb_n=C, ldc=0, M=M,
                 dbias=G[f"{p}.{name}.fn.fn.net.0.bias"])
            return dxv, None
        dh = _empty(M, 4 * C, dev=dev)
        gemm(A=dz, lda=C, W=W2, sb_k=4 * C, sb_n=1, C=dh, ldc=4 * C, M=M, N=4 * C, Cin=C, epi=EPI_DSWISH_DROP, aux=f["h"], ldaux=4 * C, seed=s1,
             drop_p=dp)
        gemm(wgrad=True, A=f["a"], lda=4 * C, Cin=4 * C, D=dz, ldd=C, N=C, W=None, C=G[f"{p}.{name}.fn.fn.net.3.weight"], sb_k=1, sb_n=4 * C,
             ldc=0, M=M, dbias=G[f"{p}.{name}.fn.fn.net.3.bias"])
        dln = _empty(M, C, dev=dev)
        gemm(A=dh, lda=4 * C, W=W1, sb_k=C, sb_n=1, C=dln, ldc=C, M=M, N=C, Cin=4 * C)
        gemm(wgrad=True, A=f["xn"], lda=C, Cin=C, D=dh, ldd=4 * C, N=4 * C, W=None, C=G[f"{p}.{name}.fn.fn.net.0.weight"], sb_k=1, sb_n=C, ldc=0,
             M=M, dbias=G[f"{p}.{name}.fn.fn.net.0.bias"])
        return ln_bwd(dln, xin, f["st"], f"{p}.{name}.fn.norm", dout, res2, **znext)

    # y = LN(x4) * g + b + x
    dx4, dz4 = ln_bwd(dy, S["x4"], S["st5"], f"{p}.post_norm", None, None, zalpha=0.5, zseed=sd[4], zp=dp)
    dx3, _ = ff_bwd(dx4, dz4, S["x3"], S["f2"], "ff2", sd[3])
    # ---- convolution module: x3 = x2 + W7 swish(bn(d)) + b7
    bn = S["bn"]
    dbn = _empty(M, 2 * C, dev=dev)
    gemm(A=dx3, lda=C, W=P[f"{p}.conv.net.7.weight"], sb_k=2 * C, sb_n=1, C=dbn, ldc=2 * C, M=M, N=2 * C, Cin=C, epi=EPI_DBNSWISH, aux=S["d"],
         ldaux=2 * C, e0=bn.scale, e1=bn.shift)
    gemm(wgrad=True, A=S["dsw"], lda=2 * C, Cin=2 * C, D=dx3, ldd=C, N=C, W=None, C=G[f"{p}.conv.net.7.weight"], sb_k=1, sb_n=2 * C, ldc=0, M=M,
         dbias=G[f"{p}.conv.net.7.bias"])
    dd = _empty(M, 2 * C, dev=dev)
    _norm_bwd(S["d"], 2 * C, dbn, 2 * C, 1, M, 2 * C, 0, S["training"], bn, 0, None, dd, 2 * C, G[f"{p}.conv.net.5.weight"],
              G[f"{p}.conv.net.5.bias"], None, sums)
    dg = _empty(M, 4 * C, dev=dev)
    call("cmgan_glu_dwconv_bwd", S["g"], dd, P[f"{p}.conv.net.4.conv.weight"], B, T, F2, axis, dg, G[f"{p}.conv.net.4.conv.weight"],
         G[f"{p}.conv.net.4.conv.bias"])
    dln3 = _empty(M, C, dev=dev)
    gemm(A=dg, lda=4 * C, W=P[f"{p}.conv.net.2.weight"], sb_k=C, sb_n=1, C=dln3, ldc=C, M=M, N=C, Cin=4 * C)
    gemm(wgrad=True, A=S["xn3"], lda=C, Cin=C, D=dg, ldd=4 * C, N=4 * C, W=None, C=G[f"{p}.conv.net.2.weight"], sb_k=1, sb_n=C, ldc=0, M=M,
         dbias=G[f"{p}.conv.net.2.bias"])
    dx2, dz2 = ln_bwd(dln3, S["x2"], S["st3"], f"{p}.conv.net.0", dx3, None, zalpha=1.0 if da > 0.0 else None, zseed=sd[2], zp=da)
    if dz2 is None:
        dz2 = dx2
    # ---- attention: x2 = x1 + drop(ctx Wo^T + bo);  dz2 = drop-mask * dx2
    dctx = _empty(M, C, dev=dev)
    gemm(A=dz2, lda=C, W=P[f"{p}.attn.fn.to_out.weight"], sb_k=C, sb_n=1, C=dctx, ldc=C, M=M, N=C, Cin=C)
    gemm(wgrad=True, A=S["ctx"], lda=C, Cin=C, D=dz2, ldd=C, N=C, W=None, C=G[f"{p}.attn.fn.to_out.weight"], sb_k=1, sb_n=C, ldc=0, M=M,
         dbias=G[f"{p}.attn.fn.to_out.bias"])
    dqkv = _empty(M, 3 * C, dev=dev)
    delta = _empty(M, 4, dev=dev)
    attn_args = (S["qkv"], P[f"{p}.attn.fn.rel_pos_emb.weight"], S["ctx"], dctx, S["lse"], B, T, F2, axis, delta, dqkv, G[f"{p}.attn.fn.rel_pos_emb.weight"])
    if ops.PRECISION == 1:
        ws, nws = None, 0
        if ops.ATTN_BWD_WS:         # block-private dE accumulators in global memory: the dq kernel runs 3 blocks / SM instead of 2
            nws = lib().cdll.cmgan_attention_bwd_ws_floats(B, T, F2, axis)
            ws = _empty(max(nws, 1), dev=dev)
        if ops.AUX_STREAM is not None and ops.PROBE is None:
            # delta first; then the dq / dE kernel and the dk / dv kernel side by side (each alone leaves most of every SM idle)
            call("cmgan_attention_bwd_tf32_ws", *attn_args, 1, None, 0)
            ops.call_on(ops.AUX_STREAM, "cmgan_attention_bwd_tf32_ws", *attn_args, 4, None, 0)
            call("cmgan_attention_bwd_tf32_ws", *attn_args, 2, ws, nws)
            ops.join(ops.AUX_STREAM)
        else:
            call("cmgan_attention_bwd_tf32_ws", *attn_args, 7, ws, nws)
    else:
        call("cmgan_attention_bwd", *attn_args)
    dln2 = _empty(M, C, dev=dev)
    Wq, Wkv = P[f"{p}.attn.fn.to_q.weight"], P[f"{p}.attn.fn.to_kv.weight"]
    Gq, Gkv = G[f"{p}.attn.fn.to_q.weight"], G[f"{p}.attn.fn.to_kv.weight"]
    if _adjacent(Wq, Wkv) and _adjacent(Gq, Gkv):      # merged (192, 64) projection (see conformer_fwd)
        gemm(A=dqkv, lda=3 * C, W=Wq, sb_k=C, sb_n=1, C=dln2, ldc=C, M=M, N=C, Cin=3 * C)
        gemm(wgrad=True, A=S["xn2"], lda=C, Cin=C, D=dqkv, ldd=3 * C, N=3 * C, W=None, C=Gq, sb_k=1, sb_n=C, ldc=0, M=M)
    else:
        gemm(A=dqkv, lda=3 * C, W=Wq, sb_k=C, sb_n=1, C=dln2, ldc=C, M=M, N=C, Cin=C)
        gemm(A=(dqkv, C), lda=3 * C, W=Wkv, sb_k=C, sb_n=1, C=dln2, ldc=C, M=M, N=C, Cin=2 * C, epi=EPI_ACC, alpha=1.0)
        gemm(wgrad=True, A=S["xn2"], lda=C, Cin=C, D=dqkv, ldd=3 * C, N=C, W=None, C=Gq, sb_k=1, sb_n=C, ldc=0, M=M)
        gemm(wgrad=True, A=S["xn2"], lda=C, Cin=C, D=(dqkv, C), ldd=3 * C, N=2 * C, W=None, C=Gkv, sb_k=1, sb_n=C, ldc=0, M=M)
    dx1, dz1 = ln_bwd(dln2, S["x1"], S["st2"], f"{p}.attn.norm", dx2, None, zalpha=0.5, zseed=sd[1], zp=dp)
    # ---- first feed-forward; the outer residual adds dy
    return ff_bwd(dx1, dz1, S["x"], S["f1"], "ff1", sd[0], res2=dy)[0]

"""TSCNet forward / backward orchestration over the CUDA kernels (ref: generator.py:6-196).

Data layout: every activation is channel-last rows (b, t, f) x channels.  A DilatedDenseNet works in one (M, 320) concat
buffer ``cat`` = [out4 | out3 | out2 | out1 | x] holding *activated* values (InstanceNorm + PReLU already applied, rounded to
tf32 when the tensor-core path consumes them), so that layer i's implicit-GEMM convolution reads channels [(5-i)*64, 320)
with plain 16-byte async copies and writes its raw output to a separate (M, 64) buffer (kept for the InstanceNorm backward).
The reference's pad / cat / permute / contiguous copies do not exist here.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from . import ops
from .conformer_block import C, CAT, _Sums, _Tabs, _empty, _inst_norm_site, _norm_bwd, conformer_bwd, conformer_fwd
from .ops import EPI_ACC, EPI_NONE, call, gemm

_W3 = [(0, -1), (0, 0), (0, 1)]
_W3T = [(0, 1), (0, 0), (0, -1)]


def _dense_taps(dil):
    return [((kh - 1) * dil, kw - 1) for kh in range(2) for kw in range(3)]     # tap = kh*3 + kw  (ref: generator.py:12-13,17,21)


def _act_code():
    return 1 | (16 if ops.PRECISION == 1 else 0)       # PReLU (+ round to tf32 for the tensor-core consumers)


def _norm_prelu_to(raw, ldr, G, rows, gamma, beta, slope, dst, ldd, sums: _Sums, dev, frames=None, T=None) -> _Tabs:
    """InstanceNorm2d(affine) + PReLU of a raw (M, 64) tensor, materialised into ``dst`` (ref: generator.py:35-37)"""
    tab = _Tabs(G, C, dev)
    _inst_norm_site(raw, ldr, G, rows, C, gamma, beta, tab, 0, None, sums, frames, T)
    call("cmgan_norm_apply", raw, ldr, G, rows, C, _act_code(), tab.scale, tab.shift, C, slope, dst, ldd)
    return tab


def dense_block_fwd(cat, P, p, B, T, Fw, sums: _Sums, frames=None):
    """DilatedDenseNet (ref: generator.py:39-47).  ``cat`` slot 4 holds the (activated) block input; returns the per-layer raw
    conv outputs and normalisation tables.  Layer i leaves act(out_i) in slot 4 - i.  The convolutions are causal in time, so with
    ``frames`` (ragged batch) only the InstanceNorm statistics need to know the lengths."""
    dev = cat.device
    M, rows = B * T * Fw, T * Fw
    raws, tabs = [], []
    for i in range(1, 5):
        dil, c0, Cin, co = 2 ** (i - 1), (5 - i) * C, C * i, (4 - i) * C
        raw = _empty(M, C, dev=dev)
        gemm(A=(cat, c0), lda=CAT, W=P[f"{p}.conv{i}.weight"], sb_tap=1, sb_k=6, sb_n=Cin * 6, bias=P[f"{p}.conv{i}.bias"], C=raw, ldc=C,
             M=M, N=C, Cin=Cin, taps=_dense_taps(dil), conv=dict(OH=T, OW=Fw, IH=T, IW=Fw))
        tabs.append(_norm_prelu_to(raw, C, B, rows, P[f"{p}.norm{i}.weight"], P[f"{p}.norm{i}.bias"], P[f"{p}.prelu{i}.weight"], (cat, co), CAT,
                                   sums, dev, frames, T))
        raws.append(raw)
    return raws, tabs


def dense_block_bwd(cat, raws, tabs, dcat, P, G, p, B, T, Fw, sums: _Sums):
    """dcat slot 0 holds the gradient wrt act(out4); on return dcat slot 4 holds the gradient wrt the block input."""
    dev = cat.device
    M, rows = B * T * Fw, T * Fw
    for i in range(4, 0, -1):
        dil, c0, Cin, co = 2 ** (i - 1), (5 - i) * C, C * i, (4 - i) * C
        draw = _empty(M, C, dev=dev)        # one per layer: the weight-gradient GEMM may still be reading it on the side stream
        _norm_bwd(raws[i - 1], C, (dcat, co), CAT, B, rows, C, 1, True, tabs[i - 1], 0, P[f"{p}.prelu{i}.weight"], draw, C,
                  G[f"{p}.norm{i}.weight"], G[f"{p}.norm{i}.bias"], G[f"{p}.prelu{i}.weight"], sums, operand=True)
        taps = _dense_taps(dil)
        gemm(wgrad=True, A=(cat, c0), lda=CAT, Cin=Cin, taps=taps, conv=dict(OH=T, OW=Fw, IH=T, IW=Fw), D=draw, ldd=C, N=C, W=None,
             C=G[f"{p}.conv{i}.weight"], sb_tap=1, sb_k=6, sb_n=Cin * 6, ldc=0, M=M, dbias=G[f"{p}.conv{i}.bias"])
        gemm(A=draw, lda=C, W=P[f"{p}.conv{i}.weight"], sb_tap=1, sb_k=Cin * 6, sb_n=6, C=(dcat, c0), ldc=CAT, M=M, N=Cin, Cin=C,
             taps=[(-dy, -dx) for dy, dx in taps], conv=dict(OH=T, OW=Fw, IH=T, IW=Fw), epi=EPI_NONE if i == 4 else EPI_ACC, alpha=1.0)


def _sums_size(B):
    return (16 * C + 2) * B * 2 + 8 * 2 * C * 2 + 64


def tscnet_fwd(x, P, training: bool, seed: int, save: Optional[dict], frames=None):
    """TSCNet.forward (ref: generator.py:174-196).  x (B, 2, T, F) any strides -> final_real, final_imag (B, 1, T, F).
    ``frames`` (inference only): ragged batch, device int32 (B,) with 1 <= frames[b] <= T.  For t < frames[b] the outputs equal this
    function on x[b:b+1, :, :frames[b]] alone; the rows of padded frames are never read by a valid row and their outputs are unspecified."""
    if frames is not None and (training or save is not None):
        raise ValueError("tscnet_fwd: ragged batches (frames) are inference only")
    dev = x.device
    B, two, T, F = x.shape
    assert two == 2 and F % 2 == 1, "expected x of shape (B, 2, T, F) with odd F"
    F2 = (F - 1) // 2 + 1
    M, M2 = B * T * F, B * T * F2
    xs = x.stride()
    sums = _Sums(_sums_size(B), dev)
    # ---- dense encoder (ref: generator.py:50-69)
    pe = "dense_encoder"
    catE = _empty(M, CAT, dev=dev)
    raw0 = _empty(M, C, dev=dev)
    call("cmgan_head_conv", x, xs[0], xs[1], xs[2], xs[3], B, T, F, P[pe + ".conv_1.0.weight"], P[pe + ".conv_1.0.bias"], raw0, C)
    tab0 = _norm_prelu_to(raw0, C, B, T * F, P[pe + ".conv_1.1.weight"], P[pe + ".conv_1.1.bias"], P[pe + ".conv_1.2.weight"], (catE, 4 * C), CAT,
                          sums, dev, frames, T)
    rawsE, tabsE = dense_block_fwd(catE, P, pe + ".dilated_dense", B, T, F, sums, frames)
    e2 = _empty(M2, C, dev=dev)
    gemm(A=catE, lda=CAT, W=P[pe + ".conv_2.0.weight"], sb_tap=1, sb_k=3, sb_n=3 * C, bias=P[pe + ".conv_2.0.bias"], C=e2, ldc=C, M=M2, N=C, Cin=C,
         taps=_W3, conv=dict(OH=T, OW=F2, IH=T, IW=F, mul_x=2))
    h = _empty(M2, C, dev=dev)
    tab2 = _Tabs(B, C, dev)
    _inst_norm_site(e2, C, B, T * F2, C, P[pe + ".conv_2.1.weight"], P[pe + ".conv_2.1.bias"], tab2, 0, None, sums, frames, T)
    call("cmgan_norm_apply", e2, C, B, T * F2, C, 1, tab2.scale, tab2.shift, C, P[pe + ".conv_2.2.weight"], h, C)
    # ---- 4 x TSCB (ref: generator.py:92-99)
    conf_saves = []
    for i in range(1, 5):
        for axis, name in ((0, "time_conformer"), (1, "freq_conformer")):
            sv = {} if save is not None else None
            h = conformer_fwd(h, P, f"TSCB_{i}.{name}", B, T, F2, axis, training, seed, (i - 1) * 2 + axis, sums, sv, frames)
            conf_saves.append(sv)
    # ---- decoders (ref: generator.py:122-156)
    dec = {}
    for pd in ("mask_decoder", "complex_decoder"):
        cat = _empty(M2, CAT, dev=dev)
        call("cmgan_copy_rows_operand", h, C, (cat, 4 * C), CAT, M2, C)         # operand of the decoder's first convolution
        raws, tabs = dense_block_fwd(cat, P, pd + ".dense_block", B, T, F2, sums, frames)
        sp = _empty(M2, 2 * C, dev=dev)      # == (B, T, 2*F2, 64): the sub-pixel shuffle is a free reinterpretation
        gemm(A=cat, lda=CAT, W=P[pd + ".sub_pixel.conv.weight"], sb_tap=1, sb_k=3, sb_n=3 * C, bias=P[pd + ".sub_pixel.conv.bias"], C=sp, ldc=2 * C,
             M=M2, N=2 * C, Cin=C, taps=_W3, conv=dict(OH=T, OW=F2, IH=T, IW=F2))
        dec[pd] = dict(cat=cat, raws=raws, tabs=tabs, sp=sp)
    pm, pc = "mask_decoder", "complex_decoder"
    m1 = _empty(M, dev=dev)
    call("cmgan_rowdot_fwd", dec[pm]["sp"], B, T, F, 1, None, None, None, P[pm + ".conv_1.weight"], P[pm + ".conv_1.bias"], m1)
    tabM = _Tabs(B, 1, dev)
    _inst_norm_site(m1, 1, B, T * F, 1, P[pm + ".norm.weight"], P[pm + ".norm.bias"], tabM, 0, None, sums, frames, T)
    tabC = _Tabs(B, C, dev)
    _inst_norm_site(dec[pc]["sp"], C, B, T * 2 * F2, C, P[pc + ".norm.weight"], P[pc + ".norm.bias"], tabC, 0, None, sums, frames, T)
    cplx = _empty(M, 2, dev=dev)
    call("cmgan_rowdot_fwd", dec[pc]["sp"], B, T, F, 2, tabC.scale, tabC.shift, P[pc + ".prelu.weight"], P[pc + ".conv.weight"],
         P[pc + ".conv.bias"], cplx)
    fr = _empty(B, 1, T, F, dev=dev)
    fi = _empty(B, 1, T, F, dev=dev)
    call("cmgan_recombine", m1, tabM.scale, tabM.shift, P[pm + ".prelu.weight"], P[pm + ".final_conv.weight"], P[pm + ".final_conv.bias"],
         P[pm + ".prelu_out.weight"], x, xs[0], xs[1], xs[2], xs[3], cplx, B, T, F, fr, fi)
    if save is not None:
        save.update(x=x, B=B, T=T, F=F, F2=F2, catE=catE, raw0=raw0, tab0=tab0, rawsE=rawsE, tabsE=tabsE, e2=e2, tab2=tab2, conf=conf_saves,
                    dec=dec, m1=m1, tabM=tabM, tabC=tabC)
    return fr, fi


def tscnet_bwd(S: dict, dfr, dfi, P, G: Dict[str, torch.Tensor], after_tscb=None):
    """Backward of tscnet_fwd.  dfr / dfi: gradients wrt final_real / final_imag ((B,1,T,F), any strides, or None).
    Parameter gradients are accumulated (+=) into the tensors of G.  ``after_tscb`` (optional callable) runs once the decoders'
    and the TSCB stack's gradients are complete (the trainer starts their all-reduce there, under the encoder's backward)."""
    x = S["x"]
    dev = x.device
    B, T, F, F2 = S["B"], S["T"], S["F"], S["F2"]
    M, M2 = B * T * F, B * T * F2
    xs = x.stride()
    sums = _Sums(_sums_size(B), dev)
    if dfr is None:
        dfr = torch.zeros(B, 1, T, F, device=dev)
    if dfi is None:
        dfi = torch.zeros(B, 1, T, F, device=dev)
    if dfi.stride() != dfr.stride():
        dfi = dfi.contiguous()
        dfr = dfr.contiguous()
    gs = dfr.stride()
    pm, pc = "mask_decoder", "complex_decoder"
    dec, tabM, tabC = S["dec"], S["tabM"], S["tabC"]
    dcplx = _empty(M, 2, dev=dev)
    dz = _empty(M, dev=dev)
    call("cmgan_recombine_bwd", S["m1"], tabM.scale, tabM.shift, P[pm + ".prelu.weight"], P[pm + ".final_conv.weight"], P[pm + ".final_conv.bias"],
         P[pm + ".prelu_out.weight"], x, xs[0], xs[1], xs[2], xs[3], dfr, dfi, gs[0], gs[2], gs[3], B, T, F, dcplx, dz, G[pm + ".prelu_out.weight"],
         G[pm + ".final_conv.weight"], G[pm + ".final_conv.bias"])
    dm1 = _empty(M, dev=dev)
    _norm_bwd(S["m1"], 1, dz, 1, B, T * F, 1, 1, True, tabM, 0, P[pm + ".prelu.weight"], dm1, 1, G[pm + ".norm.weight"], G[pm + ".norm.bias"],
              G[pm + ".prelu.weight"], sums)
    dsp = {}
    dsp[pm] = _empty(M2, 2 * C, dev=dev)
    call("cmgan_rowdot_bwd", dec[pm]["sp"], B, T, F, 1, None, None, None, P[pm + ".conv_1.weight"], dm1, dsp[pm], G[pm + ".conv_1.weight"],
         G[pm + ".conv_1.bias"])
    call("cmgan_copy_rows_operand", dsp[pm], 2 * C, dsp[pm], 2 * C, M2, 2 * C)      # operand of the sub-pixel convolution's gradient GEMMs
    dactc = _empty(M2, 2 * C, dev=dev)
    call("cmgan_rowdot_bwd", dec[pc]["sp"], B, T, F, 2, tabC.scale, tabC.shift, P[pc + ".prelu.weight"], P[pc + ".conv.weight"], dcplx, dactc,
         G[pc + ".conv.weight"], G[pc + ".conv.bias"])
    dsp[pc] = _empty(M2, 2 * C, dev=dev)
    _norm_bwd(dec[pc]["sp"], C, dactc, C, B, T * 2 * F2, C, 1, True, tabC, 0, P[pc + ".prelu.weight"], dsp[pc], C, G[pc + ".norm.weight"],
              G[pc + ".norm.bias"], G[pc + ".prelu.weight"], sums, operand=True)
    dh = None
    for pd in (pm, pc):
        cat = dec[pd]["cat"]
        dcat = _empty(M2, CAT, dev=dev)
        gemm(wgrad=True, A=cat, lda=CAT, Cin=C, taps=_W3, conv=dict(OH=T, OW=F2, IH=T, IW=F2), D=dsp[pd], ldd=2 * C, N=2 * C, W=None,
             C=G[pd + ".sub_pixel.conv.weight"], sb_tap=1, sb_k=3, sb_n=3 * C, ldc=0, M=M2, dbias=G[pd + ".sub_pixel.conv.bias"])
        gemm(A=dsp[pd], lda=2 * C, W=P[pd + ".sub_pixel.conv.weight"], sb_tap=1, sb_k=3 * C, sb_n=3, C=dcat, ldc=CAT, M=M2, N=C, Cin=2 * C,
             taps=_W3T, conv=dict(OH=T, OW=F2, IH=T, IW=F2))
        dense_block_bwd(cat, dec[pd]["raws"], dec[pd]["tabs"], dcat, P, G, pd + ".dense_block", B, T, F2, sums)
        if dh is None:
            dh = _empty(M2, C, dev=dev)
            call("cmgan_copy_rows", (dcat, 4 * C), CAT, dh, C, M2, C)
        else:
            call("cmgan_add_rows", (dcat, 4 * C), CAT, dh, C, M2, C)
    # ---- TSCBs in reverse
    k = 7
    for i in range(4, 0, -1):
        for axis in (1, 0):
            dh = conformer_bwd(dh, S["conf"][k], P, G, B, T, F2, sums)
            k -= 1
    if after_tscb is not None:
        after_tscb()
    # ---- encoder
    pe = "dense_encoder"
    catE, tab2 = S["catE"], S["tab2"]
    de2 = _empty(M2, C, dev=dev)
    _norm_bwd(S["e2"], C, dh, C, B, T * F2, C, 1, True, tab2, 0, P[pe + ".conv_2.2.weight"], de2, C, G[pe + ".conv_2.1.weight"],
              G[pe + ".conv_2.1.bias"], G[pe + ".conv_2.2.weight"], sums, operand=True)
    gemm(wgrad=True, A=catE, lda=CAT, Cin=C, taps=_W3, conv=dict(OH=T, OW=F2, IH=T, IW=F, mul_x=2), D=de2, ldd=C, N=C, W=None,
         C=G[pe + ".conv_2.0.weight"], sb_tap=1, sb_k=3, sb_n=3 * C, ldc=0, M=M2, dbias=G[pe + ".conv_2.0.bias"])
    dcatE = _empty(M, CAT, dev=dev)
    gemm(A=de2, lda=C, W=P[pe + ".conv_2.0.weight"], sb_tap=1, sb_k=3 * C, sb_n=3, C=dcatE, ldc=CAT, M=M, N=C, Cin=C, taps=_W3T,
         conv=dict(OH=T, OW=F, IH=T, IW=F2, div_x=2))
    dense_block_bwd(catE, S["rawsE"], S["tabsE"], dcatE, P, G, pe + ".dilated_dense", B, T, F, sums)
    draw1 = _empty(M, C, dev=dev)
    _norm_bwd(S["raw0"], C, (dcatE, 4 * C), CAT, B, T * F, C, 1, True, S["tab0"], 0, P[pe + ".conv_1.2.weight"], draw1, C,
              G[pe + ".conv_1.1.weight"], G[pe + ".conv_1.1.bias"], G[pe + ".conv_1.2.weight"], sums)
    call("cmgan_head_conv_wgrad", x, xs[0], xs[1], xs[2], xs[3], B, T, F, draw1, C, G[pe + ".conv_1.0.weight"], G[pe + ".conv_1.0.bias"])
    ops.join_wgrad()        # weight-gradient GEMMs launched on the side stream (ops.WGRAD_STREAM) are complete from here on

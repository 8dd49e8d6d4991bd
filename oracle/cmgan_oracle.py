"""CPU oracle for the CMGAN hot path -- TEST INFRASTRUCTURE ONLY.

This file is a functional, stateless restatement (torch CPU fp32/fp64 tensor math,
no nn.Module, weights passed as a flat ``state_dict``-style mapping) of the
reference's per-step path

    waveform -> RMS normalise -> STFT -> power_compress -> TSCNet -> power_uncompress
             -> iSTFT (+ the metric Discriminator and the generator/discriminator losses)

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline /
``--impl reference`` legs may import it, and only as the *checker* (or the thing
timed as the CPU baseline); the product package ``cmgan_b200`` never imports it.

Parity status: **pinned**.  ``tests/test_oracle_vs_reference.py`` checks the
generator, the power compression and the train-mode discriminator against outputs
the reference's own modules computed on the shipped checkpoint
(``tools/make_golden_oracle_pins.py``); ``tools/make_golden.py`` (committed) wrote the fixtures under
``tests/golden/`` from the *reference* modules, and ``tests/test_oracle_golden.py``
checks this oracle against those fixtures everywhere (GPU box included, where
``/root/reference`` does not exist).  The one unpinned quantity is PESQ (the ``pesq``
package is third-party C code that is not vendored and not installed): see DESIGN.md.

Every function cites the reference lines it follows as ``ref: file:line``.
Layouts are the reference's (NCHW) so that the citations are easy to check.
"""
from __future__ import annotations

import math
from typing import Dict, Mapping, Optional, Tuple

import torch
import torch.nn.functional as F

Tensor = torch.Tensor
SD = Mapping[str, Tensor]

N_FFT = 400
HOP = 100


# --------------------------------------------------------------------------- signal front/back end
def hamming_window(n: int = N_FFT, dtype=torch.float32) -> Tensor:
    """Periodic Hamming window, torch.hamming_window default (ref: train.py:84)."""
    k = torch.arange(n, dtype=torch.float64)
    return (0.54 - 0.46 * torch.cos(2.0 * math.pi * k / n)).to(dtype)


def rms_scale(noisy: Tensor) -> Tensor:
    """c = sqrt(L / sum(x^2)) per utterance (ref: train.py:75, evaluation.py:21)."""
    return torch.sqrt(noisy.size(-1) / torch.sum(noisy ** 2.0, dim=-1))


def stft(x: Tensor) -> Tensor:
    """(B, L) -> (B, 201, T, 2) real view, T = L/100 + 1.

    ref: train.py:81-87 / evaluation.py:36-38 (centre=True, reflect pad 200, periodic
    Hamming-400, hop 100, one-sided, not normalised).  Written as an explicit framed DFT
    (matrix product with a float64-generated basis) instead of calling an FFT library so
    the oracle does not share code with the op it checks.
    """
    B, L = x.shape
    dt = x.dtype
    xp = F.pad(x.unsqueeze(1), (N_FFT // 2, N_FFT // 2), mode="reflect").squeeze(1)
    T = L // HOP + 1
    idx = torch.arange(T).unsqueeze(1) * HOP + torch.arange(N_FFT).unsqueeze(0)
    frames = xp[:, idx] * hamming_window(N_FFT, dt)                 # (B, T, 400)
    n = torch.arange(N_FFT, dtype=torch.float64).unsqueeze(1)
    k = torch.arange(N_FFT // 2 + 1, dtype=torch.float64).unsqueeze(0)
    ang = 2.0 * math.pi * torch.remainder(n * k, N_FFT) / N_FFT     # (400, 201)
    re = frames @ torch.cos(ang).to(dt)                             # (B, T, 201)
    im = frames @ (-torch.sin(ang)).to(dt)
    return torch.stack([re, im], dim=-1).permute(0, 2, 1, 3).contiguous()


def istft(spec: Tensor) -> Tensor:
    """(B, 201, T, 2) -> (B, 100*(T-1)).

    ref: train.py:106-112 / evaluation.py:44-50 (torch.istft: one-sided C2R inverse DFT
    (imaginary parts of bins 0 and 200 ignored), times window, overlap-add, divided by the
    overlap-added squared window, 200 samples trimmed on both sides).
    """
    B, Fq, T, _ = spec.shape
    dt = spec.dtype
    n = torch.arange(N_FFT, dtype=torch.float64).unsqueeze(0)
    k = torch.arange(Fq, dtype=torch.float64).unsqueeze(1)
    ang = 2.0 * math.pi * torch.remainder(k * n, N_FFT) / N_FFT     # (201, 400)
    wk = torch.full((Fq, 1), 2.0, dtype=torch.float64)
    wk[0, 0] = 1.0
    wk[Fq - 1, 0] = 1.0
    cr = (wk * torch.cos(ang) / N_FFT).to(dt)
    ci = (-wk * torch.sin(ang) / N_FFT).to(dt)
    re = spec[..., 0].permute(0, 2, 1)                              # (B, T, 201)
    im = spec[..., 1].permute(0, 2, 1)
    win = hamming_window(N_FFT, dt)
    frames = (re @ cr + im @ ci) * win                              # (B, T, 400)
    out_len = N_FFT + HOP * (T - 1)
    y = torch.zeros(B, out_len, dtype=dt)
    env = torch.zeros(out_len, dtype=dt)
    w2 = win * win
    for t in range(T):
        y[:, t * HOP:t * HOP + N_FFT] += frames[:, t]
        env[t * HOP:t * HOP + N_FFT] += w2
    y = y[:, N_FFT // 2: out_len - N_FFT // 2]
    env = env[N_FFT // 2: out_len - N_FFT // 2]
    return y / env


def power_compress(x: Tensor) -> Tensor:
    """(..., 2) -> stack([re, im], 1) of |X|^0.3 * e^{j angle X} (ref: utils.py:20-29)."""
    real, imag = x[..., 0], x[..., 1]
    mag = torch.sqrt(real * real + imag * imag)
    phase = torch.atan2(imag, real)
    mag = mag ** 0.3
    return torch.stack([mag * torch.cos(phase), mag * torch.sin(phase)], 1)


def power_uncompress(real: Tensor, imag: Tensor) -> Tensor:
    """|Y|^(1/0.3) e^{j angle Y}, stacked on the last dim (ref: utils.py:32-39)."""
    mag = torch.sqrt(real * real + imag * imag)
    phase = torch.atan2(imag, real)
    mag = mag ** (1.0 / 0.3)
    return torch.stack([mag * torch.cos(phase), mag * torch.sin(phase)], -1)


# --------------------------------------------------------------------------- small building blocks
def _instance_norm(x: Tensor, w: Tensor, b: Tensor, eps: float = 1e-5) -> Tensor:
    """InstanceNorm2d(affine=True, track_running_stats=False): statistics over (H, W) per
    (b, c), biased variance, in train and eval (ref: generator.py:35,55,61,128,148)."""
    mean = x.mean(dim=(2, 3), keepdim=True)
    var = ((x - mean) ** 2).mean(dim=(2, 3), keepdim=True)
    return (x - mean) / torch.sqrt(var + eps) * w.view(1, -1, 1, 1) + b.view(1, -1, 1, 1)


def _prelu(x: Tensor, a: Tensor) -> Tensor:
    """PReLU with per-channel slope on dim 1 (ref: generator.py:37)."""
    shape = [1, -1] + [1] * (x.dim() - 2)
    return torch.where(x >= 0, x, x * a.view(shape))


def _layer_norm(x: Tensor, w: Tensor, b: Tensor, eps: float = 1e-5) -> Tensor:
    """LayerNorm over the last dim (ref: conformer.py:68,161,214)."""
    mean = x.mean(-1, keepdim=True)
    var = ((x - mean) ** 2).mean(-1, keepdim=True)
    return (x - mean) / torch.sqrt(var + eps) * w + b


def _swish(x: Tensor) -> Tensor:
    """x * sigmoid(x) (ref: conformer.py:25-27)."""
    return x * torch.sigmoid(x)


def _dropout(x: Tensor, p: float, masks: Optional[dict], key: str) -> Tensor:
    """Dropout as an explicit mask multiply.  ``masks`` is None in eval mode; in train
    mode it maps ``key`` to a {0,1} keep mask (the CUDA path exports the masks it drew so
    that train-mode parity can be checked exactly)."""
    if masks is None or p == 0.0:
        return x
    return x * masks[key].to(x.dtype) / (1.0 - p)


# --------------------------------------------------------------------------- conformer (conformer.py)
def feed_forward(x: Tensor, sd: SD, p: str, masks=None, mkey="") -> Tensor:
    """Scale(0.5, PreNorm(LN, Linear 64->256, Swish, Dropout, Linear 256->64, Dropout))
    ref: conformer.py:54-72,136-148,211-212.  Returns 0.5 * FF(LN(x)) (without residual)."""
    h = _layer_norm(x, sd[p + ".fn.norm.weight"], sd[p + ".fn.norm.bias"])
    h = h @ sd[p + ".fn.fn.net.0.weight"].t() + sd[p + ".fn.fn.net.0.bias"]
    h = _dropout(_swish(h), 0.2, masks, mkey + ".d1")
    h = h @ sd[p + ".fn.fn.net.3.weight"].t() + sd[p + ".fn.fn.net.3.bias"]
    h = _dropout(h, 0.2, masks, mkey + ".d2")
    return 0.5 * h


def attention(x: Tensor, sd: SD, p: str, heads: int = 4, max_pos: int = 512, masks=None, mkey="") -> Tensor:
    """PreNorm MHSA with Shaw relative positions (ref: conformer.py:75-133, no mask branch).

    x: (N, L, 64).  q has no bias, kv has no bias, k = first half of to_kv, v = second;
    heads are the outer factor of the channel split; both the content and the positional
    logits are scaled by dim_head^-0.5; dist[i, j] = clamp(i - j, +-512) + 512 indexes a
    (1025, 16) table shared by all heads; dropout acts on the projected output."""
    N, L, C = x.shape
    h = _layer_norm(x, sd[p + ".norm.weight"], sd[p + ".norm.bias"])
    q = h @ sd[p + ".fn.to_q.weight"].t()
    kv = h @ sd[p + ".fn.to_kv.weight"].t()
    k, v = kv[..., :C], kv[..., C:]
    d = C // heads
    scale = d ** -0.5
    q = q.view(N, L, heads, d).permute(0, 2, 1, 3)
    k = k.view(N, L, heads, d).permute(0, 2, 1, 3)
    v = v.view(N, L, heads, d).permute(0, 2, 1, 3)
    dots = torch.matmul(q, k.transpose(-1, -2)) * scale
    seq = torch.arange(L)
    dist = (seq.view(L, 1) - seq.view(1, L)).clamp(-max_pos, max_pos) + max_pos
    E = sd[p + ".fn.rel_pos_emb.weight"][dist]                      # (L, L, d)
    pos = torch.einsum("bhnd,nrd->bhnr", q, E) * scale
    attn = torch.softmax(dots + pos, dim=-1)
    out = torch.matmul(attn, v).permute(0, 2, 1, 3).reshape(N, L, C)
    out = out @ sd[p + ".fn.to_out.weight"].t() + sd[p + ".fn.to_out.bias"]
    return _dropout(out, 0.2, masks, mkey + ".d")


def conv_module(x: Tensor, sd: SD, p: str, training: bool = False, bn_out: Optional[dict] = None) -> Tensor:
    """LN, pointwise 64->256, GLU, zero-pad (15,15), depthwise k=31, BatchNorm1d(128),
    Swish, pointwise 128->64 (ref: conformer.py:30-48,151-176).  In training mode the batch
    statistics over (N, L) are used (biased var for the normalisation); ``bn_out`` receives
    the batch mean / unbiased var that update the running stats (momentum 0.1)."""
    N, L, C = x.shape
    h = _layer_norm(x, sd[p + ".net.0.weight"], sd[p + ".net.0.bias"])
    h = h @ sd[p + ".net.2.weight"][:, :, 0].t() + sd[p + ".net.2.bias"]          # (N, L, 256)
    inner = h.shape[-1] // 2
    h = h[..., :inner] * torch.sigmoid(h[..., inner:])
    w = sd[p + ".net.4.conv.weight"]                                              # (128, 1, 31)
    ks = w.shape[-1]
    hp = F.pad(h.transpose(1, 2), (ks // 2, ks // 2 - (ks + 1) % 2))              # (N, 128, L+30)
    h = F.conv1d(hp, w, sd[p + ".net.4.conv.bias"], groups=inner)                 # (N, 128, L)
    if training:
        mean = h.mean(dim=(0, 2))
        var = ((h - mean.view(1, -1, 1)) ** 2).mean(dim=(0, 2))
        if bn_out is not None:
            cnt = h.shape[0] * h.shape[2]
            bn_out[p] = (mean.detach(), (var * cnt / max(cnt - 1, 1)).detach())
    else:
        mean, var = sd[p + ".net.5.running_mean"], sd[p + ".net.5.running_var"]
    h = (h - mean.view(1, -1, 1)) / torch.sqrt(var.view(1, -1, 1) + 1e-5)
    h = h * sd[p + ".net.5.weight"].view(1, -1, 1) + sd[p + ".net.5.bias"].view(1, -1, 1)
    h = _swish(h).transpose(1, 2)
    return h @ sd[p + ".net.7.weight"][:, :, 0].t() + sd[p + ".net.7.bias"]


def conformer_block(x: Tensor, sd: SD, p: str, training: bool = False, masks=None, bn_out=None) -> Tensor:
    """Macaron block: x + 0.5 FF1; + Attn; + Conv; + 0.5 FF2; post LN (ref: conformer.py:216-222)."""
    x = feed_forward(x, sd, p + ".ff1", masks, p + ".ff1") + x
    x = attention(x, sd, p + ".attn", masks=masks, mkey=p + ".attn") + x
    x = conv_module(x, sd, p + ".conv", training, bn_out) + x
    x = feed_forward(x, sd, p + ".ff2", masks, p + ".ff2") + x
    return _layer_norm(x, sd[p + ".post_norm.weight"], sd[p + ".post_norm.bias"])


# --------------------------------------------------------------------------- generator (generator.py)
def dilated_dense(x: Tensor, sd: SD, p: str, depth: int = 4) -> Tensor:
    """4 x [causal-in-time zero pad (dil rows on top, 1/1 in freq), Conv2d(64i->64, k=(2,3),
    dilation (2^(i-1), 1)), InstanceNorm, PReLU, cat([out, skip])] (ref: generator.py:14-47)."""
    skip = x
    out = x
    for i in range(depth):
        dil = 2 ** i
        o = F.pad(skip, (1, 1, dil, 0))
        o = F.conv2d(o, sd[f"{p}.conv{i+1}.weight"], sd[f"{p}.conv{i+1}.bias"], dilation=(dil, 1))
        o = _instance_norm(o, sd[f"{p}.norm{i+1}.weight"], sd[f"{p}.norm{i+1}.bias"])
        out = _prelu(o, sd[f"{p}.prelu{i+1}.weight"])
        skip = torch.cat([out, skip], dim=1)
    return out


def dense_encoder(x: Tensor, sd: SD, p: str = "dense_encoder") -> Tensor:
    """1x1 conv 3->64 + IN + PReLU; dilated dense block; (1,3) stride (1,2) pad (0,1) conv +
    IN + PReLU (ref: generator.py:50-69)."""
    x = F.conv2d(x, sd[p + ".conv_1.0.weight"], sd[p + ".conv_1.0.bias"])
    x = _prelu(_instance_norm(x, sd[p + ".conv_1.1.weight"], sd[p + ".conv_1.1.bias"]), sd[p + ".conv_1.2.weight"])
    x = dilated_dense(x, sd, p + ".dilated_dense")
    x = F.conv2d(x, sd[p + ".conv_2.0.weight"], sd[p + ".conv_2.0.bias"], stride=(1, 2), padding=(0, 1))
    return _prelu(_instance_norm(x, sd[p + ".conv_2.1.weight"], sd[p + ".conv_2.1.bias"]), sd[p + ".conv_2.2.weight"])


def tscb(x: Tensor, sd: SD, p: str, training: bool = False, masks=None, bn_out=None) -> Tensor:
    """Two-stage conformer: time sequences (b*f, t, c) then frequency sequences (b*t, f, c),
    each with an outer residual (ref: generator.py:92-99)."""
    b, c, t, f = x.shape
    x_t = x.permute(0, 3, 2, 1).contiguous().view(b * f, t, c)
    x_t = conformer_block(x_t, sd, p + ".time_conformer", training, masks, bn_out) + x_t
    x_f = x_t.view(b, f, t, c).permute(0, 2, 1, 3).contiguous().view(b * t, f, c)
    x_f = conformer_block(x_f, sd, p + ".freq_conformer", training, masks, bn_out) + x_f
    return x_f.view(b, t, f, c).permute(0, 3, 1, 2)


def sp_conv_transpose(x: Tensor, sd: SD, p: str, r: int = 2) -> Tensor:
    """Sub-pixel up-sampling in F: pad (1,1), Conv2d(64 -> 64 r, (1,3)), then
    out[b, c, t, r*w + j] = conv[b, j*64 + c, t, w] (ref: generator.py:102-119)."""
    o = F.conv2d(F.pad(x, (1, 1, 0, 0)), sd[p + ".conv.weight"], sd[p + ".conv.bias"])
    B, nch, H, W = o.shape
    o = o.view(B, r, nch // r, H, W).permute(0, 2, 3, 4, 1)
    return o.contiguous().view(B, nch // r, H, -1)


def mask_decoder(x: Tensor, sd: SD, p: str = "mask_decoder") -> Tensor:
    """dense block, sub-pixel, (1,2) conv 64->1, IN(1), PReLU(1), 1x1 conv, PReLU with one
    slope per frequency bin; returns (B, 1, T, F) (ref: generator.py:122-139)."""
    x = dilated_dense(x, sd, p + ".dense_block")
    x = sp_conv_transpose(x, sd, p + ".sub_pixel")
    x = F.conv2d(x, sd[p + ".conv_1.weight"], sd[p + ".conv_1.bias"])
    x = _prelu(_instance_norm(x, sd[p + ".norm.weight"], sd[p + ".norm.bias"]), sd[p + ".prelu.weight"])
    x = F.conv2d(x, sd[p + ".final_conv.weight"], sd[p + ".final_conv.bias"])     # (B, 1, T, F)
    x = x.permute(0, 3, 2, 1).squeeze(-1)                                         # (B, F, T)
    return _prelu(x, sd[p + ".prelu_out.weight"]).permute(0, 2, 1).unsqueeze(1)


def complex_decoder(x: Tensor, sd: SD, p: str = "complex_decoder") -> Tensor:
    """dense block, sub-pixel, IN(64), PReLU(64), (1,2) conv 64->2 (ref: generator.py:142-156)."""
    x = dilated_dense(x, sd, p + ".dense_block")
    x = sp_conv_transpose(x, sd, p + ".sub_pixel")
    x = _prelu(_instance_norm(x, sd[p + ".norm.weight"], sd[p + ".norm.bias"]), sd[p + ".prelu.weight"])
    return F.conv2d(x, sd[p + ".conv.weight"], sd[p + ".conv.bias"])


def tscnet_forward(x: Tensor, sd: SD, training: bool = False, masks=None, bn_out=None,
                   taps: Optional[dict] = None) -> Tuple[Tensor, Tensor]:
    """TSCNet.forward: x (B, 2, T, F) -> (final_real, final_imag), each (B, 1, T, F)
    (ref: generator.py:174-196).  ``taps`` (optional dict) receives intermediate tensors."""
    mag = torch.sqrt(x[:, 0] ** 2 + x[:, 1] ** 2).unsqueeze(1)
    phase = torch.atan2(x[:, 1], x[:, 0]).unsqueeze(1)
    x_in = torch.cat([mag, x], dim=1)
    out = dense_encoder(x_in, sd)
    if taps is not None:
        taps["encoder"] = out
    for i in range(1, 5):
        out = tscb(out, sd, f"TSCB_{i}", training, masks, bn_out)
        if taps is not None:
            taps[f"tscb{i}"] = out
    mask = mask_decoder(out, sd)
    out_mag = mask * mag
    cplx = complex_decoder(out, sd)
    if taps is not None:
        taps["mask"] = mask
        taps["complex"] = cplx
    final_real = out_mag * torch.cos(phase) + cplx[:, 0].unsqueeze(1)
    final_imag = out_mag * torch.sin(phase) + cplx[:, 1].unsqueeze(1)
    return final_real, final_imag


# --------------------------------------------------------------------------- discriminator
def spectral_norm_weight(w_orig: Tensor, u: Tensor, v: Tensor, training: bool, eps: float = 1e-12):
    """Legacy torch.nn.utils.spectral_norm (ref: discriminator.py:33-58): in training one
    power iteration (v = normalize(W^T u), u = normalize(W v)) updates u, v; sigma = u^T W v;
    returns (W / sigma, u, v).  W is weight_orig flattened to (out, -1)."""
    wm = w_orig.reshape(w_orig.shape[0], -1)
    if training:
        with torch.no_grad():
            v = F.normalize(wm.t() @ u, dim=0, eps=eps)
            u = F.normalize(wm @ v, dim=0, eps=eps)
    sigma = torch.dot(u, wm @ v)
    return w_orig / sigma, u, v


def discriminator_forward(x: Tensor, y: Tensor, sd: SD, training: bool = False, drop_mask: Optional[Tensor] = None,
                          uv_out: Optional[dict] = None) -> Tensor:
    """Discriminator.forward(x, y), x and y (B, 1, F, T) -> (B, 1) (ref: discriminator.py:29-64,
    utils.py:42-50).  4 x [SN conv 4x4 s2 p1 no bias, IN(affine), PReLU], global max pool,
    SN linear, Dropout(0.3), PReLU, SN linear, LearnableSigmoid (beta 1)."""
    h = torch.cat([x, y], dim=1)
    for li in (0, 3, 6, 9):
        w, u, v = spectral_norm_weight(sd[f"layers.{li}.weight_orig"], sd[f"layers.{li}.weight_u"],
                                       sd[f"layers.{li}.weight_v"], training)
        if uv_out is not None:
            uv_out[li] = (u, v)
        h = F.conv2d(h, w, None, stride=2, padding=1)
        h = _instance_norm(h, sd[f"layers.{li+1}.weight"], sd[f"layers.{li+1}.bias"])
        h = _prelu(h, sd[f"layers.{li+2}.weight"])
    h = h.amax(dim=(2, 3))                                                        # AdaptiveMaxPool2d(1)+Flatten
    w, u, v = spectral_norm_weight(sd["layers.14.weight_orig"], sd["layers.14.weight_u"], sd["layers.14.weight_v"], training)
    if uv_out is not None:
        uv_out[14] = (u, v)
    h = h @ w.t() + sd["layers.14.bias"]
    if training and drop_mask is not None:
        h = h * drop_mask.to(h.dtype) / 0.7
    h = _prelu(h, sd["layers.16.weight"])
    w, u, v = spectral_norm_weight(sd["layers.17.weight_orig"], sd["layers.17.weight_u"], sd["layers.17.weight_v"], training)
    if uv_out is not None:
        uv_out[17] = (u, v)
    h = h @ w.t() + sd["layers.17.bias"]
    return torch.sigmoid(sd["layers.18.slope"] * h)


# --------------------------------------------------------------------------- call-site glue
def enhance(noisy: Tensor, sd: SD, cut_len: Optional[int] = None, normalise: bool = True) -> Tensor:
    """evaluation.enhance_one_track between load and save (ref: evaluation.py:21-53):
    (1, L) waveform -> (L,) enhanced waveform in the original scale.  Wrap-pads to a multiple
    of 100 with the signal's own head, folds into a batch when padded_len > cut_len."""
    assert noisy.dim() == 2
    c = rms_scale(noisy) if normalise else torch.ones(noisy.shape[0], dtype=noisy.dtype)
    noisy = (noisy.t() * c).t()
    length = noisy.size(-1)
    frame_num = int(math.ceil(length / 100))
    padded_len = frame_num * 100
    noisy = torch.cat([noisy, noisy[:, :padded_len - length]], dim=-1)
    if cut_len is not None and padded_len > cut_len:
        batch_size = int(math.ceil(padded_len / cut_len))
        while 100 % batch_size != 0:
            batch_size += 1
        noisy = noisy.reshape(batch_size, -1)
    spec = power_compress(stft(noisy)).permute(0, 1, 3, 2)
    er, ei = tscnet_forward(spec, sd)
    er, ei = er.permute(0, 1, 3, 2), ei.permute(0, 1, 3, 2)
    audio = istft(power_uncompress(er, ei).squeeze(1))
    audio = audio / c
    return torch.flatten(audio)[:length]


def forward_generator_step(clean: Tensor, noisy: Tensor, sd: SD, training: bool = False, masks=None, bn_out=None) -> Dict[str, Tensor]:
    """Trainer.forward_generator_step (ref: train.py:72-122)."""
    c = rms_scale(noisy)
    noisy = (noisy.t() * c).t()
    clean = (clean.t() * c).t()
    noisy_spec = power_compress(stft(noisy)).permute(0, 1, 3, 2)
    clean_spec = power_compress(stft(clean))
    clean_real, clean_imag = clean_spec[:, 0:1], clean_spec[:, 1:2]
    er, ei = tscnet_forward(noisy_spec, sd, training, masks, bn_out)
    er, ei = er.permute(0, 1, 3, 2), ei.permute(0, 1, 3, 2)
    est_mag = torch.sqrt(er ** 2 + ei ** 2)
    clean_mag = torch.sqrt(clean_real ** 2 + clean_imag ** 2)
    est_audio = istft(power_uncompress(er, ei).squeeze(1))
    return dict(est_real=er, est_imag=ei, est_mag=est_mag, clean_real=clean_real, clean_imag=clean_imag,
                clean_mag=clean_mag, est_audio=est_audio)


def generator_loss(go: Dict[str, Tensor], clean_unnormalised: Tensor, d_fake: Tensor,
                   weights=(0.1, 0.9, 0.2, 0.05)) -> Tensor:
    """Trainer.calculate_generator_loss (ref: train.py:124-151).  ``d_fake`` = D(clean_mag,
    est_mag).  The time loss compares est_audio (RMS-normalised scale) with the *un-normalised*
    clean put into the dict by train_step (ref: train.py:188) -- reproduced as is."""
    ones = torch.ones(d_fake.shape[0], dtype=d_fake.dtype)
    gan = F.mse_loss(d_fake.flatten(), ones)
    mag = F.mse_loss(go["est_mag"], go["clean_mag"])
    ri = F.mse_loss(go["est_real"], go["clean_real"]) + F.mse_loss(go["est_imag"], go["clean_imag"])
    time_l = torch.mean(torch.abs(go["est_audio"] - clean_unnormalised))
    return weights[0] * ri + weights[1] * mag + weights[2] * time_l + weights[3] * gan


def discriminator_loss(d_max: Tensor, d_enh: Tensor, pesq_target: Tensor) -> Tensor:
    """Trainer.calculate_discriminator_loss once the PESQ targets exist (ref: train.py:161-170):
    MSE(D(clean, clean), 1) + MSE(D(clean, est.detach()), (pesq - 1) / 3.5)."""
    ones = torch.ones(d_max.shape[0], dtype=d_max.dtype)
    return F.mse_loss(d_max.flatten(), ones) + F.mse_loss(d_enh.flatten(), pesq_target)


def load_weights_npz(path: str, dtype=torch.float32) -> Dict[str, Tensor]:
    """Load a fixture written by tools/make_golden.py (np.savez of a state dict)."""
    import numpy as np
    z = np.load(path)
    out = {}
    for k in z.files:
        a = torch.from_numpy(z[k])
        out[k] = a.to(dtype) if a.is_floating_point() else a
    return out

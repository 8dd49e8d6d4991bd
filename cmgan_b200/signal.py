"""Signal front/back end of the hot path on the GPU: RMS normalise -> STFT -> power compression, and
power un-compression -> iSTFT (ref: train.py:75-112, evaluation.py:21-51, utils.py:20-39).

The framed DFT (n_fft 400, hop 100, periodic Hamming, centre/reflect) is a GEMM over overlapping rows of the
padded waveform (lda = hop) against a window-folded DFT basis; the inverse is a GEMM against the window-folded
inverse basis followed by overlap-add.  Both run in exact fp32 FFMA (0.1 GFLOP per utterance).
"""
from __future__ import annotations

import math
from typing import Dict, List, Sequence, Tuple

import torch

from .ops import call, gemm

N_FFT, HOP, NF = 400, 100, 201
_CACHE: Dict[Tuple, torch.Tensor] = {}


def _window64():
    k = torch.arange(N_FFT, dtype=torch.float64)
    return 0.54 - 0.46 * torch.cos(2.0 * math.pi * k / N_FFT)


def _fwd_basis(dev) -> torch.Tensor:
    """(400, 402): [w[n] cos(2 pi k n / 400) | -w[n] sin(2 pi k n / 400)], generated in float64"""
    key = ("fwd", dev)
    if key not in _CACHE:
        n = torch.arange(N_FFT, dtype=torch.float64).unsqueeze(1)
        k = torch.arange(NF, dtype=torch.float64).unsqueeze(0)
        ang = 2.0 * math.pi * torch.remainder(n * k, N_FFT) / N_FFT
        w = _window64().unsqueeze(1)
        _CACHE[key] = torch.cat([w * torch.cos(ang), -w * torch.sin(ang)], dim=1).to(torch.float32).contiguous().to(dev)
    return _CACHE[key]


def _inv_basis(dev) -> torch.Tensor:
    """(402, 400): one-sided inverse DFT (weights 1, 2, ..., 2, 1; /400) times the synthesis window"""
    key = ("inv", dev)
    if key not in _CACHE:
        n = torch.arange(N_FFT, dtype=torch.float64).unsqueeze(0)
        k = torch.arange(NF, dtype=torch.float64).unsqueeze(1)
        ang = 2.0 * math.pi * torch.remainder(k * n, N_FFT) / N_FFT
        wk = torch.full((NF, 1), 2.0, dtype=torch.float64)
        wk[0, 0] = 1.0
        wk[NF - 1, 0] = 1.0
        w = _window64().unsqueeze(0)
        _CACHE[key] = torch.cat([wk * torch.cos(ang) * w / N_FFT, -wk * torch.sin(ang) * w / N_FFT], dim=0).to(torch.float32).contiguous().to(dev)
    return _CACHE[key]


def _window_sq(dev) -> torch.Tensor:
    """(400,) float64 squared analysis window: the terms _inv_envelope sums (the ragged overlap-add sums them on the GPU)"""
    key = ("wsq", dev)
    if key not in _CACHE:
        _CACHE[key] = (_window64() ** 2).contiguous().to(dev)
    return _CACHE[key]


def _inv_envelope(T: int, dev) -> torch.Tensor:
    """1 / sum_t w^2[n + 200 - 100 t] for n < 100 (T - 1)"""
    key = ("env", T, dev)
    if key not in _CACHE:
        w2 = _window64() ** 2
        out_len = N_FFT + HOP * (T - 1)
        env = torch.zeros(out_len, dtype=torch.float64)
        for t in range(T):
            env[t * HOP:t * HOP + N_FFT] += w2
        env = env[N_FFT // 2: out_len - N_FFT // 2]
        _CACHE[key] = (1.0 / env).to(torch.float32).contiguous().to(dev)
    return _CACHE[key]


def rms_scale(wav: torch.Tensor) -> torch.Tensor:
    """c[b] = sqrt(L / sum x^2)  (ref: train.py:75, evaluation.py:21)"""
    assert wav.is_cuda and wav.dtype == torch.float32 and wav.dim() == 2 and wav.stride(1) == 1
    c = torch.empty(wav.shape[0], device=wav.device)
    call("cmgan_rms_scale", wav, wav.stride(0), wav.shape[0], wav.shape[1], c)
    return c


def stft_compress(wav: torch.Tensor, scale: torch.Tensor = None) -> torch.Tensor:
    """(B, L) waveform (optionally scaled per utterance by ``scale``) -> power-compressed spectrogram with the shape
    the reference's ``power_compress(torch.stft(...))`` has, (B, 2, F, T), as a permuted view of (B, 2, T, F) memory
    (so that ``.permute(0, 1, 3, 2)`` -- train.py:95 -- yields a contiguous tensor)."""
    assert wav.is_cuda and wav.dtype == torch.float32 and wav.dim() == 2 and wav.stride(1) == 1
    dev = wav.device
    B, L = wav.shape
    T = L // HOP + 1
    Lp = ((L + N_FFT + HOP - 1) // HOP) * HOP
    xp = torch.empty(B, Lp, device=dev)
    call("cmgan_pad_reflect", wav, wav.stride(0), B, L, scale, xp, Lp)
    return _stft_padded(xp, T)


def _stft_padded(xp: torch.Tensor, T: int) -> torch.Tensor:
    """(B, Lp) padded waveform (Lp a multiple of 100, >= 100 (T - 1) + 400) -> power-compressed (B, 2, T, F) as the (B, 2, F, T) view"""
    dev = xp.device
    B, Lp = xp.shape
    S = torch.empty(B * T, 2 * NF, device=dev)
    gemm(A=xp, lda=HOP, W=_fwd_basis(dev), sb_k=2 * NF, sb_n=1, C=S, ldc=2 * NF, M=B * T, N=2 * NF, Cin=N_FFT, taps=[(0, 0)],
         conv=dict(OH=1, OW=T, IH=1, IW=Lp // HOP), precision=0)      # the DFTs stay exact fp32
    X = torch.empty(B, 2, T, NF, device=dev)
    call("cmgan_compress", S, B, T, X)
    return X.permute(0, 1, 3, 2)


def uncompress_istft_fwd(fr: torch.Tensor, fi: torch.Tensor, c_div: torch.Tensor = None) -> torch.Tensor:
    """un-compress (B,1,T,F) x 2 -> inverse DFT (GEMM) -> overlap-add -> (B, 100 (T-1)); no autograd"""
    dev = fr.device
    B, _, T, F = fr.shape
    assert F == NF and fi.stride() == fr.stride()
    s = fr.stride()
    U = torch.empty(B * T, 2 * NF, device=dev)
    call("cmgan_uncompress", fr, fi, s[0], s[2], s[3], B, T, U)
    frames = torch.empty(B * T, N_FFT, device=dev)
    gemm(A=U, lda=2 * NF, W=_inv_basis(dev), sb_k=N_FFT, sb_n=1, C=frames, ldc=N_FFT, M=B * T, N=N_FFT, Cin=2 * NF, precision=0)
    y = torch.empty(B, HOP * (T - 1), device=dev)
    call("cmgan_ola", frames, B, T, _inv_envelope(T, dev), c_div, y, y.stride(0))
    return y


def uncompress_istft_bwd(fr: torch.Tensor, fi: torch.Tensor, dy: torch.Tensor, dre: torch.Tensor, dim: torch.Tensor, accumulate: bool) -> None:
    """gradient of uncompress_istft_fwd wrt (fr, fi) written (or added) into dre / dim ((B,1,T,F) contiguous)"""
    dev = fr.device
    B, _, T, F = fr.shape
    dframes = torch.empty(B * T, N_FFT, device=dev)
    call("cmgan_ola_bwd", dy, dy.stride(0), B, T, _inv_envelope(T, dev), dframes)
    dU = torch.empty(B * T, 2 * NF, device=dev)
    gemm(A=dframes, lda=N_FFT, W=_inv_basis(dev), sb_k=1, sb_n=N_FFT, C=dU, ldc=2 * NF, M=B * T, N=2 * NF, Cin=N_FFT, precision=0)
    s = fr.stride()
    call("cmgan_uncompress_bwd", fr, fi, s[0], s[2], s[3], B, T, dU, dre, dim, 1 if accumulate else 0)


class _UncompressISTFT(torch.autograd.Function):
    @staticmethod
    def forward(ctx, fr, fi, c_div):
        if fi.stride() != fr.stride():
            fr, fi = fr.contiguous(), fi.contiguous()
        y = uncompress_istft_fwd(fr, fi, c_div)
        ctx.save_for_backward(fr, fi)
        ctx.has_c = c_div is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        fr, fi = ctx.saved_tensors
        assert not ctx.has_c, "the de-normalised (evaluation) path is inference only"
        B, _, T, F = fr.shape
        dre = torch.empty(B, 1, T, F, device=fr.device)
        dim = torch.empty(B, 1, T, F, device=fr.device)
        uncompress_istft_bwd(fr, fi, dy.contiguous(), dre, dim, False)
        return dre, dim, None


def uncompress_istft(final_real: torch.Tensor, final_imag: torch.Tensor, c_div: torch.Tensor = None) -> torch.Tensor:
    """(B, 1, T, F) x 2 (TSCNet outputs, any strides) -> waveform (B, 100 (T - 1)); differentiable.
    ``c_div``: optional per-utterance divisor (evaluation.py:51 de-normalisation)."""
    return _UncompressISTFT.apply(final_real, final_imag, c_div)


@torch.no_grad()
def enhance_batch(model, noisy: torch.Tensor) -> torch.Tensor:
    """(B, L) clips of ONE length, each treated exactly as ``enhance`` treats a single file no longer than cut_len (per-utterance RMS
    normalisation, wrap padding, de-normalisation, truncation): the batched form used by the file front end and the throughput sweep."""
    assert noisy.dim() == 2
    noisy = noisy.contiguous()
    B, length = noisy.shape
    c = rms_scale(noisy)
    padded_len = int(math.ceil(length / 100)) * 100
    if padded_len != length:
        noisy = torch.cat([noisy, noisy[:, :padded_len - length]], dim=-1)
    spec = stft_compress(noisy, c).permute(0, 1, 3, 2)
    fr, fi = model(spec)
    return uncompress_istft(fr, fi, c)[:, :length]


@torch.no_grad()
def enhance(model, noisy: torch.Tensor, cut_len: int = 16000 * 16) -> torch.Tensor:
    """evaluation.enhance_one_track between load and save (ref: evaluation.py:21-53) on the GPU: (1, L) -> (L,)."""
    assert noisy.dim() == 2 and noisy.shape[0] == 1
    noisy = noisy.contiguous()
    length = noisy.size(-1)
    c = rms_scale(noisy)
    padded_len = int(math.ceil(length / 100)) * 100
    if padded_len != length:            # wrap padding with the signal's own head (evaluation.py:25-29)
        noisy = torch.cat([noisy, noisy[:, :padded_len - length]], dim=-1)
    batch = 1
    if padded_len > cut_len:            # fold long files into the batch (evaluation.py:30-34)
        batch = int(math.ceil(padded_len / cut_len))
        while 100 % batch != 0:
            batch += 1
        noisy = noisy.reshape(batch, -1)
    cb = c.expand(batch).contiguous() if batch > 1 else c
    spec = stft_compress(noisy, cb).permute(0, 1, 3, 2)
    fr, fi = model(spec)
    audio = uncompress_istft(fr, fi, cb)
    return audio.reshape(-1)[:length]


# ---------------------------------------------------------------------------------------------------------- ragged batches
MAX_CAT_ELEMS = 2 ** 31     # the encoder's (B T F, 320) concat buffer is indexed with 32-bit element counts


def clip_frames(length: int) -> int:
    """STFT frames of a clip of ``length`` samples after the wrap padding to a multiple of 100 (evaluation.py:25-29)"""
    return int(math.ceil(length / HOP)) + 1


def plan_ragged(lengths: Sequence[int], max_batch: int = 16, cut_len: int = 16000 * 16) -> Tuple[List[List[int]], List[int]]:
    """Batch plan for ``enhance_ragged``: -> (batches, solo), lists of indices into ``lengths``.
    Clips whose wrap-padded length exceeds ``cut_len`` go to ``solo`` (the folding path of ``enhance``, one at a time).  The others are
    sorted by length and cut into consecutive groups of at most ``max_batch`` clips, so a batch pads little; a group also stops before
    B * T_max * 201 * 320 reaches 2^31 (the encoder's concat buffer).  Clips of 200 samples or fewer are rejected: the reflect padding
    of the STFT needs more."""
    if max_batch < 1:
        raise ValueError("plan_ragged: max_batch must be >= 1")
    for i, n in enumerate(lengths):
        if n <= N_FFT // 2:
            raise ValueError(f"plan_ragged: clip {i} has {n} samples; at least {N_FFT // 2 + 1} are needed")
    solo = [i for i, n in enumerate(lengths) if int(math.ceil(n / HOP)) * HOP > cut_len]
    rest = sorted((i for i, n in enumerate(lengths) if int(math.ceil(n / HOP)) * HOP <= cut_len), key=lambda i: (lengths[i], i))
    batches: List[List[int]] = []
    cur: List[int] = []
    for i in rest:
        t_max = clip_frames(lengths[i])          # sorted ascending: the clip being added is the longest of its group
        if cur and (len(cur) == max_batch or (len(cur) + 1) * t_max * NF * 320 >= MAX_CAT_ELEMS):
            batches.append(cur)
            cur = []
        cur.append(i)
    if cur:
        batches.append(cur)
    return batches, solo


def uncompress_istft_varlen(fr: torch.Tensor, fi: torch.Tensor, nframes: torch.Tensor, c_div: torch.Tensor) -> torch.Tensor:
    """``uncompress_istft_fwd`` of a ragged batch: utterance b has nframes[b] (device int32) of the T frames; its samples
    0 .. 100 (nframes[b] - 1) equal those of a run on its frames alone (per-utterance synthesis envelope), the rest are zero"""
    dev = fr.device
    B, _, T, F = fr.shape
    assert F == NF and fi.stride() == fr.stride()
    s = fr.stride()
    U = torch.empty(B * T, 2 * NF, device=dev)
    call("cmgan_uncompress", fr, fi, s[0], s[2], s[3], B, T, U)
    frames = torch.empty(B * T, N_FFT, device=dev)
    gemm(A=U, lda=2 * NF, W=_inv_basis(dev), sb_k=N_FFT, sb_n=1, C=frames, ldc=N_FFT, M=B * T, N=N_FFT, Cin=2 * NF, precision=0)
    y = torch.empty(B, HOP * (T - 1), device=dev)
    call("cmgan_ola_varlen", frames, B, T, nframes, _window_sq(dev), c_div, y, y.stride(0))
    return y


@torch.no_grad()
def enhance_ragged(model, waves: Sequence[torch.Tensor], cut_len: int = 16000 * 16) -> List[torch.Tensor]:
    """Enhance clips of different lengths in one forward pass: each 1-D clip (200 < length, wrap-padded length <= ``cut_len``) gets
    exactly what ``enhance`` does to one file -- RMS normalisation, wrap padding with its own head, STFT, TSCNet, iSTFT,
    de-normalisation, truncation -- and the list of enhanced clips (on the model's device) comes back in the input order.
    The clips are zero-padded to the longest; TSCNet runs on the ragged batch (``TSCNet.forward(x, frames)``)."""
    if len(waves) == 0:
        return []
    lengths = [int(w.numel()) for w in waves]
    for i, n in enumerate(lengths):
        if n <= N_FFT // 2 or int(math.ceil(n / HOP)) * HOP > cut_len:
            raise ValueError(f"enhance_ragged: clip {i} has {n} samples; need {N_FFT // 2} < length and a padded length <= cut_len ({cut_len})")
    dev = next(model.parameters()).device
    B = len(waves)
    x = torch.nn.utils.rnn.pad_sequence([w.reshape(-1) for w in waves], batch_first=True).to(dev, torch.float32).contiguous()
    nfr = [clip_frames(n) for n in lengths]
    T = max(nfr)
    meta = torch.tensor([lengths, nfr], dtype=torch.int32).to(dev)       # one upload: sample counts, frame counts
    lens, nframes = meta[0], meta[1]
    c = torch.empty(B, device=dev)
    call("cmgan_rms_scale_varlen", x, x.stride(0), B, lens, c)
    Lp = HOP * (T - 1) + N_FFT
    xp = torch.empty(B, Lp, device=dev)
    call("cmgan_wrap_pad_reflect_varlen", x, x.stride(0), B, lens, c, xp, Lp)
    spec = _stft_padded(xp, T).permute(0, 1, 3, 2)
    fr, fi = model(spec, frames=nfr)
    if fi.stride() != fr.stride():
        fr, fi = fr.contiguous(), fi.contiguous()
    y = uncompress_istft_varlen(fr, fi, nframes, c)
    return [y[b, :n] for b, n in enumerate(lengths)]

"""The callers on the inference side of the hot path (reference evaluation.py:12-106): wav files in, enhanced wav files (+ scores) out.

``enhance_one_track`` keeps the reference function's signature and semantics -- load, RMS-normalise, wrap-pad to a multiple of 100 with
the signal's own head, fold files longer than ``cut_len`` into a batch, STFT -> TSCNet -> iSTFT, de-normalise, truncate, optionally save
-- with the model path on the GPU (signal.enhance) and the file I/O on scipy.io.wavfile (torchaudio.load needs torchcodec and soundfile
is absent here; 16-bit PCM, 32-bit float and 32-bit PCM files are read to float32 in [-1, 1) exactly as torchaudio does, float32 is
written like soundfile's default for float input would be on a FLOAT-subtype file -- pass ``subtype='PCM_16'`` for 16-bit output).

``enhance_files`` is the throughput front-end: files of different lengths share one forward pass as a ragged batch (signal.plan_ragged sorts
them by length and cuts groups of at most ``max_batch``; signal.enhance_ragged pads each group to its longest clip and TSCNet reads only
each clip's own frames -- the convolutions are causal in time, attention, the depthwise convolution and the InstanceNorm statistics stop at
each clip's length), so every file gets its per-file result.  ``evaluation`` enhances through it and scores file by file.
"""
from __future__ import annotations

import os
import re
from typing import Callable, Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import signal

SR = 16000


def read_wav(path: str) -> Tuple[torch.Tensor, int]:
    """-> ((channels, samples) float32 in [-1, 1), sample rate), the layout torchaudio.load returns (evaluation.py:17)"""
    from scipy.io import wavfile
    sr, x = wavfile.read(path)
    if x.dtype == np.int16:
        y = x.astype(np.float32) / 32768.0
    elif x.dtype == np.int32:
        y = (x.astype(np.float64) / 2147483648.0).astype(np.float32)
    elif x.dtype == np.uint8:
        y = (x.astype(np.float32) - 128.0) / 128.0
    else:
        y = x.astype(np.float32)
    y = y.reshape(len(y), -1).T                    # (channels, samples)
    return torch.from_numpy(np.ascontiguousarray(y)), int(sr)


def write_wav(path: str, audio: np.ndarray, sr: int = SR, subtype: str = "FLOAT") -> None:
    from scipy.io import wavfile
    a = np.asarray(audio)
    if subtype == "PCM_16":
        a = np.clip(np.round(a * 32768.0), -32768, 32767).astype(np.int16)
    else:
        a = a.astype(np.float32)
    wavfile.write(path, sr, a)


def natural_sorted(names: Iterable[str]) -> List[str]:
    """natsort.natsorted for plain file names (evaluation.py:70): digit runs compare as integers"""
    def key(s):
        return [int(t) if t.isdigit() else t for t in re.split(r"(\d+)", s)]
    return sorted(names, key=key)


@torch.no_grad()
def enhance_one_track(model, audio_path: str, saved_dir: Optional[str], cut_len: int, n_fft: int = 400, hop: int = 100,
                      save_tracks: bool = False) -> Tuple[np.ndarray, int]:
    """reference evaluation.py:12-58, same arguments and return value ((length,) float32 numpy array, length)"""
    assert n_fft == 400 and hop == 100, "the CUDA front end is specialised for n_fft 400 / hop 100 (the reference's only setting)"
    name = os.path.split(audio_path)[-1]
    noisy, sr = read_wav(audio_path)
    assert sr == SR
    dev = next(model.parameters()).device
    est = signal.enhance(model, noisy[:1].to(dev), cut_len=cut_len)
    est_audio = est.cpu().numpy()
    length = noisy.size(-1)
    assert len(est_audio) == length
    if save_tracks:
        write_wav(os.path.join(saved_dir, name), est_audio, sr)
    return est_audio, length


@torch.no_grad()
def enhance_files(model, paths: Sequence[str], cut_len: int = SR * 16, max_batch: int = 16) -> Dict[str, np.ndarray]:
    """Enhance many files -> {path: enhanced (length,) float32}, the per-file results of ``enhance_one_track``.  Files up to ``cut_len``
    go through ragged batches of at most ``max_batch`` clips of mixed lengths (signal.plan_ragged / signal.enhance_ragged); longer files
    take the reference's folding path one at a time."""
    dev = next(model.parameters()).device
    paths = list(paths)
    waves = []
    for p in paths:
        x, sr = read_wav(p)
        assert sr == SR
        waves.append(x[0])
    batches, solo = signal.plan_ragged([w.numel() for w in waves], max_batch=max_batch, cut_len=cut_len)
    out: Dict[str, np.ndarray] = {}
    for i in solo:
        out[paths[i]] = signal.enhance(model, waves[i][None].to(dev), cut_len=cut_len).cpu().numpy()
    for idx in batches:
        est = signal.enhance_ragged(model, [waves[i] for i in idx], cut_len=cut_len)
        for i, e in zip(idx, est):
            out[paths[i]] = e.cpu().numpy()
    return out


@torch.no_grad()
def evaluation(model, noisy_dir: str, clean_dir: str, save_tracks: bool, saved_dir: str,
               metrics: Optional[Callable[[np.ndarray, np.ndarray], Sequence[float]]] = None, cut_len: int = SR * 16, max_batch: int = 16):
    """reference evaluation.py:60-97 with an already-loaded ``model``: enhance every file of ``noisy_dir`` (``enhance_files``: ragged batches
    of up to ``max_batch`` files, the per-file results), then in natural order save it and score it against the file of the same name in
    ``clean_dir`` with ``metrics(clean, enhanced) -> sequence`` (default: the PESQ-free pair SSNR, STOI from cmgan_b200.metrics on the GPU);
    returns the per-metric averages."""
    model.eval()
    if save_tracks and not os.path.exists(saved_dir):
        os.mkdir(saved_dir)
    if metrics is None:
        from . import metrics as gpu_metrics
        dev = next(model.parameters()).device

        def metrics(clean, est):
            return gpu_metrics.ssnr_stoi(torch.from_numpy(clean).to(dev), torch.from_numpy(est).to(dev))
    names = natural_sorted(os.listdir(noisy_dir))
    enhanced = enhance_files(model, [os.path.join(noisy_dir, name) for name in names], cut_len=cut_len, max_batch=max_batch)
    total = None
    for name in names:
        est_audio = enhanced[os.path.join(noisy_dir, name)]
        length = len(est_audio)
        if save_tracks:
            write_wav(os.path.join(saved_dir, name), est_audio, SR)
        clean, sr = read_wav(os.path.join(clean_dir, name))
        assert sr == SR
        m = np.asarray(metrics(clean[0].numpy()[:length], est_audio), dtype=np.float64)
        total = m if total is None else total + m
    return total / max(len(names), 1)

"""Ragged-batch inference on the CPU: the batch planner (pure function) and the new C declarations binding through the header."""
import os

import numpy as np
import pytest

from cmgan_b200 import signal
from conftest import GOLDEN

NEW_ENTRIES = {
    "cmgan_attention_fwd_varlen": 10, "cmgan_attention_fwd_tf32_varlen": 10, "cmgan_glu_dwconv_fwd_varlen": 10,
    "cmgan_norm_stats_varlen": 9, "cmgan_norm_finalize_varlen": 14, "cmgan_rms_scale_varlen": 6, "cmgan_wrap_pad_reflect_varlen": 8,
    "cmgan_ola_varlen": 9, "cmgan_tscnet_fwd_varlen": 16,
}


def test_new_declarations_bind():
    from cmgan_b200._lib import lib, parse_header
    protos = parse_header()
    for name, nargs in NEW_ENTRIES.items():
        assert name in protos, name
        assert len(protos[name][1]) == nargs, name
        getattr(lib().cdll, name)           # the library exports it (AttributeError otherwise)


def _cap_ok(lengths, batch):
    return len(batch) * max(signal.clip_frames(lengths[i]) for i in batch) * 201 * 320 < 2 ** 31


def test_plan_sorts_and_respects_max_batch():
    rng = np.random.default_rng(0)
    lengths = [int(v) for v in rng.integers(int(2.1 * 16000), int(9.8 * 16000), size=203)]
    for max_batch in (1, 4, 8, 16, 32):
        batches, solo = signal.plan_ragged(lengths, max_batch=max_batch)
        assert solo == []
        flat = [i for b in batches for i in b]
        assert sorted(flat) == list(range(len(lengths)))                               # every clip exactly once
        assert [lengths[i] for i in flat] == sorted(lengths)                           # sorted by length, consecutive groups
        assert all(1 <= len(b) <= max_batch for b in batches)
        if max_batch <= 16:                # 16 x 1564 frames stay under the element cap; 32 of the longest clips do not
            assert all(len(b) == max_batch for b in batches[:-1])
        assert all(_cap_ok(lengths, b) for b in batches)


def test_plan_element_cap_splits_audiosamples_length_clips():
    n = 1563 * 100                         # 1564 STFT frames: the longest AudioSamples clip (9.8 s)
    assert signal.clip_frames(n) == 1564
    lengths = [n] * 25
    assert 25 * 1564 * 201 * 320 >= 2 ** 31
    batches, solo = signal.plan_ragged(lengths, max_batch=32)
    assert solo == [] and len(batches) >= 2
    assert all(_cap_ok(lengths, b) for b in batches)
    assert sum(len(b) for b in batches) == 25
    # the real AudioSamples set at max_batch 32 splits the same way
    z = np.load(os.path.join(GOLDEN, "audiosamples.npz"))
    real = [int(v) for v in z["lengths"]]
    batches, _ = signal.plan_ragged(real, max_batch=32)
    assert len(batches) >= 2 and all(_cap_ok(real, b) for b in batches)


def test_plan_routes_long_clips_to_solo():
    cut = 16000 * 2
    lengths = [cut, cut + 1, 5000, cut + 100, cut - 99, 300]
    batches, solo = signal.plan_ragged(lengths, max_batch=4, cut_len=cut)
    assert solo == [1, 3]                  # wrap-padded length > cut_len: cut + 1 -> cut + 100
    assert [i for b in batches for i in b] == [5, 2, 4, 0]


def test_plan_rejects_short_clips():
    with pytest.raises(ValueError, match="clip 1"):
        signal.plan_ragged([1000, 200, 5000])
    signal.plan_ragged([201])
    with pytest.raises(ValueError):
        signal.plan_ragged([1000], max_batch=0)


def test_tscnet_module_conversions():
    """TSCNet.forward grew a ``frames`` argument; nn.Module's own machinery (``.to``, ``.float``, ``.eval``) is untouched"""
    import cmgan_b200
    m = cmgan_b200.TSCNet(64, 201).to("cpu").float().eval()
    assert not m.training and next(m.parameters()).dtype.is_floating_point

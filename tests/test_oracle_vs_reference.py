"""Pin the oracle against the reference modules: their outputs on the inputs below are stored in
tests/golden/oracle_vs_reference.npz (tools/make_golden_oracle_pins.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import cmgan_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def inputs():
    """numpy's legacy RandomState streams are frozen across numpy versions: the same inputs wherever the fixture is checked"""
    r = np.random.RandomState(3)
    tscnet = 0.7 * r.standard_normal((1, 2, 23, 201))
    compress = np.random.RandomState(1).standard_normal((2, 201, 9, 2))
    compress[0, 0, 0] = 0.0                        # zero magnitude: atan2(0, 0) and 0 ** 0.3
    r = np.random.RandomState(11)
    disc_x, disc_y = r.random_sample((3, 1, 201, 33)), r.random_sample((3, 1, 201, 33))
    return {k: torch.from_numpy(v.astype(np.float32)) for k, v in
            dict(tscnet=tscnet, compress=compress, disc_x=disc_x, disc_y=disc_y).items()}


@pytest.fixture(scope="module")
def ref():
    z = np.load(os.path.join(GOLDEN, "oracle_vs_reference.npz"))
    return {k: torch.from_numpy(z[k]) for k in z.files}


def test_tscnet_random_input(ref, g_weights):
    x = inputs()["tscnet"]
    with torch.no_grad():
        b = O.tscnet_forward(x, g_weights)
    for u, v in zip((ref["tscnet_real"], ref["tscnet_imag"]), b):
        assert (u - v).abs().max().item() < 3e-5


def test_stft_matches_torch():
    torch.manual_seed(0)
    x = torch.randn(3, 1700) * 0.1
    a = torch.view_as_real(torch.stft(x, 400, 100, window=torch.hamming_window(400), onesided=True, return_complex=True))
    assert (a - O.stft(x)).abs().max().item() < 2e-5
    y = torch.istft(torch.view_as_complex(a.contiguous()), 400, 100, window=torch.hamming_window(400), onesided=True)
    assert (y - O.istft(a)).abs().max().item() < 2e-6


def test_compress_matches(ref):
    x = inputs()["compress"]
    assert (ref["compress"] - O.power_compress(x)).abs().max().item() < 1e-6
    c = ref["compress"]
    assert (ref["uncompress"] - O.power_uncompress(c[:, 0:1], c[:, 1:2])).abs().max().item() < 1e-5


def test_discriminator_train_mode(ref, d_weights):
    x = inputs()
    b = O.discriminator_forward(x["disc_x"], x["disc_y"], d_weights, training=True)
    assert (ref["disc_train"] - b).abs().max().item() < 1e-6

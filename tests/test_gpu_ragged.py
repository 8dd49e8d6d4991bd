"""Ragged-batch inference (clips of different lengths in one forward pass) on the GPU.

Kernels: every *_varlen entry against the uniform entry run on each utterance's slice alone, with the padded rows of every input filled
with NaN (a kernel that read one would turn a valid row into NaN).  Lengths straddle the key tile (64), the 16-query warp tile, the
relative-position clamp (+-512) and T_max = 700.  Network and front end: TSCNet.forward(x, frames), the C entry, enhance_files /
evaluation on the 25 AudioSamples against the per-file path and the reference's own output."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda"
if torch.cuda.is_available():
    import cmgan_b200
    from cmgan_b200 import evaluation, module_abi, ops, signal
    from cmgan_b200._lib import lib
from conftest import GOLDEN

LENS = [4, 63, 64, 65, 513, 700]
T_MAX = 700


def _frames(lens=LENS):
    return torch.tensor(lens, dtype=torch.int32, device=DEV)


def _nan_pad(x, lens, axis=1):
    """x (B, T, ...): rows t >= lens[b] along ``axis`` set to NaN"""
    for b, n in enumerate(lens):
        x.select(0, b).narrow(axis - 1, n, x.shape[axis] - n).fill_(float("nan"))
    return x


def _ulp_close(a, b):
    a, b = a.double().cpu().numpy(), b.double().cpu().numpy()
    return bool(np.all(np.abs(a - b) <= np.spacing(np.abs(b).astype(np.float32)).astype(np.float64)))


# ================================================================================================= kernels
@pytest.mark.parametrize("axis", [0, 1])
@pytest.mark.parametrize("mode", ["fp32", "tf32"])
def test_attention_varlen(axis, mode):
    torch.manual_seed(0)
    F = 33
    B = len(LENS)
    qkv = _nan_pad(torch.randn(B, T_MAX, F, 192, device=DEV), LENS)
    E = torch.randn(1025, 16, device=DEV)
    ctx = torch.full((B, T_MAX, F, 64), float("nan"), device=DEV)
    lse = torch.full((B, T_MAX, F, 4), float("nan"), device=DEV)
    var, uni = ("cmgan_attention_fwd_varlen", "cmgan_attention_fwd") if mode == "fp32" else ("cmgan_attention_fwd_tf32_varlen", "cmgan_attention_fwd_tf32")
    ops.call(var, qkv, E, B, T_MAX, F, axis, _frames(), ctx, lse)
    for b, n in enumerate(LENS):
        q1 = qkv[b, :n].contiguous()
        c1 = torch.empty(n, F, 64, device=DEV)
        l1 = torch.empty(n, F, 4, device=DEV)
        ops.call(uni, q1, E, 1, n, F, axis, c1, l1)
        assert torch.isfinite(ctx[b, :n]).all() and torch.isfinite(lse[b, :n]).all(), (b, n)
        assert torch.equal(ctx[b, :n], c1) and torch.equal(lse[b, :n], l1), (b, n)


@pytest.mark.parametrize("axis", [0, 1])
def test_glu_dwconv_varlen(axis):
    torch.manual_seed(1)
    F = 33
    B = len(LENS)
    g = _nan_pad(torch.randn(B, T_MAX, F, 256, device=DEV), LENS)
    w = torch.randn(128, 31, device=DEV) * 0.2
    bias = torch.randn(128, device=DEV)
    out = torch.full((B, T_MAX, F, 128), float("nan"), device=DEV)
    ops.call("cmgan_glu_dwconv_fwd_varlen", g, w, bias, B, T_MAX, F, axis, _frames(), out)
    for b, n in enumerate(LENS):
        o1 = torch.empty(n, F, 128, device=DEV)
        ops.call("cmgan_glu_dwconv_fwd", g[b, :n].contiguous(), w, bias, 1, n, F, axis, o1, None)
        assert torch.isfinite(out[b, :n]).all() and torch.equal(out[b, :n], o1), (b, n)


@pytest.mark.parametrize("rpf,C", [(201, 64), (101, 64), (202, 64), (201, 1)])
def test_norm_stats_varlen(rpf, C):
    """InstanceNorm sites: rows per frame F (head, encoder block, mask m1 with C = 1), F2 (encoder conv_2, decoder blocks), 2 F2 (sp)"""
    torch.manual_seed(2)
    lens = [4, 65, 513, 700]
    B = len(lens)
    x = _nan_pad(torch.randn(B, T_MAX, rpf, C, device=DEV) * 2 + 0.5, lens)
    gamma, beta = torch.randn(C, device=DEV), torch.randn(C, device=DEV)

    def tables(xx, G, T, frames):
        sums = torch.zeros(G * C * 2, dtype=torch.float64, device=DEV)
        sc, sh, mu, rs = (torch.empty(G, C, device=DEV) for _ in range(4))
        if frames is None:
            ops.call("cmgan_norm_stats", xx, C, G, T * rpf, C, sums)
            ops.call("cmgan_norm_finalize", sums, T * rpf, G, C, 0, gamma, beta, None, None, 0.0, sc, sh, mu, rs, C)
        else:
            ops.call("cmgan_norm_stats_varlen", xx, C, G, T * rpf, C, frames, rpf, sums)
            ops.call("cmgan_norm_finalize_varlen", sums, frames, rpf, T, G, C, gamma, beta, sc, sh, mu, rs, C)
        return sc, sh

    sc, sh = tables(x, B, T_MAX, _frames(lens))
    for b, n in enumerate(lens):
        s1, h1 = tables(x[b, :n].contiguous(), 1, n, None)
        assert torch.isfinite(sc[b]).all() and torch.isfinite(sh[b]).all()
        assert _ulp_close(sc[b], s1[0]) and _ulp_close(sh[b], h1[0]), (b, n)        # double atomics: summation order differs


def test_frontend_varlen():
    """RMS scale, wrap + reflect pad and overlap-add against the per-row path (torch.cat wrap + cmgan_pad_reflect, cmgan_ola)"""
    torch.manual_seed(3)
    lens = [201, 250, 1234, 16000, 31999, 40000]
    B, Lmax = len(lens), max(lens)
    x = torch.randn(B, Lmax, device=DEV) * 0.1
    for b, n in enumerate(lens):
        x[b, n:] = float("nan")
    dl = torch.tensor(lens, dtype=torch.int32, device=DEV)
    c = torch.empty(B, device=DEV)
    ops.call("cmgan_rms_scale_varlen", x, x.stride(0), B, dl, c)
    nfr = [signal.clip_frames(n) for n in lens]
    T = max(nfr)
    Lp = 100 * (T - 1) + 400
    xp = torch.full((B, Lp), float("nan"), device=DEV)
    ops.call("cmgan_wrap_pad_reflect_varlen", x, x.stride(0), B, dl, c, xp, Lp)
    frames = torch.randn(B, T, 400, device=DEV)
    for b, n in enumerate(nfr):
        frames[b, n:] = float("nan")
    y = torch.full((B, 100 * (T - 1)), float("nan"), device=DEV)
    ops.call("cmgan_ola_varlen", frames, B, T, torch.tensor(nfr, dtype=torch.int32, device=DEV), signal._window_sq(x.device), c, y, y.stride(0))
    for b, n in enumerate(lens):
        row = x[b:b + 1, :n].contiguous()
        c1 = torch.empty(1, device=DEV)
        ops.call("cmgan_rms_scale", row, n, 1, n, c1)
        assert torch.equal(c[b:b + 1], c1), b
        Lw = (n + 99) // 100 * 100
        wrapped = torch.cat([row, row[:, :Lw - n]], dim=-1).contiguous()
        xp1 = torch.empty(1, Lw + 400, device=DEV)
        ops.call("cmgan_pad_reflect", wrapped, Lw, 1, Lw, c1, xp1, Lw + 400)
        assert torch.equal(xp[b, :Lw + 400], xp1[0]) and bool((xp[b, Lw + 400:] == 0).all()), b
        Tb = nfr[b]
        y1 = torch.empty(1, 100 * (Tb - 1), device=DEV)
        ops.call("cmgan_ola", frames[b, :Tb].contiguous(), 1, Tb, signal._inv_envelope(Tb, x.device), c1, y1, y1.stride(0))
        assert torch.isfinite(y[b, :100 * (Tb - 1)]).all() and torch.equal(y[b, :100 * (Tb - 1)], y1[0]), b


# ================================================================================================= network and public interface
def _random_model(seed=3):
    torch.manual_seed(seed)
    model = cmgan_b200.TSCNet(64, 201).to(DEV).eval()
    with torch.no_grad():
        for name, buf in model.named_buffers():             # non-trivial BatchNorm running statistics
            if name.endswith("running_mean"):
                buf.normal_(0.0, 0.3)
            elif name.endswith("running_var"):
                buf.uniform_(0.5, 1.5)
    return model


NET_LENS = [700, 513, 65, 4, 64]


@pytest.mark.parametrize("mode", ["fp32", "tf32"])
def test_tscnet_forward_frames(mode):
    ops.set_precision(mode)
    try:
        model = _random_model()
        torch.manual_seed(4)
        B = len(NET_LENS)
        x = _nan_pad(torch.randn(B, 2, T_MAX, 201, device=DEV), NET_LENS, axis=2)
        with torch.no_grad():
            fr, fi = model(x, frames=NET_LENS)
            worst, peak = 0.0, 0.0
            for b, n in enumerate(NET_LENS):
                r1, i1 = model(x[b:b + 1, :, :n])
                assert torch.isfinite(fr[b, :, :n]).all() and torch.isfinite(fi[b, :, :n]).all()
                worst = max(worst, float((fr[b, :, :n] - r1[0]).abs().max()), float((fi[b, :, :n] - i1[0]).abs().max()))
                peak = max(peak, float(r1.abs().max()), float(i1.abs().max()))
        bound = 1e-6 * max(1.0, peak) if mode == "fp32" else 1e-5 * peak
        print(f"[ragged-{mode}] TSCNet.forward(x, frames) vs per-utterance forward: max-abs {worst:.3e} (peak {peak:.3e}, bound {bound:.3e})")
        assert worst <= bound
    finally:
        ops.set_precision("fp32")


@pytest.mark.parametrize("mode", ["fp32", "tf32"])
def test_tscnet_fwd_varlen_c_entry(mode):
    ops.set_precision(mode)
    try:
        model = _random_model()
        torch.manual_seed(5)
        lens = [321, 97, 200]
        B, T = len(lens), max(lens)
        x = _nan_pad(torch.randn(B, 2, T, 201, device=DEV), lens, axis=2)
        p = 1 if mode == "tf32" else 0
        flat = module_abi.pack_params(model.state_dict(), DEV)
        with torch.no_grad():
            ref_r, ref_i = model(x, frames=lens)
        fr, fi = module_abi.tscnet_forward(flat, x, p, frames=_frames(lens))
        torch.cuda.synchronize()
        for b, n in enumerate(lens):
            tol = 1e-6 * max(1.0, float(ref_r[b, :, :n].abs().max()), float(ref_i[b, :, :n].abs().max()))
            assert float((fr[b, :, :n] - ref_r[b, :, :n]).abs().max()) <= tol and float((fi[b, :, :n] - ref_i[b, :, :n]).abs().max()) <= tol
        # frames == NULL is cmgan_tscnet_fwd
        xu = torch.randn(2, 2, 81, 201, device=DEV)
        ws = torch.empty(module_abi.workspace_bytes(2, 81, 201, p), dtype=torch.uint8, device=DEV)
        u_r, u_i = module_abi.tscnet_forward(flat, xu, p, workspace=ws)
        n_r, n_i = torch.empty_like(u_r), torch.empty_like(u_i)
        sb, sc, st, sf = xu.stride()
        lib().call("cmgan_tscnet_fwd_varlen", flat.data_ptr(), xu.data_ptr(), sb, sc, st, sf, 2, 81, 201, None, n_r.data_ptr(), n_i.data_ptr(),
                   ws.data_ptr(), ws.numel(), p, torch.cuda.current_stream().cuda_stream)
        tol = 1e-6 * max(1.0, float(u_r.abs().max()), float(u_i.abs().max()))      # same launches; the statistics sums are atomics
        assert float((u_r - n_r).abs().max()) <= tol and float((u_i - n_i).abs().max()) <= tol
    finally:
        ops.set_precision("fp32")


def test_ragged_errors():
    model = _random_model()
    x = torch.randn(2, 2, 50, 201, device=DEV)
    with torch.no_grad():
        with pytest.raises(ValueError, match="frame counts"):
            model(x, frames=[50, 0])
        with pytest.raises(ValueError, match="frame counts"):
            model(x, frames=[51, 3])
        with pytest.raises(ValueError, match="expected 2"):
            model(x, frames=[50])
    with pytest.raises(ValueError, match="inference only"):
        model(x, frames=[50, 3])                        # gradients enabled
    model.train()
    with torch.no_grad(), pytest.raises(ValueError, match="inference only"):
        model(x, frames=[50, 3])
    model.eval()
    ops.set_precision("tf32")
    old = ops.ATTN_TC
    ops.ATTN_TC = True
    try:
        with torch.no_grad(), pytest.raises(ValueError, match="CMGAN_ATTN_TC"):
            model(x, frames=[50, 3])
    finally:
        ops.ATTN_TC = old
        ops.set_precision("fp32")


# ================================================================================================= AudioSamples through the file front end
@pytest.fixture(scope="module")
def shipped(g_weights):
    m = cmgan_b200.TSCNet(64, 201)
    m.load_state_dict(g_weights, strict=True)
    return m.to(DEV).eval()


@pytest.fixture(scope="module")
def sample_dirs(tmp_path_factory):
    """the 25 AudioSamples as 16-bit wav files: noisy/ and clean/"""
    from scipy.io import wavfile
    z = np.load(os.path.join(GOLDEN, "audiosamples.npz"))
    off = np.concatenate([[0], np.cumsum(z["lengths"])])
    root = tmp_path_factory.mktemp("audiosamples")
    for sub in ("noisy", "clean"):
        os.mkdir(root / sub)
    for i, name in enumerate(z["names"]):
        for sub in ("noisy", "clean"):
            wavfile.write(str(root / sub / str(name)), 16000, z[sub][off[i]:off[i + 1]].astype(np.int16))
    return str(root / "noisy"), str(root / "clean"), z, off


def _enhance_files_vs_per_file(shipped, sample_dirs, mode, idx):
    noisy_dir, _, z, off = sample_dirs
    names = [str(z["names"][i]) for i in idx]
    paths = [os.path.join(noisy_dir, n) for n in names]
    lengths = [int(z["lengths"][i]) for i in idx]
    batches, solo = signal.plan_ragged(lengths, max_batch=16)
    assert solo == [] and any(len({lengths[i] for i in b}) > 1 for b in batches), "at least one batch mixes lengths"
    ops.set_precision(mode)
    try:
        out = evaluation.enhance_files(shipped, paths, max_batch=16)
        worst_self, worst_ref = 0.0, 0.0
        for k, i in enumerate(idx):
            noisy, _ = evaluation.read_wav(paths[k])
            solo_out = signal.enhance(shipped, noisy[:1].to(DEV)).cpu().numpy().astype(np.float64)
            got = out[paths[k]].astype(np.float64)
            ref = z["enhanced_ref"][off[i]:off[i + 1]].astype(np.float64)
            assert got.shape == solo_out.shape == ref.shape
            d_self = np.abs(got - solo_out).max() / np.abs(solo_out).max()
            d_ref = np.abs(got - ref).max()
            worst_self, worst_ref = max(worst_self, d_self), max(worst_ref, d_ref)
            assert d_self <= 1e-5, (names[k], d_self)
            assert d_ref <= 1e-3, (names[k], d_ref)
        print(f"[ragged-files-{mode}] {len(idx)} files in {len(batches)} batches: vs per-file max-abs/peak {worst_self:.3e}, "
              f"vs reference max-abs {worst_ref:.3e}")
    finally:
        ops.set_precision("fp32")


def test_enhance_files_audiosamples_tf32(shipped, sample_dirs):
    _enhance_files_vs_per_file(shipped, sample_dirs, "tf32", list(range(25)))


def test_enhance_files_audiosamples_fp32_subset(shipped, sample_dirs):
    _enhance_files_vs_per_file(shipped, sample_dirs, "fp32", [0, 8, 10, 12, 13])     # incl. the two longest and the two shortest files


def test_evaluation_matches_per_file_loop(shipped, sample_dirs):
    from cmgan_b200 import metrics as gpu_metrics
    noisy_dir, clean_dir, _, _ = sample_dirs
    ops.set_precision("tf32")
    try:
        got = evaluation.evaluation(shipped, noisy_dir, clean_dir, False, None)
        total = None
        names = evaluation.natural_sorted(os.listdir(noisy_dir))
        for name in names:
            est, length = evaluation.enhance_one_track(shipped, os.path.join(noisy_dir, name), None, 16000 * 16)
            clean, _ = evaluation.read_wav(os.path.join(clean_dir, name))
            m = np.asarray(gpu_metrics.ssnr_stoi(clean[0, :length].to(DEV), torch.from_numpy(est).to(DEV)), dtype=np.float64)
            total = m if total is None else total + m
        want = total / len(names)
    finally:
        ops.set_precision("fp32")
    print(f"[ragged-evaluation] SSNR/STOI ragged {got} vs per-file {want}")
    assert np.all(np.abs(got - want) <= 1e-6 * np.abs(want))

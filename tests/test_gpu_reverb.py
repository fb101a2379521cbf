"""Reverb view through the FFT overlap-save entry ``rb_reverb`` / ``Engine.reverb`` (SURVEY.md 8f-4): parity with the float64
arithmetic of audio_augmentor/reverb.py:39-42 across the partition and block boundaries, ragged and bad rows, NaN semantics,
agreement with the direct FIR path and stream ordering. The argument checks run before any CUDA call, so the first test needs
no device."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import rawboost_oracle as orc  # noqa: E402  (checker only)

P = 8192  # taps per partition = output samples per block (rb_reverb.cu kP)


def test_reverb_argument_checks_and_workspace_bound():
    from scl_deepfake_audio_detection_b200 import _lib
    lib = _lib.load()
    wb = lib.rb_reverb_workspace_bytes
    assert wb(0, 8000) == 0
    assert wb(2, 8000) > wb(1, 8000) > 0
    assert wb(1, 16000) > wb(1, 8000) and wb(1, P + 1) > wb(1, P)
    assert wb(64, 32000) >= 64 * 4 * 8192 * 8  # four spectra of 8192 complex bins per row
    # x, len, B, ld, rir, rir_off, y, ld_out, out_len, workspace, workspace_bytes, stream
    assert lib.rb_reverb(None, None, 2, 64, None, None, None, 64, None, None, 0, None) == -1
    assert lib.rb_reverb(16, 16, 2, 64, 16, 16, 32, 64, None, 256, 1 << 30, None) == -1   # out_len missing
    assert lib.rb_reverb(16, 16, 2, 63, 16, 16, 32, 64, 16, 256, 1 << 30, None) == -2
    assert lib.rb_reverb(16, 16, 2, 64, 16, 16, 32, 66, 16, 256, 1 << 30, None) == -2
    assert lib.rb_reverb(16, 16, 2, 64, 16, 16, 16, 64, 16, 256, 1 << 30, None) == -1   # x == y
    assert lib.rb_reverb(16, 16, 2, 64, 16, 16, 32, 64, 16, None, 0, None) == -3
    assert lib.rb_reverb(16, 16, 2, 64, 16, 16, 32, 64, 16, 256, 100, None) == -3
    assert lib.rb_reverb(16, 16, 2, 64, 16, 16, 32, 64, 16, 128, 1 << 30, None) == -2     # workspace not 256-byte aligned
    assert lib.rb_reverb(None, None, 0, 64, None, None, None, 64, None, None, 0, None) == 0
    assert lib.rb_reverb(None, None, -1, 64, None, None, None, 64, None, None, 0, None) == -1


# ---------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def eng():
    from scl_deepfake_audio_detection_b200.engine import Engine
    assert torch.cuda.is_available()
    return Engine(0)


def _signal(rs, L, loud=False):
    return ((0.9 if loud else 0.05) * rs.standard_normal(L)).astype(np.float32)


def _rir(rs, K):
    return (rs.standard_normal(K) * np.exp(-np.arange(K) / max(1.0, K / 6.0))).astype(np.float32)


def _reference(x, h):
    """float64 normWav(np.convolve(x, h), 1); scipy's float64 FFT convolution stands in for the largest cases."""
    if x.shape[0] * h.shape[0] <= 64600 * 4097:
        return orc.reverb_convolve(x, h)
    from scipy.signal import fftconvolve
    r = fftconvolve(x.astype(np.float64), h.astype(np.float64))
    return r / np.max(np.abs(r))


def _upload(eng, waves, rirs, ld=None):
    from scl_deepfake_audio_detection_b200 import reverb
    x, ln = eng.pack_waveforms(waves, ld=ld)
    taps, off = reverb.pack_rirs(eng, rirs)
    return x, ln, taps, off


PARITY = [(64600, 8000), (64600, 16000), (64600, 32000),                      # K = 8000 / 16000 / 32000: 1 / 2 / 4 partitions
          (64600, 1), (64600, P - 1), (64600, P), (64600, P + 1), (64600, 2 * P + 1),  # partition boundaries
          (2 * P - 1, 700), (2 * P, 700), (2 * P + 1, 700), (2 * P - 700 + 1, 700),     # L at a block boundary +- 1; output = two blocks
          (3 * P - 1, 1), (3 * P + 1, 1),                                      # third block boundary
          (300, 2049), (1000, 9000),                                           # K > L
          (1, 700), (1, 1), (1, 9000),                                         # L = 1
          (211000, 16000)]


@pytest.mark.gpu
@pytest.mark.parametrize("L,K", PARITY)
def test_reverb_fft_matches_float64_convolution(eng, L, K):
    rs = np.random.RandomState(L * 7 + K)
    waves = [_signal(rs, L), _signal(rs, L, loud=True)]
    rirs = [_rir(rs, K), _rir(rs, K)]
    x, ln, taps, off = _upload(eng, waves, rirs)
    y, out_len = eng.reverb(x, ln, taps, off)
    y, out_len = y.cpu().numpy(), out_len.cpu().numpy()
    worst = 0.0
    for u in range(2):
        ref = _reference(waves[u], rirs[u])
        assert out_len[u] == L + K - 1 == ref.shape[0]
        got = y[u, :out_len[u]]
        err = float(np.max(np.abs(got.astype(np.float64) - ref)))
        worst = max(worst, err)
        assert err <= 1e-5, (u, err)
        assert abs(float(np.max(np.abs(got))) - 1.0) <= 1e-6
    print(f"rb_reverb L={L} K={K}: max-abs error vs float64 {worst:.2e}")


@pytest.mark.gpu
def test_reverb_ragged_batch_with_empty_row_keeps_sentinels(eng):
    rs = np.random.RandomState(11)
    lens = [64600, 0, 5000, 1, 20000, 64600, 7]
    ks = [513, 800, 2 * P + 3, 4000, 1, 16000, 12000]
    waves = [_signal(rs, n) for n in lens]
    rirs = [_rir(rs, k) for k in ks]
    x, ln, taps, off = _upload(eng, waves, rirs)
    want = [n + k - 1 if n else 0 for n, k in zip(lens, ks)]
    ld_out = (max(want) + 100) // 4 * 4
    sentinel = -7.25
    out = torch.full((len(lens), ld_out), sentinel, dtype=torch.float32, device=eng.device)
    y, out_len = eng.reverb(x, ln, taps, off, out=out)
    assert y is out
    y, out_len = y.cpu().numpy(), out_len.cpu().numpy()
    assert out_len.tolist() == want
    for u, n in enumerate(want):
        assert np.all(y[u, n:] == sentinel), u
        if n:
            ref = _reference(waves[u], rirs[u])
            assert np.max(np.abs(y[u, :n].astype(np.float64) - ref)) <= 1e-5, u


@pytest.mark.gpu
def test_reverb_bad_rows_are_reported_and_untouched(eng):
    from scl_deepfake_audio_detection_b200 import reverb
    rs = np.random.RandomState(12)
    waves = [_signal(rs, 3000), _signal(rs, 3000), _signal(rs, 3000), _signal(rs, 10000)]
    rirs = [_rir(rs, 100), np.zeros(0, np.float32), _rir(rs, 200), _rir(rs, 100)]
    x, ln, taps, off = _upload(eng, waves, rirs)
    ld_out = 3400  # row 3 needs 10099 samples
    sentinel = 3.5
    out = torch.full((4, ld_out), sentinel, dtype=torch.float32, device=eng.device)
    y, out_len = eng.reverb(x, ln, taps, off, out=out)
    y, out_len = y.cpu().numpy(), out_len.cpu().numpy()
    assert out_len.tolist() == [3099, -1, 3199, -1]
    assert np.all(y[1] == sentinel) and np.all(y[3] == sentinel)
    for u in (0, 2):
        assert np.max(np.abs(y[u, :out_len[u]].astype(np.float64) - _reference(waves[u], rirs[u]))) <= 1e-5
        assert np.all(y[u, out_len[u]:] == sentinel)
    with pytest.raises(ValueError):
        eng.reverb(x, ln, taps, off)                      # sized from the lengths: the empty impulse response is reported
    with pytest.raises(ValueError):
        reverb.reverb_device(eng, x, ln, rirs, ld_out=ld_out)
    with pytest.raises(ValueError):
        reverb.reverb_device(eng, x[3:], ln[3:], rirs[3:], ld_out=ld_out)  # ld_out too small only


@pytest.mark.gpu
def test_reverb_max_taps_sizes_the_workspace(eng):
    """max_taps sets the partitions the workspace holds: rows within them are computed, a longer one is reported (-1)."""
    rs = np.random.RandomState(16)
    waves = [_signal(rs, 20000), _signal(rs, 20000)]
    rirs = [_rir(rs, P), _rir(rs, P + 5)]
    x, ln, taps, off = _upload(eng, waves, rirs)
    ld_out = (20000 + P + 8) // 4 * 4
    y, out_len = eng.reverb(x, ln, taps, off, ld_out=ld_out, max_taps=P)
    y, out_len = y.cpu().numpy(), out_len.cpu().numpy()
    assert out_len.tolist() == [20000 + P - 1, -1]
    assert np.max(np.abs(y[0, :out_len[0]].astype(np.float64) - _reference(waves[0], rirs[0]))) <= 1e-5
    assert np.all(y[1] == 0)
    y, out_len = eng.reverb(x, ln, taps, off, ld_out=ld_out, max_taps=P + 5)
    assert out_len.cpu().numpy().tolist() == [20000 + P - 1, 20000 + P + 4]
    assert np.max(np.abs(y[1, :20000 + P + 4].cpu().numpy().astype(np.float64) - _reference(waves[1], rirs[1]))) <= 1e-5


@pytest.mark.gpu
def test_reverb_zero_and_nan_rows_follow_numpy(eng):
    rs = np.random.RandomState(13)
    zero = np.zeros(5000, np.float32)
    nan = _signal(rs, 5000)
    nan[1234] = np.nan
    good = _signal(rs, 5000)
    rirs = [_rir(rs, 3000) for _ in range(3)]
    x, ln, taps, off = _upload(eng, [zero, nan, good], rirs)
    y, out_len = eng.reverb(x, ln, taps, off)
    y, out_len = y.cpu().numpy(), out_len.cpu().numpy()
    with np.errstate(invalid="ignore"):
        ref_zero = orc.reverb_convolve(zero, rirs[0])
        ref_nan = orc.reverb_convolve(nan, rirs[1])
    assert np.all(np.isnan(ref_zero)) and np.all(np.isnan(ref_nan))
    assert np.all(np.isnan(y[0, :out_len[0]])) and np.all(np.isnan(y[1, :out_len[1]]))
    assert np.max(np.abs(y[2, :out_len[2]].astype(np.float64) - orc.reverb_convolve(good, rirs[2]))) <= 1e-5


@pytest.mark.gpu
def test_reverb_fft_agrees_with_direct_path(eng):
    from scl_deepfake_audio_detection_b200 import reverb
    rs = np.random.RandomState(14)
    lens = [64600, 30000, 64600, 1200]
    ks = [8000, 513, P + 1, 2049]
    waves = [_signal(rs, n, loud=bool(u % 2)) for u, n in enumerate(lens)]
    rirs = [_rir(rs, k) for k in ks]
    yd, ld_direct = reverb.reverb_batch(eng, waves, rirs)
    x, ln = eng.pack_waveforms(waves)
    yf, ld_fft = reverb.reverb_device(eng, x, ln, rirs)
    ld_direct, ld_fft = ld_direct.cpu().numpy(), ld_fft.cpu().numpy()
    assert ld_direct.tolist() == ld_fft.tolist()
    yd, yf = yd.cpu().numpy(), yf.cpu().numpy()
    for u, n in enumerate(ld_fft):
        assert np.max(np.abs(yd[u, :n].astype(np.float64) - yf[u, :n])) <= 1e-5, u


@pytest.mark.gpu
def test_reverb_on_a_side_stream_without_host_sync(eng):
    rs = np.random.RandomState(15)
    waves = [_signal(rs, 64600) for _ in range(6)]
    rirs = [_rir(rs, k) for k in (8000, 16000, 1, 3000, 9000, 700)]
    x, ln, taps, off = _upload(eng, waves, rirs)
    ld_out = (64600 + 16000) // 4 * 4
    y0, n0 = eng.reverb(x, ln, taps, off, ld_out=ld_out)
    torch.cuda.synchronize()
    side = torch.cuda.Stream(eng.device)
    side.wait_stream(torch.cuda.current_stream(eng.device))
    with torch.cuda.stream(side):
        torch.cuda.set_sync_debug_mode("error")  # any torch-side host synchronisation inside the call raises
        try:
            y1, n1 = eng.reverb(x, ln, taps, off, ld_out=ld_out)
        finally:
            torch.cuda.set_sync_debug_mode("default")
    side.synchronize()
    assert torch.equal(n0, n1)
    assert torch.equal(y0, y1)

"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle and the reference's golden outputs.

Tolerances (BASELINE.json north_star): integer work bit-exact; ISD / normWav on float32 input bit-exact; every
FIR-based result max-abs <= 1e-5 against the float64 oracle on peak-normalised scale.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from oracle import rawboost_oracle as orc  # noqa: E402  (checker only)

TOL = 1e-5
ARGS = orc.make_args()


@pytest.fixture(scope="module")
def eng():
    from scl_deepfake_audio_detection_b200.engine import Engine
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return Engine(0)


@pytest.fixture(scope="module")
def P():
    from scl_deepfake_audio_detection_b200 import plans
    return plans


def run_batch(eng, P, algo, waves, seeds, args=ARGS):
    """Draw plans (host, reference stream order), run the whole batch on the device, return per-utterance arrays."""
    bp = P.draw_batch([w.shape[0] for w in waves], 16000, args, algo, seeds=seeds)
    x, ln = eng.pack_waveforms(waves, ld=bp.ld)
    dp = eng.upload_plan(bp)
    y = eng.process(algo, x, ln, dp)
    torch.cuda.synchronize()
    y = y.cpu().numpy()
    return [y[u, :w.shape[0]] for u, w in enumerate(waves)], bp


def oracle_batch(algo, waves, seeds, args=ARGS):
    out = []
    for w, s in zip(waves, seeds):
        np.random.seed(int(s))
        out.append(np.asarray(orc.process(w, 16000, args, algo)))
    return out


def max_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b))) if a.size else 0.0


# ---------------------------------------------------------------------------------------------------------
# operators
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [1, 2, 3, 4, 11, 64, 491])
def test_filter_fir_golden(eng, golden, K):
    arrays, _ = golden
    from scl_deepfake_audio_detection_b200 import RawBoost as rb
    x, b, ref = arrays[f"fir_x_K{K}"], arrays[f"fir_b_K{K}"], arrays[f"fir_y_K{K}"]
    y = rb.filterFIR(x, b)
    assert y.dtype == np.float32 and y.shape == ref.shape
    assert max_err(y, ref) <= TOL * max(1.0, np.abs(ref).max())


@pytest.mark.parametrize("K,L", [(513, 3000), (700, 9000), (1500, 5200), (2049, 2600), (491, 1), (7, 2561), (24, 2560),
                                 (7, 3584), (24, 3585), (131, 7167), (131, 7168), (491, 7169), (51, 10752), (271, 11008), (1001, 14337)])
def test_filter_fir_long_and_edge(eng, K, L):
    """Filters longer than one staged segment (512 taps) and tile-boundary lengths -- of the 2560-output tile of the bank and
    of the 3584-output tile the plain filter runs with, including rows whose middle tiles take the batched staging path while
    the first and last ones take the zero-filling one."""
    rs = np.random.RandomState(K * 7 + L)
    x = rs.standard_normal(L).astype(np.float32)
    b = rs.standard_normal(K) / np.sqrt(K)
    from scl_deepfake_audio_detection_b200 import RawBoost as rb
    y = rb.filterFIR(x, b)
    ref = orc.filter_fir_closed_form(x, b.astype(np.float32))
    assert max_err(y, ref) <= TOL * max(1.0, np.abs(ref).max())
    assert max_err(orc.filter_fir(x, b), ref) <= 1e-6  # the closed form is the reference formula


def test_filter_fir_ragged_batch(eng):
    """One rb_filter_fir launch over rows of different lengths and tap counts: every row equals the closed form of filterFIR on
    its own samples, whatever lies in the row's padding beyond its length (the batched staging path reads whole float4 chunks
    only inside [0, len); the edge tiles zero-fill), and nothing is written beyond a row's length."""
    lens = [1, 5, 2559, 3583, 3584, 3585, 7168, 9001, 12000, 14336, 14337, 20000]
    Ks = [3, 51, 131, 7, 491, 24, 271, 700, 11, 1, 99, 513]
    ld = 20000
    rs = np.random.RandomState(99)
    x = rs.standard_normal((len(lens), ld)).astype(np.float32) * 100.0  # the padding is loud garbage
    taps = [(rs.standard_normal(K) / np.sqrt(K)).astype(np.float32) for K in Ks]
    off = np.concatenate([[0], np.cumsum(Ks)]).astype(np.int32)
    rows = [rs.uniform(-1, 1, L).astype(np.float32) for L in lens]
    for r, (L, row) in enumerate(zip(lens, rows)):
        x[r, :L] = row
    out = torch.full((len(lens), ld), 7.0, dtype=torch.float32, device="cuda")
    y = eng.filter_fir(torch.from_numpy(x).cuda(), torch.tensor(lens, dtype=torch.int32, device="cuda"),
                       torch.from_numpy(np.concatenate(taps)).cuda(), torch.from_numpy(off).cuda(), out=out).cpu().numpy()
    for r, (L, row, t) in enumerate(zip(lens, rows, taps)):
        ref = orc.filter_fir_closed_form(row, t)
        assert max_err(y[r, :L], ref) <= TOL * max(1.0, np.abs(ref).max()), f"row {r} (L={L}, K={t.shape[0]})"
        assert np.all(y[r, L:] == 7.0), f"row {r}: samples beyond the row's length were written"


def test_filter_fir_linearity_full_size(eng):
    """Size-independent property at BASELINE size: FIR(a*x1 + x2) == a*FIR(x1) + FIR(x2) (to fp32 rounding)."""
    B, L = 64, 64600
    rs = np.random.RandomState(1)
    x1 = rs.uniform(-1, 1, (B, L)).astype(np.float32)
    x2 = rs.uniform(-1, 1, (B, L)).astype(np.float32)
    np.random.seed(3)
    taps = [orc.draw_notch_taps(5, 20, 8000, 100, 1000, 10, 100, 0, 0, 16000).astype(np.float32) for _ in range(B)]
    off = np.concatenate([[0], np.cumsum([t.shape[0] for t in taps])]).astype(np.int32)
    td = torch.from_numpy(np.concatenate(taps)).cuda()
    od = torch.from_numpy(off).cuda()
    ln = torch.full((B,), L, dtype=torch.int32, device="cuda")
    f = lambda a: eng.filter_fir(torch.from_numpy(a).cuda(), ln, td, od).cpu().numpy()
    lhs = f((0.5 * x1 + x2).astype(np.float32))
    rhs = 0.5 * f(x1) + f(x2)
    assert max_err(lhs, rhs) <= 2e-6 * max(1.0, np.abs(rhs).max())
    # spot-check three rows against the oracle
    for u in (0, 31, 63):
        assert max_err(f(x1)[u], orc.filter_fir_closed_form(x1[u], taps[u])) <= TOL


def test_normwav_bit_exact(eng, golden):
    arrays, _ = golden
    from scl_deepfake_audio_detection_b200 import RawBoost as rb
    for tag in ("quiet", "loud"):
        x = arrays[f"norm_x_{tag}"]
        for always in (0, 1):
            y = rb.normWav(x, always)
            assert y.dtype == np.float32
            assert np.array_equal(y, arrays[f"norm_y{always}_{tag}"]), (tag, always)
    x = arrays["norm_x_quiet"]
    assert rb.normWav(x, 0) is x
    y = rb.normWav(arrays["norm_x_loud"], 0)
    assert np.array_equal(rb.normWav(y, 0), y)  # idempotent once the peak is 1


# ---------------------------------------------------------------------------------------------------------
# dispatcher vs the reference's golden outputs (small) and the oracle (full size)
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("algo", list(range(0, 9)))
def test_dispatcher_matches_reference_golden(eng, golden, algo):
    arrays, meta = golden
    from conftest import stream_digest
    from scl_deepfake_audio_detection_b200 import RawBoost as rb
    for loud in (0, 1):
        for u in (0, 1):
            key = f"algo{algo}_loud{loud}_u{u}"
            x = orc.synth_utterance(u, 16000, bool(loud))
            x0 = x.copy()
            np.random.seed(orc.seed_for(u))
            y = rb.process_Rawboost_feature(x, 16000, ARGS, algo)
            assert stream_digest() == meta["cases"][key]["stream"], f"{key}: RNG stream diverged from the reference"
            assert np.array_equal(x, x0), "input mutated"
            ref = arrays[key]
            assert y.shape == ref.shape
            if algo == 0:
                assert y is x
            elif algo == 2:
                assert y.dtype == np.float32 and np.array_equal(y, ref), f"{key}: ISD must be bit-exact on float32 input"
            else:
                assert y.dtype == np.float32
                assert max_err(y, ref) <= TOL, f"{key}: max-abs {max_err(y, ref):.3e}"


def test_ragged_batch_matches_oracle_and_golden(eng, P, golden):
    arrays, _ = golden
    lens = [1, 2, 37, 600, 4097, 2560, 2561, 16000]
    waves = [orc.synth_utterance(7, L, False) for L in lens]
    seeds = [orc.seed_for(7)] * len(lens)
    got, _ = run_batch(eng, P, 5, waves, seeds)
    want = oracle_batch(5, waves, seeds)
    for L, g, w in zip(lens, got, want):
        assert g.shape == (L,)
        assert max_err(g, w) <= TOL, f"L={L}: {max_err(g, w):.3e}"
        key = f"ragged_algo5_L{L}"
        if key in arrays:
            assert max_err(g, arrays[key]) <= TOL


@pytest.mark.parametrize("algo", [1, 2, 3, 4, 5, 6, 7, 8])
def test_full_length_batch_matches_oracle(eng, P, golden, algo):
    """64600-sample utterances, both amplitude variants, in one batch; also the reference's own summaries."""
    _, meta = golden
    us = [0, 3, 5, 0, 3, 5]
    loud = [0, 0, 0, 1, 1, 1]
    waves = [orc.synth_utterance(u, 64600, bool(l)) for u, l in zip(us, loud)]
    seeds = [orc.seed_for(u) for u in us]
    got, _ = run_batch(eng, P, algo, waves, seeds)
    want = oracle_batch(algo, waves, seeds)
    for u, l, g, w in zip(us, loud, got, want):
        if algo == 2:
            assert np.array_equal(g, w), "ISD must be bit-exact on float32 input"
        else:
            assert max_err(g, w) <= TOL, f"algo {algo} u{u} loud{l}: {max_err(g, w):.3e}"
        key = f"algo{algo}_loud{l}_u{u}"
        if key in meta["full"]:
            s = meta["full"][key]
            assert max_err(g[np.array(s["probe_idx"])], s["probe_val"]) <= TOL
            assert abs(float(np.abs(g.astype(np.float64)).max()) - max(abs(s["min"]), abs(s["max"]))) <= TOL


def test_isd_indices_are_integer_exact(eng, P):
    """The samples ISD changes are exactly the drawn permutation prefix (quiet input: no rescaling)."""
    x = orc.synth_utterance(11, 64600, False)
    np.random.seed(orc.seed_for(11))
    plan = orc.draw_isd_plan(64600, 10)
    got, bp = run_batch(eng, P, 2, [x], [orc.seed_for(11)])
    assert np.array_equal(bp.isd_idx, plan.idx.astype(np.int32)) and bp.isd_off.tolist() == [0, plan.idx.shape[0]]
    changed = np.flatnonzero(got[0] != x)
    assert set(changed.tolist()) <= set(plan.idx.tolist())       # nothing outside the drawn positions moves
    assert changed.shape[0] >= plan.idx.shape[0] - 8             # (a gain can round to a no-op on a tiny sample)
    np.random.seed(orc.seed_for(11))
    assert np.array_equal(got[0], orc.isd(x, 10, 2))


def test_algo5_properties_at_config_size(eng, P):
    """BASELINE config 3 shape (algo 5, 64600 samples) at a batch the oracle cannot cover: size-independent checks."""
    B = 256
    waves = [orc.synth_utterance(u, 64600, bool(u % 2)) for u in range(B)]
    seeds = [orc.seed_for(u) for u in range(B)]
    got, bp = run_batch(eng, P, 5, waves, seeds)
    got1, _ = run_batch(eng, P, 1, waves, seeds)  # same seeds -> same LnL taps
    for u in range(B):
        y5, y1 = got[u], got1[u]
        assert np.all(np.isfinite(y5)) and np.abs(y5).max() <= 1.0 + 1e-6
        assert np.abs(y1).max() <= 1.0 + 1e-6
        idx = bp.isd_idx[bp.isd_off[u]:bp.isd_off[u + 1]]
        untouched = np.ones(64600, dtype=bool)
        untouched[idx] = False
        peak = np.abs(y5).max()
        # untouched samples are the LnL output up to the one common ISD rescale (a divisor >= 1)
        ratio = np.abs(y1[untouched]).max() / max(np.abs(y5[untouched]).max(), 1e-30)
        assert ratio >= 1.0 - 1e-6
        np.testing.assert_allclose(y5[untouched] * ratio, y1[untouched], rtol=0, atol=2e-6)
        if ratio > 1.0 + 1e-6:
            assert abs(peak - 1.0) <= 1e-6  # rescaled => the new peak is exactly 1
    # spot-check a few utterances against the oracle
    for u in (0, 1, 100, 255):
        np.random.seed(seeds[u])
        assert max_err(got[u], orc.process(waves[u], 16000, ARGS, 5)) <= TOL
    # determinism: same plan, same bits
    again, _ = run_batch(eng, P, 5, waves[:8], seeds[:8])
    for u in range(8):
        assert np.array_equal(again[u], got[u])


def test_host_entry_point_equals_device_path(eng, P):
    waves = [orc.synth_utterance(u, 64600, bool(u % 2)) for u in range(4)]
    seeds = [orc.seed_for(u) for u in range(4)]
    for algo in (1, 3, 5, 7):
        got, bp = run_batch(eng, P, algo, waves, seeds)
        xh = np.zeros((4, bp.ld), dtype=np.float32)
        for u, w in enumerate(waves):
            xh[u, :w.shape[0]] = w
        yh = eng.process_host(algo, xh, bp)
        for u, w in enumerate(waves):
            assert np.array_equal(yh[u, :w.shape[0]], got[u])
        h2d, d2h = eng.last_host_traffic()
        assert d2h == xh.nbytes and h2d >= xh.nbytes


def test_nondefault_arguments(eng, P):
    """Longer cascades (K up to 991 -> two staged segments), more bands, N_f = 3, other ISD / SSI knobs."""
    args = orc.make_args(nBands=6, maxCoeff=200, N_f=3, P=25, g_sd=3, SNRmin=5, SNRmax=15, minG=-3, maxG=2)
    waves = [orc.synth_utterance(u, 20000 + 17 * u, bool(u % 2)) for u in range(4)]
    seeds = [orc.seed_for(40 + u) for u in range(4)]
    for algo in (4, 5, 8):
        got, _ = run_batch(eng, P, algo, waves, seeds, args)
        want = oracle_batch(algo, waves, seeds, args)
        for g, w in zip(got, want):
            assert max_err(g, w) <= TOL, f"algo {algo}: {max_err(g, w):.3e}"


def test_error_codes(eng):
    import ctypes as C
    from scl_deepfake_audio_detection_b200 import _lib
    lib = _lib.load()
    x = torch.zeros(2, 64, device="cuda")
    y = torch.zeros_like(x)
    ln = torch.full((2,), 64, dtype=torch.int32, device="cuda")
    ws = eng.workspace(2, 64)
    wp = C.c_void_p(eng._ws_ptr(ws))
    # algo 5 without a plan
    assert lib.rb_process(5, x.data_ptr(), ln.data_ptr(), 2, 64, None, y.data_ptr(), wp, ws.numel() - 256, None) == -5
    # ld not a multiple of 4
    assert lib.rb_process(5, x.data_ptr(), ln.data_ptr(), 2, 63, None, y.data_ptr(), wp, ws.numel() - 256, None) == -2
    # workspace too small
    assert lib.rb_process(1, x.data_ptr(), ln.data_ptr(), 2, 64, None, y.data_ptr(), wp, 16, None) == -3
    # in-place is refused for real algos
    assert lib.rb_process(1, x.data_ptr(), ln.data_ptr(), 2, 64, None, x.data_ptr(), wp, ws.numel() - 256, None) == -1
    with pytest.raises(_lib.RawBoostLibraryError):
        _lib.check(-5, "rb_process")
    assert lib.rb_launch_count() > 0


def test_dropin_patches_loader_namespace(eng):
    """A stand-in loader module that binds the operator names like the reference loaders do (augall_3.py:10)."""
    import types
    from scl_deepfake_audio_detection_b200 import dropin, RawBoost as rb
    fake = types.ModuleType("fake_loader")
    for n in dropin.OPERATORS + dropin.DISPATCH:
        setattr(fake, n, lambda *a, **k: (_ for _ in ()).throw(AssertionError("reference path called")))
    dropin.patch_loader(fake)
    x = orc.synth_utterance(2, 8000, False)
    np.random.seed(5)
    y = fake.RawBoost12(x, orc.make_args(online_aug=True, aug_dir="/nonexistent"), 16000, audio_path="/a/b.wav")
    np.random.seed(5)
    want = orc.process(x, 16000, ARGS, 5)
    assert max_err(y, want) <= TOL and fake.LnL_convolutive_noise is rb.LnL_convolutive_noise


# ---------------------------------------------------------------------------------------------------------
# round-2 fixtures from the unmodified reference: inputs above full scale, float64 / zero / NaN inputs, long utterances
# ---------------------------------------------------------------------------------------------------------
def test_inputs_above_full_scale_match_reference(eng, golden2):
    """Stand-alone ISD must apply its impulses to the RAW x and normalise afterwards (RawBoost.py:76-84): with max|x| > 1 a
    first normalisation of the input changes which sample carries the peak. Algos 2, 7, 8 and the operator itself."""
    from conftest import sha1_of, stream_digest
    from scl_deepfake_audio_detection_b200 import RawBoost as rb
    arrays, meta = golden2
    for key, s in meta["over"].items():
        algo, u = int(key.split("_")[1][4:]), int(key.split("_")[2][1:])
        x = orc.overscale_utterance(u, 16000)
        np.random.seed(orc.seed_for(50 + u))
        y = rb.process_Rawboost_feature(x, 16000, ARGS, algo)
        assert stream_digest() == s["stream"], key
        assert max_err(y[np.array(s["probe_idx"])], s["probe_val"]) <= TOL, key
        assert abs(float(y.astype(np.float64).max()) - s["max"]) <= TOL and abs(float(y.astype(np.float64).min()) - s["min"]) <= TOL, key
        if algo == 2:
            assert sha1_of(y) == s["sha1_f32"], "ISD must be bit-exact on float32 input, also above full scale"
        if key in arrays:
            assert max_err(y, arrays[key]) <= TOL, key
    for u in (0, 1):
        np.random.seed(orc.seed_for(50 + u))
        assert np.array_equal(rb.ISD_additive_noise(orc.overscale_utterance(u, 16000), 10, 2), arrays[f"over_op_isd_u{u}"])


def test_float64_zero_and_nan_inputs_match_reference(eng, golden2):
    from scl_deepfake_audio_detection_b200 import RawBoost as rb
    arrays, meta = golden2
    x64 = 0.3 * np.random.RandomState(31).standard_normal(4000)
    for algo in (1, 2, 3, 5):  # float64 in: the reference computes in float64; here the input is rounded to float32 first
        np.random.seed(orc.seed_for(60))
        y = rb.process_Rawboost_feature(x64, 16000, ARGS, algo)
        assert y.dtype == np.float32 and max_err(y, arrays[f"f64_algo{algo}"]) <= TOL, algo
    z = np.zeros(1000, dtype=np.float32)
    xn = orc.synth_utterance(9, 3000, True).copy()
    xn[100] = np.nan
    for algo in (1, 2, 3, 5):
        np.random.seed(orc.seed_for(61))
        assert np.array_equal(rb.process_Rawboost_feature(z, 16000, ARGS, algo), arrays[f"zeros_algo{algo}"], equal_nan=True), algo
        np.random.seed(orc.seed_for(62))
        y = rb.process_Rawboost_feature(xn, 16000, ARGS, algo)
        ref = arrays[f"nan_algo{algo}"]
        assert np.array_equal(np.isnan(y), np.isnan(ref)), f"algo {algo}: NaN must propagate exactly like numpy"
        assert np.allclose(y, ref, rtol=0, atol=TOL, equal_nan=True)
    assert np.array_equal(rb.normWav(z, 0), z) and np.isnan(rb.normWav(z, 1)).all()  # 0/0 stays NaN, as in the reference
    assert np.array_equal(rb.normWav(xn, 0), arrays["nan_norm0"], equal_nan=True)
    assert np.isnan(rb.normWav(xn, 1)).all() and np.isnan(arrays["nan_norm1"]).all()


@pytest.mark.parametrize("L", [65537, 100000, 211000])
def test_long_utterances_match_reference(eng, P, golden2, L):
    """Un-cropped utterances, as the loaders feed them (asvspoof_2019_augall_3.py:105-117): ISD / normWav bit-exact by digest,
    algo 5 within tolerance of the reference's summary and of the oracle."""
    from conftest import sha1_of
    from scl_deepfake_audio_detection_b200 import RawBoost as rb
    _, meta = golden2
    for loud in (0, 1):
        x = orc.synth_utterance(70 + loud, L, bool(loud))
        if loud:
            x = (x * 2.0).astype(np.float32)
        for algo in (2, 5):
            s = meta["long"][f"long_algo{algo}_L{L}_loud{loud}"]
            got, _ = run_batch(eng, P, algo, [x], [orc.seed_for(70)])
            y = got[0]
            if algo == 2:
                assert sha1_of(y) == s["sha1_f32"], (L, loud)
            else:
                assert max_err(y[np.array(s["probe_idx"])], s["probe_val"]) <= TOL
                assert abs(float(np.abs(y.astype(np.float64)).max()) - max(abs(s["min"]), abs(s["max"]))) <= TOL
                np.random.seed(orc.seed_for(70))
                assert max_err(y, orc.process(x, 16000, ARGS, 5)) <= TOL
        for always in (0, 1):
            assert sha1_of(rb.normWav(x, always)) == meta["long"][f"long_norm{always}_L{L}_loud{loud}"]["sha1_f32"]


def test_ragged_batch_with_long_rows(eng, P):
    """One batch mixing lengths on both sides of 65536 and of the streaming tile (4096): algos 2, 5 and 8 vs the oracle."""
    lens = [211000, 70001, 65537, 65536, 4097, 4096, 4095, 5, 1]
    waves = [orc.synth_utterance(20 + i, n, bool(i % 2)) * (2.0 if i % 3 == 0 else 1.0) for i, n in enumerate(lens)]
    waves = [w.astype(np.float32) for w in waves]
    seeds = [orc.seed_for(300 + i) for i in range(len(lens))]
    for algo in (2, 5, 8):
        got, _ = run_batch(eng, P, algo, waves, seeds)
        want = oracle_batch(algo, waves, seeds)
        for n, g, w in zip(lens, got, want):
            if algo == 2:
                assert np.array_equal(g, w), f"algo 2, L={n}"
            else:
                assert max_err(g, w) <= TOL, f"algo {algo}, L={n}: {max_err(g, w):.3e}"


def test_normwav_in_place_and_batched(eng):
    """rb_normwav with y == x (the copy is skipped) equals the out-of-place result, rows on both sides of the threshold."""
    rs = np.random.RandomState(4)
    lens = [64600, 64600, 30000, 4096, 7]
    waves = [(a * rs.uniform(-1, 1, n)).astype(np.float32) for a, n in zip((0.5, 3.0, 1.0001, 0.999, 2.0), lens)]
    x, ln = eng.pack_waveforms(waves)
    for always in (False, True):
        y = eng.normwav(x, ln, always)
        z = x.clone()
        eng.normwav(z, ln, always, out=z)
        torch.cuda.synchronize()
        assert torch.equal(y, z)
        for u, w in enumerate(waves):
            assert np.array_equal(y[u, :lens[u]].cpu().numpy(), orc.norm_wav(w, always)), (always, u)


def test_rawboost12_offline_cache_branch(eng, tmp_path, monkeypatch):
    """``RawBoost12`` with ``online_aug`` off (asvspoof_2019_augall_3.py:365-374): compute once and write ``<aug_dir>/RawBoost12/<utt>``
    as 16-bit PCM, afterwards load the file instead of computing (no draw is consumed then). soundfile / librosa are absent
    here exactly as in the survey container, so the two calls the branch makes are served by stand-ins."""
    import sys
    import types
    from conftest import stream_digest
    from scl_deepfake_audio_detection_b200 import RawBoost as rb
    store = {}
    sf = types.ModuleType("soundfile")
    sf.write = lambda path, wav, sr, subtype=None: store.__setitem__(path, (np.clip(np.round(np.asarray(wav) * 32768.0), -32768, 32767).astype(np.int16), sr, subtype))
    lr = types.ModuleType("librosa")
    lr.load = lambda path, sr=None, mono=True: (store[path][0].astype(np.float32) / 32768.0, sr)
    monkeypatch.setitem(sys.modules, "soundfile", sf)
    monkeypatch.setitem(sys.modules, "librosa", lr)
    monkeypatch.setattr("os.path.exists", lambda p, _orig=__import__("os").path.exists: p in store or _orig(p))
    args = orc.make_args(online_aug=False, aug_dir=str(tmp_path))
    x = orc.synth_utterance(5, 9000, False)
    np.random.seed(17)
    first = rb.RawBoost12(x, args, 16000, audio_path="/corpus/bonafide/LA_T_1.wav")
    after_first = stream_digest()
    np.random.seed(17)
    want = orc.process(x, 16000, ARGS, 5)
    assert max_err(first, want) <= TOL
    (path, (pcm, sr, subtype)), = store.items()
    assert path.endswith("RawBoost12/LA_T_1.wav") and sr == 16000 and subtype == "PCM_16"
    np.random.seed(17)
    second = rb.RawBoost12(x, args, 16000, audio_path="/corpus/bonafide/LA_T_1.wav")
    np.random.seed(17)
    untouched = stream_digest()
    assert np.array_equal(second, pcm.astype(np.float32) / 32768.0) and max_err(second, first) <= 1.0 / 32768.0
    np.random.seed(17)
    rb.RawBoost12(x, args, 16000, audio_path="/corpus/bonafide/LA_T_1.wav")
    assert stream_digest() == untouched and after_first != untouched  # the cached call draws nothing


def test_bench_dump_outputs_is_the_timed_result_and_repeats(tmp_path):
    """``bench.py --dump-outputs`` from the command line: the dumped rows are the algo-5 result of the headline batch (checked
    against the oracle), ``--steps`` is the number of timed steps reported, and two runs with different step counts dump the
    same arrays."""
    import json
    import os
    import subprocess
    import sys
    from conftest import ROOT
    from scl_deepfake_audio_detection_b200 import workload
    B, L = 16, 64600
    runs = []
    for steps in (1, 3):
        out = tmp_path / f"s{steps}"
        cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "3", "--batch", str(B), "--no-e2e",
               "--no-cpu", "--no-configs", "--dump-outputs", str(out)]
        res = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr[-2000:]
        line = json.loads(res.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps and line["config"]["batch_per_gpu"] == B
        runs.append((np.load(out / "rows.npy"), np.load(out / "y.npy")))
    (rows, y), (rows3, y3) = runs
    assert rows.dtype == np.float64 and rows.tolist() == list(range(B)) and y.dtype == np.float32 and y.shape == (B, L)
    assert np.array_equal(rows, rows3) and np.array_equal(y, y3)
    for u in (0, B - 1):
        np.random.seed(workload.seed_for(u))
        ref = orc.process(workload.synth_utterance(u, L, bool(u % 2)), 16000, ARGS, 5)
        assert max_err(y[u], ref) <= TOL, u

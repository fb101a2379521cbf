"""Pin the CPU oracle (oracle/rawboost_oracle.py) to the reference's own outputs.

The fixtures were produced by importing /root/reference unmodified (oracle/make_golden.py).
Plans / indices / stream positions must match bit-exactly; float64 waveforms to 1e-12.
"""
import numpy as np
import pytest

from conftest import stream_digest
from oracle import rawboost_oracle as orc

ARGS = orc.make_args()
TOL = 1e-12


def _case_keys(meta, section):
    return sorted(meta[section].keys())


def test_dispatcher_all_algos_match_reference(golden):
    arrays, meta = golden
    for key in _case_keys(meta, "cases"):
        c = meta["cases"][key]
        x = orc.synth_utterance(c["u"], c["L"], bool(c["loud"]))
        x_before = x.copy()
        np.random.seed(orc.seed_for(c["u"]))
        y = orc.process(x, 16000, ARGS, c["algo"])
        ref = arrays[key]
        assert np.asarray(y).dtype == ref.dtype, key
        assert np.asarray(y).shape == ref.shape, key
        assert np.array_equal(x, x_before), f"{key}: input mutated"
        assert (y is x) == c["same_object"], key
        np.testing.assert_allclose(y, ref, rtol=0, atol=TOL, err_msg=key)
        assert stream_digest() == c["stream"], f"{key}: RNG stream diverged"


def test_full_length_summaries_match_reference(golden):
    _, meta = golden
    for key in _case_keys(meta, "full"):
        s = meta["full"][key]
        algo = int(key.split("_")[0][4:])
        loud = int(key.split("_")[1][4:])
        u = int(key.split("_")[2][1:])
        x = orc.synth_utterance(u, 64600, bool(loud))
        np.random.seed(orc.seed_for(u))
        y = np.asarray(orc.process(x, 16000, ARGS, algo))
        assert str(y.dtype) == s["dtype"], key
        y = y.astype(np.float64)
        assert abs(y.sum() - s["sum"]) <= 1e-9, key
        assert abs((y * y).sum() - s["sumsq"]) <= 1e-9 * max(1.0, s["sumsq"]), key
        assert abs(y.min() - s["min"]) <= TOL and abs(y.max() - s["max"]) <= TOL, key
        assert int(np.argmax(np.abs(y))) == s["argmax_abs"], key
        np.testing.assert_allclose(y[np.array(s["probe_idx"])], s["probe_val"], rtol=0, atol=TOL)
        assert stream_digest() == s["stream"], key


def test_notch_taps_match_reference(golden):
    arrays, meta = golden
    for u in range(6):
        np.random.seed(orc.seed_for(u))
        b = orc.draw_notch_taps(5, 20, 8000, 100, 1000, 10, 100, 0, 0, 16000)
        ref = arrays[f"notch_u{u}"]
        assert b.shape[0] == meta["ops"][f"notch_u{u}"]["K"] and b.shape[0] % 2 == 1
        np.testing.assert_allclose(b, ref, rtol=0, atol=1e-15)
        assert stream_digest() == meta["ops"][f"notch_u{u}"]["stream"]
    np.random.seed(99)
    b = orc.draw_notch_taps(5, 20, 8000, 100, 1000, 10, 100, -5, -20, 16000)
    np.testing.assert_allclose(b, arrays["notch_gain"], rtol=0, atol=1e-15)
    assert stream_digest() == meta["ops"]["notch_gain"]["stream"]


@pytest.mark.parametrize("K", [1, 2, 3, 4, 11, 64, 491])
def test_filter_fir_matches_reference_and_closed_form(golden, K):
    arrays, _ = golden
    x, b, ref = arrays[f"fir_x_K{K}"], arrays[f"fir_b_K{K}"], arrays[f"fir_y_K{K}"]
    y = orc.filter_fir(x, b)
    assert y.dtype == ref.dtype and y.shape == ref.shape == x.shape
    np.testing.assert_allclose(y, ref, rtol=0, atol=TOL)
    np.testing.assert_allclose(orc.filter_fir_closed_form(x, b), ref, rtol=0, atol=1e-12)


def test_norm_wav_matches_reference(golden):
    arrays, _ = golden
    for tag in ("quiet", "loud"):
        x = arrays[f"norm_x_{tag}"]
        for always in (0, 1):
            y = orc.norm_wav(x, always)
            ref = arrays[f"norm_y{always}_{tag}"]
            assert y.dtype == ref.dtype
            assert np.array_equal(y, ref)
    x = arrays["norm_x_quiet"]
    assert orc.norm_wav(x, 0) is x  # untouched input is returned as the same object


def test_rand_range_matches_reference(golden):
    _, meta = golden
    r = meta["ops"]["randRange"]
    np.random.seed(3)
    f = orc.rand_range(20, 8000, 0)
    assert isinstance(f, np.ndarray) and f.shape == (1,) and float(f[0]) == r["float"]
    i = orc.rand_range(10, 100, 1)
    assert isinstance(i, int) and i == r["int"]
    assert float(orc.rand_range(-5, -20, 0)[0]) == r["reversed"]
    assert stream_digest() == r["stream"]


def test_operators_match_reference(golden):
    arrays, _ = golden
    for u in (0, 1):
        x = orc.synth_utterance(u, 16000, False)
        np.random.seed(orc.seed_for(u))
        np.testing.assert_allclose(orc.lnl(x, 5, 5, 20, 8000, 100, 1000, 10, 100, 0, 0, 5, 20, 16000),
                                   arrays[f"op_lnl_u{u}"], rtol=0, atol=TOL)
        np.random.seed(orc.seed_for(u))
        y = orc.isd(x, 10, 2)
        assert y.dtype == np.float32 and np.array_equal(y, arrays[f"op_isd_u{u}"])
        np.random.seed(orc.seed_for(u))
        np.testing.assert_allclose(orc.ssi(x, 10, 40, 5, 20, 8000, 100, 1000, 10, 100, 0, 0, 16000),
                                   arrays[f"op_ssi_u{u}"], rtol=0, atol=TOL)


def test_lnl_consumes_80_uniforms_and_isd_plan_is_integer_exact():
    np.random.seed(11)
    plan = orc.draw_lnl_plan(5, 5, 20, 8000, 100, 1000, 10, 100, 0, 0, 5, 20, 16000)
    after = stream_digest()
    np.random.seed(11)
    np.random.uniform(size=80)
    assert stream_digest() == after
    for t in plan.taps:
        assert 51 <= t.shape[0] <= 491 and t.shape[0] % 2 == 1
    np.random.seed(12)
    p = orc.draw_isd_plan(64600, 10)
    assert p.idx.dtype == np.int64 and len(np.unique(p.idx)) == len(p.idx) == int(64600 * (p.beta / 100))
    assert p.idx.min() >= 0 and p.idx.max() < 64600 and np.all(np.abs(p.f_r) < 1)


# ---------------------------------------------------------------------------------------------------------
# the step after the path: batch_pad_for_multiview and the item assembly (SURVEY.md 8f-1/f-2)
# ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def mv_golden():
    import json
    import os
    from conftest import GOLDEN_DIR
    arrays = np.load(os.path.join(GOLDEN_DIR, "multiview_golden.npz"))
    with open(os.path.join(GOLDEN_DIR, "multiview_golden.json")) as f:
        return arrays, json.load(f)


def test_oracle_multiview_pad_matches_reference(mv_golden):
    from conftest import stream_digest
    arrays, meta = mv_golden
    assert len(meta["pad"]) == 32
    for key, m in meta["pad"].items():
        flat = arrays[m["input"]]
        views, o = [], 0
        for n in m["lens"]:
            views.append(flat[o:o + n].reshape(n, 1))
            o += n
        np.random.seed(m["seed"])
        out = orc.batch_pad_for_multiview(views, 16000, m["length"], random_trim_nosil=m["trim"], repeat_pad=m["repeat_pad"])
        out = np.concatenate(out, axis=1)
        assert out.shape == arrays[key].shape and out.shape[0] == m["out_len"], key
        assert np.array_equal(out.astype(np.float64), arrays[key].astype(np.float64)), key
        assert stream_digest() == m["stream"], f"{key}: the crop draw must consume the stream exactly like the reference"


def test_oracle_multiview_item_matches_reference(mv_golden):
    """RNG order of Dataset_for.__getitem__: RawBoost on the 3 vocoded copies, then on the anchor, then the shared crop."""
    from conftest import stream_digest
    arrays, meta = mv_golden
    args = orc.make_args()
    for key, m in meta["item"].items():
        item = int(key[4:])
        waves = [orc.synth_utterance(m["first_wave"] + k, m["L"] + 37 * k, bool(k % 2)) for k in range(4)]
        np.random.seed(m["seed"])
        aug_voc = [orc.process(w, 16000, args, 5) for w in waves[1:]]
        aug_anchor = orc.process(waves[0], 16000, args, 5)
        views = [waves[0], aug_anchor] + waves[1:] + aug_voc
        out = orc.batch_pad_for_multiview([np.expand_dims(v, 1) for v in views], 16000, m["trim"], random_trim_nosil=True,
                                          repeat_pad=True)
        out = np.concatenate(out, axis=1).astype(np.float32)
        assert list(out.shape) == m["shape"]
        assert np.max(np.abs(out.astype(np.float64) - arrays[key])) <= 1e-6, (key, item)
        assert stream_digest() == m["stream"]


# ---------------------------------------------------------------------------------------------------------
# round-2 fixtures: edge inputs, long utterances, reverb, whole Dataset items
# ---------------------------------------------------------------------------------------------------------
def _check_summary(y, s, key):
    y = np.asarray(y).astype(np.float64)
    assert abs(y.min() - s["min"]) <= TOL and abs(y.max() - s["max"]) <= TOL, key
    assert int(np.argmax(np.abs(y))) == s["argmax_abs"], key
    np.testing.assert_allclose(y[np.array(s["probe_idx"])], s["probe_val"], rtol=0, atol=TOL, err_msg=key)


def test_oracle_inputs_above_full_scale(golden2):
    """ISD applies its impulses to the raw x and normalises afterwards (RawBoost.py:76-84)."""
    from conftest import sha1_of
    arrays, meta = golden2
    for key, s in meta["over"].items():
        algo, u = int(key.split("_")[1][4:]), int(key.split("_")[2][1:])
        x = orc.overscale_utterance(u, 16000)
        assert np.abs(x).max() > 2.0
        np.random.seed(orc.seed_for(50 + u))
        y = np.asarray(orc.process(x, 16000, ARGS, algo))
        _check_summary(y, s, key)
        assert stream_digest() == s["stream"], key
        if algo == 2:
            assert y.dtype == np.float32 and sha1_of(y) == s["sha1_f32"]
        if key in arrays:
            assert np.max(np.abs(y.astype(np.float64) - arrays[key])) <= 1e-6, key
    for u in (0, 1):
        np.random.seed(orc.seed_for(50 + u))
        assert np.array_equal(orc.isd(orc.overscale_utterance(u, 16000), 10, 2), arrays[f"over_op_isd_u{u}"])


def test_oracle_float64_zero_and_nan_inputs(golden2):
    arrays, meta = golden2
    x64 = 0.3 * np.random.RandomState(31).standard_normal(4000)
    for algo in (1, 2, 3, 5):
        np.random.seed(orc.seed_for(60))
        y = np.asarray(orc.process(x64, 16000, ARGS, algo))
        assert str(y.dtype) == meta["f64"][f"f64_algo{algo}"]["dtype"] == "float64"
        assert np.max(np.abs(y - arrays[f"f64_algo{algo}"])) <= 1e-6
        assert stream_digest() == meta["f64"][f"f64_algo{algo}"]["stream"]
    z = np.zeros(1000, dtype=np.float32)
    xn = orc.synth_utterance(9, 3000, True).copy()
    xn[100] = np.nan
    with np.errstate(invalid="ignore", divide="ignore"):
        for algo in (1, 2, 3, 5):
            np.random.seed(orc.seed_for(61))
            y = np.asarray(orc.process(z, 16000, ARGS, algo)).astype(np.float32)
            assert np.array_equal(y, arrays[f"zeros_algo{algo}"], equal_nan=True)
            np.random.seed(orc.seed_for(62))
            y = np.asarray(orc.process(xn, 16000, ARGS, algo)).astype(np.float32)
            assert int(np.isnan(y).sum()) == meta["nan"][f"nan_algo{algo}"]["nan_count"]
            assert np.allclose(y, arrays[f"nan_algo{algo}"], rtol=0, atol=1e-6, equal_nan=True)
        assert np.array_equal(orc.norm_wav(z, 0), arrays["zeros_norm0"]) and np.isnan(arrays["zeros_norm1"]).all()
        assert np.isnan(orc.norm_wav(z, 1)).all()
        assert np.array_equal(orc.norm_wav(xn, 0), arrays["nan_norm0"], equal_nan=True)
        assert np.array_equal(orc.norm_wav(xn, 1), arrays["nan_norm1"], equal_nan=True)


@pytest.mark.parametrize("L", [65537, 100000, 211000])
def test_oracle_long_utterances(golden2, L):
    """What the loaders really feed RawBoost: the un-cropped utterance (asvspoof_2019_augall_3.py:105-117)."""
    from conftest import sha1_of
    _, meta = golden2
    for loud in (0, 1):
        x = orc.synth_utterance(70 + loud, L, bool(loud))
        if loud:
            x = (x * 2.0).astype(np.float32)
        for algo in (2, 5):
            s = meta["long"][f"long_algo{algo}_L{L}_loud{loud}"]
            np.random.seed(orc.seed_for(70))
            y = np.asarray(orc.process(x, 16000, ARGS, algo))
            _check_summary(y, s, (algo, L, loud))
            assert stream_digest() == s["stream"]
            if algo == 2:
                assert sha1_of(y) == s["sha1_f32"]
        for always in (0, 1):
            assert sha1_of(orc.norm_wav(x, always)) == meta["long"][f"long_norm{always}_L{L}_loud{loud}"]["sha1_f32"]


def test_oracle_reverb_matches_reference(golden2):
    """audio_augmentor/reverb.py:33-44 (np.convolve in float32 there; the oracle restates it in float64)."""
    arrays, meta = golden2
    rir = arrays["reverb_rir"]
    for tag, data in (("speech", orc.synth_utterance(80, 20000, False)), ("loud", orc.synth_utterance(81, 7001, True))):
        y = orc.reverb_convolve(data, rir)
        ref = arrays[f"reverb_{tag}"]
        assert y.shape == ref.shape == (meta["reverb"][f"reverb_{tag}"]["len"],)
        assert np.max(np.abs(y - ref)) <= 1e-5 and abs(np.abs(y).max() - 1.0) <= 1e-12


def test_oracle_dataset_item_matches_reference(golden2):
    """The whole ``Dataset_for.__getitem__`` (asvspoof_2019_augall_3.py:103-146): draws, view order, crop, labels."""
    arrays, meta = golden2
    g = meta["getitem"]
    for idx in (0, 3):
        m = g[f"getitem{idx}"]
        np.random.seed(m["seed"])
        utt, data, label = orc.dataset_item(idx, g["ids"], orc.corpus_wave, orc.make_args(), m["vocoders"], m["num_additional_real"],
                                            m["trim_length"])
        assert utt == m["utt"] and list(data.shape) == m["shape"]
        assert np.max(np.abs(data.astype(np.float64) - arrays[f"getitem{idx}_data"])) <= 1e-6
        assert np.array_equal(label, arrays[f"getitem{idx}_label"])
        assert stream_digest() == m["stream"]


def _same_as_reference(a, stream_a, b, algo):
    """Result ``b`` (and the stream state after it) of the numpy restatement against the reference's ``a``: bit for bit where no
    filter runs, within TOL where float64 FIR sums are ordered differently (<= 1 ulp of the peak, measured 2.2e-16)."""
    assert stream_digest() == stream_a, algo
    assert np.asarray(a).dtype == np.asarray(b).dtype, algo
    if algo in (0, 2):
        assert np.array_equal(a, b), algo
    else:
        np.testing.assert_allclose(a, b, rtol=0, atol=TOL, err_msg=str(algo))


def test_compiled_reference_matches_the_oracle(golden):
    """The reference's own code and the numpy restatement agree on every algo, quiet and loud, and consume the global stream
    identically; normWav too. On every checkout against the reference's outputs stored in tests/golden (oracle/make_golden.py);
    where ``oracle/_ref`` (the reference's bytecode, oracle/build_ref.py, which the CPU arm of the bench times) can be built,
    also against the live reference on further inputs."""
    import warnings
    arrays, meta = golden
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for algo in range(0, 9):
            for loud in (0, 1):
                for u in (0, 1):
                    key = f"algo{algo}_loud{loud}_u{u}"
                    x = orc.synth_utterance(u, meta["cases"][key]["L"], bool(loud))
                    np.random.seed(orc.seed_for(u))
                    _same_as_reference(arrays[key], meta["cases"][key]["stream"], orc.process(x, 16000, ARGS, algo), algo)
        assert np.array_equal(arrays["norm_y0_loud"], orc.norm_wav(arrays["norm_x_loud"], 0))
        from oracle import build_ref
        if not build_ref.available():
            build_ref.build()  # needs the reference's sources
        ref = build_ref.load()
        if ref is None:
            return
        ops, dispatch = ref
        for algo in range(0, 9):
            for loud in (False, True):
                x = orc.synth_utterance(3, 8000, loud)
                np.random.seed(77)
                a = dispatch(x, 16000, ARGS, algo)
                sa = stream_digest()
                np.random.seed(77)
                _same_as_reference(a, sa, orc.process(x, 16000, ARGS, algo), algo)
        x = orc.synth_utterance(4, 5000, True)
        assert np.array_equal(ops.normWav(x * 3, 0), orc.norm_wav(x * 3, 0))


def test_item_view_rows_and_labels_follow_the_dataset_order():
    """Row table / label vector of the in-place assembly == the view order and labels of Dataset_for.__getitem__
    (asvspoof_2019_augall_3.py:133, 143-146): anchor, augmented anchor, additional bona fide, vocoded, augmented vocoded."""
    from scl_deepfake_audio_detection_b200 import multiview
    rows = multiview.item_view_rows(2, 3, [[8, 9], [10, 11]])
    # per item the inputs sit as [voc0, voc1, voc2, anchor]; negative = the RawBoost result of that row
    assert rows.tolist() == [[3, -4, 8, 9, 0, 1, 2, -1, -2, -3], [7, -8, 10, 11, 4, 5, 6, -5, -6, -7]]
    assert multiview.item_view_rows(1, 3).tolist() == [[3, -4, 0, 1, 2, -1, -2, -3]]
    assert multiview.item_labels(3, 2).tolist() == [1, 1, 1, 1, 0, 0, 0, 0, 0, 0]
    _, _, label = orc.dataset_item(0, orc.CORPUS_IDS, orc.corpus_wave, orc.make_args(), orc.CORPUS_VOCODERS, 2, 4000)
    assert label.tolist() == multiview.item_labels(3, 2).tolist()

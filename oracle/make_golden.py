#!/usr/bin/env python3
"""Generate ``tests/golden/*`` from the UNMODIFIED reference, imported from /root/reference.

Run in the build container only (``/root/reference`` does not exist on the GPU box):

    python oracle/make_golden.py            # rewrites tests/golden/rawboost_golden.* (npz parts of at most 1 MB)
    python oracle/make_golden.py --multiview   # tests/golden/multiview_golden.*
    python oracle/make_golden.py --round2      # tests/golden/round2_golden.* (edge inputs, long utterances, reverb, __getitem__)

The reference's loader modules import packages that are absent here (librosa, soundfile, pydub,
torchaudio.io, torchaudio.sox_effects); five empty stub modules are registered first so that
``datautils.asvspoof_2019_augall_3`` imports unmodified (SURVEY.md 8c). Nothing is copied from the
reference: the fixtures hold *outputs* of its functions on seeded synthetic inputs, plus the state
of the global numpy stream after each call (to pin how many draws each operator consumes).

Inputs are not stored: they are regenerated from ``synth_utterance(u, L, loud)`` and
``np.random.seed(seed_for(u))`` (oracle/rawboost_oracle.py), exactly as the tests do.
"""
import hashlib
import json
import os
import sys
import tempfile
import types
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = "/root/reference"
OUT = os.path.join(ROOT, "tests", "golden")

sys.path.insert(0, ROOT)
from oracle import golden_files  # noqa: E402
from oracle.rawboost_oracle import (CORPUS_IDS, CORPUS_VOCODERS, corpus_wave, make_args, overscale_utterance, seed_for,  # noqa: E402
                                    synth_utterance)


def import_reference():
    """Import the reference operators and one loader's dispatcher, unmodified."""
    import importlib
    for name in ("librosa", "soundfile", "pydub", "torchaudio", "torchaudio.functional",
                 "torchaudio.io", "torchaudio.sox_effects"):
        try:
            importlib.import_module(name)
        except Exception:
            sys.modules[name] = types.ModuleType(name)
    for mod, attr, val in (("pydub", "AudioSegment", type("AudioSegment", (), {})),
                           ("torchaudio.io", "AudioEffector", type("AudioEffector", (), {})),
                           ("torchaudio.sox_effects", "apply_effects_tensor", lambda *a, **k: None)):
        if not hasattr(sys.modules[mod], attr):
            setattr(sys.modules[mod], attr, val)
    for sub in ("functional", "io", "sox_effects"):
        if not hasattr(sys.modules["torchaudio"], sub):
            setattr(sys.modules["torchaudio"], sub, sys.modules["torchaudio." + sub])
    sys.path.insert(0, REF)
    cwd = os.getcwd()
    os.chdir(tempfile.mkdtemp())  # the loader's logging.basicConfig drops errors.log into CWD
    try:
        import datautils.RawBoost as rb
        import datautils.asvspoof_2019_augall_3 as loader
    finally:
        os.chdir(cwd)
    assert loader.LnL_convolutive_noise is rb.LnL_convolutive_noise
    return rb, loader


def stream_digest():
    """Compact fingerprint of the global legacy stream (position + key hash + gauss cache)."""
    name, key, pos, has_gauss, cached = np.random.get_state()
    return {
        "pos": int(pos),
        "key_sha1": hashlib.sha1(np.asarray(key, dtype=np.uint32).tobytes()).hexdigest(),
        "has_gauss": int(has_gauss),
        "cached_gaussian": float(cached),
    }


def summarise(y):
    y64 = np.asarray(y, dtype=np.float64)
    probe = np.linspace(0, y64.shape[0] - 1, 64).astype(np.int64)
    return {
        "dtype": str(np.asarray(y).dtype),
        "sum": float(y64.sum()),
        "sumsq": float((y64 * y64).sum()),
        "min": float(y64.min()),
        "max": float(y64.max()),
        "argmax_abs": int(np.argmax(np.abs(y64))),
        "probe_idx": probe.tolist(),
        "probe_val": y64[probe].tolist(),
    }


def main():
    warnings.simplefilter("ignore", DeprecationWarning)  # int(ndarray) at RawBoost.py:17
    rb, loader = import_reference()
    os.makedirs(OUT, exist_ok=True)
    args = make_args()
    arrays = {}
    meta = {"numpy": np.__version__, "cases": {}, "ops": {}, "full": {}}
    import scipy
    meta["scipy"] = scipy.__version__

    # ---- dispatcher, every algo, two amplitude variants, short utterances (arrays kept) ----
    L_small = 16000
    for algo in range(0, 9):
        for loud in (0, 1):
            for u in (0, 1):
                x = synth_utterance(u, L_small, bool(loud))
                np.random.seed(seed_for(u))
                y = loader.process_Rawboost_feature(x, 16000, args, algo)
                key = f"algo{algo}_loud{loud}_u{u}"
                arrays[key] = np.asarray(y)
                meta["cases"][key] = {"algo": algo, "loud": loud, "u": u, "L": L_small,
                                      "dtype": str(np.asarray(y).dtype), "stream": stream_digest(),
                                      "same_object": bool(y is x)}

    # ---- ragged / tiny lengths through the dispatcher (algo 5) ----
    for L in (1, 2, 37, 600, 4097):
        x = synth_utterance(7, L, False)
        np.random.seed(seed_for(7))
        y = loader.process_Rawboost_feature(x, 16000, args, 5)
        key = f"ragged_algo5_L{L}"
        arrays[key] = np.asarray(y)
        meta["cases"][key] = {"algo": 5, "loud": 0, "u": 7, "L": L, "dtype": str(np.asarray(y).dtype),
                              "stream": stream_digest(), "same_object": False}

    # ---- operator surface ----
    for u in range(6):
        np.random.seed(seed_for(u))
        b = rb.genNotchCoeffs(5, 20, 8000, 100, 1000, 10, 100, 0, 0, 16000)
        arrays[f"notch_u{u}"] = b
        meta["ops"][f"notch_u{u}"] = {"K": int(b.shape[0]), "stream": stream_digest()}
    # low>high gain range, as LnL uses from order 2 on
    np.random.seed(99)
    b = rb.genNotchCoeffs(5, 20, 8000, 100, 1000, 10, 100, -5, -20, 16000)
    arrays["notch_gain"] = b
    meta["ops"]["notch_gain"] = {"K": int(b.shape[0]), "stream": stream_digest()}

    rs = np.random.RandomState(5)
    for K in (1, 2, 3, 4, 11, 64, 491):
        xs = rs.standard_normal(300).astype(np.float32)
        bs = rs.standard_normal(K)
        arrays[f"fir_x_K{K}"] = xs
        arrays[f"fir_b_K{K}"] = bs
        arrays[f"fir_y_K{K}"] = rb.filterFIR(xs, bs)
    for tag, v in (("quiet", 0.5), ("loud", 3.0)):
        xs = (v * rs.uniform(-1, 1, 257)).astype(np.float32)
        arrays[f"norm_x_{tag}"] = xs
        arrays[f"norm_y0_{tag}"] = rb.normWav(xs, 0)
        arrays[f"norm_y1_{tag}"] = rb.normWav(xs, 1)
    np.random.seed(3)
    meta["ops"]["randRange"] = {
        "float": float(rb.randRange(20, 8000, 0)[0]),
        "int": int(rb.randRange(10, 100, 1)),
        "reversed": float(rb.randRange(-5, -20, 0)[0]),
        "stream": stream_digest(),
    }
    for u in (0, 1):
        x = synth_utterance(u, L_small, False)
        np.random.seed(seed_for(u))
        arrays[f"op_lnl_u{u}"] = rb.LnL_convolutive_noise(x, 5, 5, 20, 8000, 100, 1000, 10, 100, 0, 0, 5, 20, 16000)
        np.random.seed(seed_for(u))
        arrays[f"op_isd_u{u}"] = rb.ISD_additive_noise(x, 10, 2)
        np.random.seed(seed_for(u))
        arrays[f"op_ssi_u{u}"] = rb.SSI_additive_noise(x, 10, 40, 5, 20, 8000, 100, 1000, 10, 100, 0, 0, 16000)

    # ---- BASELINE-size utterances (64600): summaries only ----
    for algo in (1, 2, 3, 4, 5, 8):
        for loud in (0, 1):
            for u in (0, 3):
                x = synth_utterance(u, 64600, bool(loud))
                np.random.seed(seed_for(u))
                y = loader.process_Rawboost_feature(x, 16000, args, algo)
                s = summarise(y)
                s["stream"] = stream_digest()
                meta["full"][f"algo{algo}_loud{loud}_u{u}"] = s

    paths = golden_files.save(OUT, "rawboost_golden", arrays)
    with open(os.path.join(OUT, "rawboost_golden.json"), "w") as f:
        json.dump(meta, f, indent=1, sort_keys=True)
    size = sum(os.path.getsize(p) for p in paths)
    print(f"wrote {len(arrays)} arrays ({size/1e6:.2f} MB in {len(paths)} files) and {len(meta['cases'])+len(meta['full'])} case records to {OUT}")


def main_multiview():
    """Fixtures for the step right after the path (SURVEY.md 8f-1/f-2): ``batch_pad_for_multiview``
    (core_scripts/data_io/wav_augmentation.py:209-282) and the view assembly of ``Dataset_for.__getitem__``
    (datautils/asvspoof_2019_augall_3.py:103-146), produced by the unmodified reference."""
    warnings.simplefilter("ignore", DeprecationWarning)
    rb, loader = import_reference()
    nii = loader.nii_wav_aug
    arrays, meta = {}, {"pad": {}, "item": {}}
    rs = np.random.RandomState(11)
    # ---- batch_pad_for_multiview: every branch (first view shorter / longer than the target, zero / repeat pad, crop) ----
    lens_sets = {"firstlong": [333, 150, 200, 90, 1000], "firstshort": [150, 333, 40, 150], "firstequal": [200, 10, 700],
                 "single": [517]}
    case = 0
    for tag, lens in lens_sets.items():
        views = [rs.standard_normal((n, 1)).astype(np.float32) for n in lens]
        arrays[f"pad_in_{tag}"] = np.concatenate([v[:, 0] for v in views])
        for length in (200, 64):
            for repeat_pad in (False, True):
                for trim in (False, True):
                    np.random.seed(1000 + case)
                    out = nii.batch_pad_for_multiview([v.copy() for v in views], 16000, length, random_trim_nosil=trim,
                                                      repeat_pad=repeat_pad)
                    key = f"pad_{tag}_L{length}_r{int(repeat_pad)}_t{int(trim)}"
                    arrays[key] = np.concatenate(out, axis=1)
                    meta["pad"][key] = {"lens": lens, "length": length, "repeat_pad": repeat_pad, "trim": trim, "seed": 1000 + case,
                                        "input": f"pad_in_{tag}", "out_len": int(out[0].shape[0]), "stream": stream_digest()}
                    case += 1
    # ---- one Dataset item, RNG order of __getitem__: 3 vocoded RawBoost12, anchor RawBoost12, (choice), crop ----
    args = make_args(online_aug=True, aug_dir="")
    for item, (L, trim_len) in enumerate(((16000, 12000), (9000, 12000))):
        waves = [synth_utterance(100 + 4 * item + k, L + 37 * k, bool(k % 2)) for k in range(4)]  # anchor, 3 vocoded
        np.random.seed(4242 + item)
        aug_voc = [loader.RawBoost12(w, args, 16000, audio_path="x") for w in waves[1:]]
        aug_anchor = loader.RawBoost12(waves[0], args, 16000, audio_path="x")
        views = [waves[0], aug_anchor] + waves[1:] + aug_voc
        batch = nii.batch_pad_for_multiview([np.expand_dims(v, 1) for v in views], 16000, trim_len, random_trim_nosil=True,
                                            repeat_pad=True)
        batch = np.concatenate(batch, axis=1)
        arrays[f"item{item}"] = batch.astype(np.float32)
        meta["item"][f"item{item}"] = {"L": L, "trim": trim_len, "seed": 4242 + item, "first_wave": 100 + 4 * item,
                                       "shape": list(batch.shape), "stream": stream_digest()}
    np.savez_compressed(os.path.join(OUT, "multiview_golden.npz"), **arrays)
    with open(os.path.join(OUT, "multiview_golden.json"), "w") as f:
        json.dump(meta, f, indent=1, sort_keys=True)
    print(f"wrote {len(arrays)} multiview arrays to {OUT}")


def sha1_of(a):
    return hashlib.sha1(np.ascontiguousarray(a).tobytes()).hexdigest()


def main_round2():
    """Round-2 fixtures, all from the UNMODIFIED reference (tests/golden/round2_golden.{npz,json}):
    inputs above full scale (every algo), float64 / all-zero / NaN inputs, utterances longer than 65536 samples
    (what the loaders feed RawBoost before the crop, asvspoof_2019_augall_3.py:105-117), the reverb augmentor's arithmetic
    (audio_augmentor/reverb.py:33-44) and one whole ``Dataset_for.__getitem__`` (asvspoof_2019_augall_3.py:103-146)."""
    warnings.simplefilter("ignore", DeprecationWarning)
    warnings.simplefilter("ignore", RuntimeWarning)  # 0/0 in normWav(zeros, 1)
    rb, loader = import_reference()
    args = make_args()
    arrays, meta = {}, {"over": {}, "f64": {}, "zeros": {}, "nan": {}, "long": {}, "reverb": {}, "getitem": {}}

    # ---- inputs above full scale: ISD must see the raw x (RawBoost.py:76-84), every algo -------------------------------
    L = 16000
    for algo in range(1, 9):
        for u in (0, 1):
            x = overscale_utterance(u, L)
            np.random.seed(seed_for(50 + u))
            y = np.asarray(loader.process_Rawboost_feature(x, 16000, args, algo))
            key = f"over_algo{algo}_u{u}"
            rec = summarise(y)
            rec["stream"] = stream_digest()
            if algo == 2:
                rec["sha1_f32"] = sha1_of(y)  # float32 in -> float32 out: bit-exact contract
            if algo in (2, 7, 8):
                arrays[key] = y.astype(np.float32)
            meta["over"][key] = rec
    for u in (0, 1):
        x = overscale_utterance(u, L)
        np.random.seed(seed_for(50 + u))
        arrays[f"over_op_isd_u{u}"] = rb.ISD_additive_noise(x, 10, 2)

    # ---- float64 input (np.power keeps float64, RawBoost.py:66; ISD returns float64) --------------------------------------
    x64 = 0.3 * np.random.RandomState(31).standard_normal(4000)
    for algo in (1, 2, 3, 5):
        np.random.seed(seed_for(60))
        y = np.asarray(loader.process_Rawboost_feature(x64, 16000, args, algo))
        arrays[f"f64_algo{algo}"] = y.astype(np.float32)
        meta["f64"][f"f64_algo{algo}"] = {"dtype": str(y.dtype), "stream": stream_digest()}

    # ---- all-zero input ---------------------------------------------------------------------------------------------------
    z = np.zeros(1000, dtype=np.float32)
    for algo in (1, 2, 3, 5):
        np.random.seed(seed_for(61))
        y = np.asarray(loader.process_Rawboost_feature(z, 16000, args, algo))
        arrays[f"zeros_algo{algo}"] = y.astype(np.float32)
        meta["zeros"][f"zeros_algo{algo}"] = {"nan_count": int(np.isnan(y).sum()), "stream": stream_digest()}
    arrays["zeros_norm0"] = np.asarray(rb.normWav(z, 0))
    arrays["zeros_norm1"] = np.asarray(rb.normWav(z, 1))  # 0/0: NaN everywhere, kept by the reference

    # ---- NaN sample -------------------------------------------------------------------------------------------------------
    xn = synth_utterance(9, 3000, True).copy()
    xn[100] = np.nan
    for algo in (1, 2, 3, 5):
        np.random.seed(seed_for(62))
        y = np.asarray(loader.process_Rawboost_feature(xn, 16000, args, algo))
        arrays[f"nan_algo{algo}"] = y.astype(np.float32)
        meta["nan"][f"nan_algo{algo}"] = {"nan_count": int(np.isnan(y).sum()), "stream": stream_digest()}
    arrays["nan_norm0"] = np.asarray(rb.normWav(xn, 0))
    arrays["nan_norm1"] = np.asarray(rb.normWav(xn, 1))

    # ---- utterances longer than 65536 samples: summaries and (for the bit-exact operators) digests ------------------------
    for Llong in (65537, 100000, 211000):
        for loud in (0, 1):
            x = synth_utterance(70 + loud, Llong, bool(loud))
            if loud:
                x = (x * 2.0).astype(np.float32)  # peak 1.8: normWav fires
            for algo in (2, 5):
                np.random.seed(seed_for(70))
                y = np.asarray(loader.process_Rawboost_feature(x, 16000, args, algo))
                rec = summarise(y)
                rec["stream"] = stream_digest()
                if algo == 2:
                    rec["sha1_f32"] = sha1_of(y)
                meta["long"][f"long_algo{algo}_L{Llong}_loud{loud}"] = rec
            for always in (0, 1):
                meta["long"][f"long_norm{always}_L{Llong}_loud{loud}"] = {"sha1_f32": sha1_of(rb.normWav(x, always))}

    # ---- reverb: ReverbAugmentor.transform on a synthetic impulse response -------------------------------------------------
    import datautils.audio_augmentor.reverb as ref_reverb
    captured = {}
    rir = (np.exp(-np.arange(3000) / 400.0) * np.random.RandomState(5).standard_normal(3000)).astype(np.float32)
    ref_reverb.librosa.load = lambda path, sr=None, **kw: (rir, sr)
    ref_reverb.librosa_to_pydub = lambda data, sr=16000: captured.__setitem__("y", np.array(data)) or "segment"
    aug = ref_reverb.ReverbAugmentor.__new__(ref_reverb.ReverbAugmentor)  # __init__ lists a corpus directory; not needed here
    aug.sr, aug.rir_file = 16000, "synthetic.wav"
    for tag, data in (("speech", synth_utterance(80, 20000, False)), ("loud", synth_utterance(81, 7001, True))):
        aug.data = data
        aug.transform()
        arrays[f"reverb_{tag}"] = captured["y"].astype(np.float32)
        meta["reverb"][f"reverb_{tag}"] = {"dtype": str(captured["y"].dtype), "len": int(captured["y"].shape[0]),
                                           "peak": float(np.abs(captured["y"]).max())}
    arrays["reverb_rir"] = rir

    # ---- one whole Dataset item through the reference's own __getitem__ ---------------------------------------------------
    ids, vocoders = list(CORPUS_IDS), list(CORPUS_VOCODERS)
    loader.librosa.load = lambda path, sr=None, mono=True, **kw: (corpus_wave(path), sr)
    ds = loader.Dataset_for(make_args(), ids, {}, "/data", vocoders=vocoders, augmentation_methods=["RawBoost12"],
                            num_additional_real=2, trim_length=12000, online_aug=True, aug_dir="", repeat_pad=True)
    for idx in (0, 3):
        np.random.seed(8000 + idx)
        utt, data, label = ds[idx]
        arrays[f"getitem{idx}_data"] = data.numpy().astype(np.float32)
        arrays[f"getitem{idx}_label"] = label.numpy().astype(np.float32)
        meta["getitem"][f"getitem{idx}"] = {"utt": utt, "seed": 8000 + idx, "shape": list(data.shape), "trim_length": 12000,
                                            "num_additional_real": 2, "vocoders": vocoders, "stream": stream_digest()}
    meta["getitem"]["ids"] = ids

    paths = golden_files.save(OUT, "round2_golden", arrays)
    with open(os.path.join(OUT, "round2_golden.json"), "w") as f:
        json.dump(meta, f, indent=1, sort_keys=True)
    size = sum(os.path.getsize(p) for p in paths)
    print(f"wrote {len(arrays)} round-2 arrays ({size/1e6:.2f} MB in {len(paths)} files) to {OUT}")


if __name__ == "__main__":
    if "--multiview" in sys.argv:
        main_multiview()
    elif "--round2" in sys.argv:
        main_round2()
    else:
        main()

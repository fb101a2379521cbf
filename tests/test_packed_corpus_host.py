"""The packed corpus without a device: PackedCorpus's packing helpers (chunk-aligned starts, zero tails, the byte counts of the
ragged ASVspoof-2019-LA-like mix), the PCM16 exactness rule, and the argument checks of rb_items_run_packed /
rb_items_stream_run_packed that fail before any CUDA call."""
import ctypes as C

import numpy as np
import pytest

from oracle import rawboost_oracle as orc


def ragged_lengths(R):
    """bench.py's ragged mix of un-cropped utterance lengths (gamma(3.2, 16 000) + 20 000, clipped to [24 000, 211 000])."""
    rs = np.random.RandomState(2019)
    return np.clip(rs.gamma(shape=3.2, scale=16000.0, size=R) + 20000, 24000, 211000).astype(np.int32)


def test_packed_layout_is_chunk_aligned_with_zero_tails():
    from scl_deepfake_audio_detection_b200 import multiview
    lens = np.array([1, 3, 7, 8, 9, 16, 17, 4, 5], dtype=np.int32)
    rs = np.random.RandomState(0)
    for dtype, per, np_t in (("pcm16", 8, np.int16), ("float32", 4, np.float32)):
        start, chunks = multiview.packed_layout(lens, dtype)
        n = (lens + per - 1) // per
        assert start.dtype == np.int64 and start[0] == 0 and np.array_equal(np.diff(start), n[:-1]) and chunks == n.sum()
        waves = [(rs.randint(1, 3000, L) * (1 if dtype == "pcm16" else 0.25)).astype(np_t) for L in lens]
        buf = multiview.pack_rows(waves, start, chunks, dtype)
        assert buf.dtype == np_t and buf.nbytes == 16 * chunks
        for w, s, k in zip(waves, start, n):
            row = buf[s * per:(s + k) * per]
            assert np.array_equal(row[:w.shape[0]], w) and not np.any(row[w.shape[0]:]), (dtype, w.shape[0])
    with pytest.raises(ValueError):
        multiview.packed_layout(lens, "float16")


def test_packed_bytes_of_the_ragged_mix():
    """R = 2580 * 4 rows of the ragged mix: the sample bytes of each storage form, against a corpus padded to the longest."""
    from scl_deepfake_audio_detection_b200 import multiview
    lens = ragged_lengths(2580 * 4).astype(np.int64)
    pcm = 16 * multiview.packed_layout(lens, "pcm16")[1]
    f32 = 16 * multiview.packed_layout(lens, "float32")[1]
    assert pcm == int(np.sum(2 * ((lens + 7) // 8 * 8))) and f32 == int(np.sum(4 * ((lens + 3) // 4 * 4)))
    padded = lens.size * 4 * ((int(lens.max()) + 3) // 4 * 4)
    assert (round(pcm / 1e9, 2), round(f32 / 1e9, 2), round(padded / 1e9, 2)) == (1.47, 2.94, 8.71)


def test_pcm16_exactness_rule_names_the_file():
    from scl_deepfake_audio_detection_b200 import multiview
    k = np.array([-32768, -1, 0, 1, 32767], dtype=np.int16)
    assert multiview.pcm16_samples(k, "a.wav") is not None and np.array_equal(multiview.pcm16_samples(k, "a.wav"), k)
    for dt in (np.float32, np.float64):
        assert np.array_equal(multiview.pcm16_samples(k.astype(dt) / 32768, "a.wav"), k)
    for bad in (np.array([0.5 / 32768], np.float32), np.array([1.0], np.float32), np.array([np.nan], np.float32),
                np.array([-32769 / 32768]), np.array([1, 2], dtype=np.int32)):
        with pytest.raises(ValueError, match="bonafide/u7.wav"):
            multiview.pcm16_samples(bad, "/data/bonafide/u7.wav")


def _lib_and_args():
    from scl_deepfake_audio_detection_b200 import _lib
    return _lib, _lib.load(), _lib.args_struct(orc.make_args(), 16000)


def test_packed_entries_argument_checks():
    """Null descriptor, unknown kind, wrong rows, negative chunks, misaligned samples, and the checks shared with the padded
    entries: all refused before any CUDA call (the pointers below are never dereferenced)."""
    _lib, lib, a = _lib_and_args()
    assert C.sizeof(_lib.RbCorpus) == 40
    N, nvoc, ws = 10, 3, 1 << 40

    def desc(samples=256, kind=_lib.RB_CORPUS_PCM16, rows=N * (1 + nvoc), chunks=100, start=16, len_=16):
        return _lib.RbCorpus(samples=samples, kind=kind, rows=rows, chunks=chunks, start=start, len=len_)

    def run(corpus, G=4, layout=0, out=16, w=256, wbytes=ws, ld=64):
        c = C.byref(corpus) if corpus is not None else None
        return lib.rb_items_run_packed(C.byref(a), G, nvoc, 2, N, ld, 16, 1, layout, c, 16, 16, out, None, None, None, w, wbytes,
                                       None)

    def stream_run(corpus, G=4, layout=0, out=16, w=256, wbytes=ws, ld=64):
        c = C.byref(corpus) if corpus is not None else None
        return lib.rb_items_stream_run_packed(C.byref(a), 1, 16, G, nvoc, 2, N, ld, 16, 1, layout, c, 16, 16, out, None, None, None,
                                              w, wbytes, None)

    for entry in (run, stream_run):
        assert entry(None) == -1
        assert entry(desc(kind=2)) == -1 and entry(desc(kind=-1)) == -1
        assert entry(desc(rows=N * (1 + nvoc) - 1)) == -1 and entry(desc(rows=N)) == -1
        assert entry(desc(chunks=-1)) == -1
        assert entry(desc(samples=None)) == -1 and entry(desc(start=None)) == -1 and entry(desc(len_=None)) == -1
        assert entry(desc(samples=264)) == -2 and entry(desc(samples=257)) == -2
        assert entry(desc(), out=None) == -1 and entry(desc(), layout=2) == -1
        assert entry(desc(), ld=66) == -2
        assert entry(desc(), w=None) == -3 and entry(desc(), wbytes=100) == -3
        assert entry(None, G=0, out=None) == 0

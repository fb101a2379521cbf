"""Ragged host batches packed back to back through the pipelined seeded entry (rb_submit_seeded_packed).

Held to: the padded entry (rb_submit_seeded_ex) on the same utterances zero-padded to the same row stride, bit for bit, for
every algo, chunking and input kind; nothing written outside the packed span; the documented traffic; the argument checks;
and, on a sample, the float64 oracle.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from conftest import ROOT  # noqa: E402
from oracle import rawboost_oracle as orc  # noqa: E402  (checker only)

ARGS = orc.make_args()
SR = 16000
# edges of the 4-sample vectors, the 1024-sample kernel tiles, the 65 536-sample planner permutation, and the longest loader row
MIXED = [1, 2, 3] + list(range(31, 66)) + [4095, 4096, 4097, 65535, 65536, 65537, 211000]


def waves_for(lengths, seed):
    rs = np.random.RandomState(seed)
    return [(0.4 * rs.standard_normal(n)).astype(np.float32) for n in lengths]


def pinned(n, dtype, lead):
    """A page-locked 1-D array of n elements starting `lead` elements into its buffer (an unaligned base for odd lead)."""
    buf = torch.zeros(n + lead, dtype=torch.int16 if dtype == np.int16 else torch.float32).pin_memory().numpy()
    return buf[lead:lead + n]


def padded_reference(eng, algo, waves, seeds, ld, dtype="f32"):
    """rb_submit_seeded_ex on the same utterances zero-padded to rows of stride ld."""
    want = np.int16 if dtype == "pcm16" else np.float32
    x = np.zeros((len(waves), ld), dtype=want)
    for u, w in enumerate(waves):
        x[u, :w.shape[0]] = w
    lengths = np.array([w.shape[0] for w in waves], dtype=np.int32)
    y = np.zeros((len(waves), ld), dtype=np.float32)
    eng.wait_host(eng.submit_host_ex(algo, x, dtype, lengths, seeds, SR, ARGS, out=y))
    return [y[u, :w.shape[0]] for u, w in enumerate(waves)]


def ld_for(waves):
    return (max(w.shape[0] for w in waves) + 3) // 4 * 4


def packed_call(eng, algo, waves, seeds, dtype="f32", lead=1):
    """The packed entry with x and y at unaligned bases inside sentinel-filled pinned buffers; checks the sentinels and returns
    the per-utterance results."""
    from scl_deepfake_audio_detection_b200.engine import pack_host_utterances, split_packed
    flat, off = pack_host_utterances(waves, dtype)
    total = int(off[-1])
    x = pinned(total, flat.dtype, lead)
    x[:] = flat
    ybuf = pinned(total + 2 * lead + 8, np.float32, 0)
    ybuf[:] = np.float32(-7.5)
    y = ybuf[lead:lead + total]
    eng.wait_host(eng.submit_host_packed(algo, x, dtype, off, seeds, SR, ARGS, out=y))
    assert np.all(ybuf[:lead] == np.float32(-7.5)) and np.all(ybuf[lead + total:] == np.float32(-7.5)), "written outside off[0]..off[B]"
    return split_packed(y, off)


@pytest.fixture(scope="module")
def eng():
    from scl_deepfake_audio_detection_b200.engine import Engine
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    e = Engine(0)
    yield e
    e.set_host_chunk(0)


@pytest.mark.gpu
@pytest.mark.parametrize("algo", range(9))
@pytest.mark.parametrize("chunk", [0, 3])
def test_packed_equals_padded_entry(eng, algo, chunk):
    """Every algo, the default chunk and chunks of three utterances (spans split mid-batch at odd offsets), x and y at odd bases."""
    waves = waves_for(MIXED, 100 + algo)
    seeds = np.arange(7000 + 50 * algo, 7000 + 50 * algo + len(waves), dtype=np.uint32)
    eng.set_host_chunk(chunk)
    try:
        want = padded_reference(eng, algo, waves, seeds, ld_for(waves))
        got = packed_call(eng, algo, waves, seeds, lead=1 + 2 * chunk)
    finally:
        eng.set_host_chunk(0)
    for u, (g, w) in enumerate(zip(got, want)):
        assert np.array_equal(g, w), (algo, chunk, u, MIXED[u])


@pytest.mark.gpu
@pytest.mark.parametrize("algo", [5, 2, 3, 0])
def test_packed_pcm16_and_device_sink(eng, algo):
    """Packed PCM16 == packed float32 of pcm / 32768 bit for bit; a device sink's rows == the host sink; PCM16 == the padded PCM16
    entry."""
    rs = np.random.RandomState(3 + algo)
    pcm = [rs.randint(-32768, 32768, size=n).astype(np.int16) for n in MIXED]
    f32 = [(p.astype(np.float32) / np.float32(32768.0)).astype(np.float32) for p in pcm]
    seeds = np.arange(300, 300 + len(pcm), dtype=np.uint32)
    got16 = packed_call(eng, algo, pcm, seeds, "pcm16", lead=1)
    got32 = packed_call(eng, algo, f32, seeds, "f32", lead=3)
    want16 = padded_reference(eng, algo, pcm, seeds, (ld_for(pcm) + 7) // 8 * 8, "pcm16")
    from scl_deepfake_audio_detection_b200.engine import pack_host_utterances
    flat, off = pack_host_utterances(pcm, "pcm16")
    ld = ld_for(pcm)
    sink = torch.full((len(pcm), ld), 3.25, dtype=torch.float32, device=eng.device)
    eng.wait_host(eng.submit_host_packed(algo, flat, "pcm16", off, seeds, SR, ARGS, out=sink))
    rows = sink.cpu().numpy()
    for u, n in enumerate(MIXED):
        assert np.array_equal(got16[u], got32[u]), (algo, u)
        assert np.array_equal(got16[u], want16[u]), (algo, u)
        assert np.array_equal(rows[u, :n], got16[u]), (algo, u)


@pytest.mark.gpu
def test_two_packed_calls_in_flight(eng):
    """Two submits of batches with different lengths before either is waited for; both equal their blocking calls."""
    from scl_deepfake_audio_detection_b200.engine import pack_host_utterances, split_packed
    la, lb = [64600, 3, 41234, 17, 211000, 9000], [5, 120000, 2561, 64600]
    wa, wb = waves_for(la, 1), waves_for(lb, 2)
    sa, sb = np.arange(10, 16, dtype=np.uint32), np.arange(90, 94, dtype=np.uint32)
    want_a, want_b = padded_reference(eng, 5, wa, sa, ld_for(wa)), padded_reference(eng, 5, wb, sb, ld_for(wb))
    (xa, oa), (xb, ob) = pack_host_utterances(wa), pack_host_utterances(wb)
    ya, yb = pinned(int(oa[-1]), np.float32, 0), pinned(int(ob[-1]), np.float32, 0)
    eng.set_host_chunk(2)
    try:
        ta = eng.submit_host_packed(5, xa, "f32", oa, sa, SR, ARGS, out=ya)
        tb = eng.submit_host_packed(5, xb, "f32", ob, sb, SR, ARGS, out=yb)
        eng.wait_host(tb)
        eng.wait_host(ta)
    finally:
        eng.set_host_chunk(0)
    assert tb > ta
    for g, w in zip(split_packed(ya, oa) + split_packed(yb, ob), want_a + want_b):
        assert np.array_equal(g, w)


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [0, 70000])
def test_packed_past_the_grid_split(eng, chunk):
    """70 000 rows of 1-16 samples (algo 2): with one chunk of every row, the unpack / pack kernels see more rows than a grid's
    y dimension holds."""
    rs = np.random.RandomState(65536)
    lengths = rs.randint(1, 17, size=70000)
    waves = [(0.9 * rs.uniform(-1, 1, n)).astype(np.float32) for n in lengths]
    seeds = rs.randint(0, 2 ** 32, size=lengths.size, dtype=np.int64).astype(np.uint32)
    eng.set_host_chunk(chunk)
    try:
        want = padded_reference(eng, 2, waves, seeds, 16)
        got = packed_call(eng, 2, waves, seeds, lead=5)
    finally:
        eng.set_host_chunk(0)
    assert np.array_equal(np.concatenate(got), np.concatenate(want))


@pytest.mark.gpu
def test_packed_traffic_is_the_documented_formula(eng):
    from scl_deepfake_audio_detection_b200.engine import pack_host_utterances
    waves = waves_for(MIXED, 9)
    B = len(waves)
    seeds = np.arange(B, dtype=np.uint32)
    flat, off = pack_host_utterances(waves)
    total = int(off[-1])
    y = np.zeros(total, np.float32)
    meta = 8 * (B + 1) + 4 * B
    eng.wait_host(eng.submit_host_packed(5, flat, "f32", off, seeds, SR, ARGS, out=y))
    assert eng.last_host_traffic() == (4 * total + meta, 4 * total)
    eng.wait_host(eng.submit_host_packed(0, flat, "f32", off, seeds, SR, ARGS, out=y))  # no plan, so no seeds go up
    assert eng.last_host_traffic() == (4 * total + 8 * (B + 1), 4 * total)
    pcm, _ = pack_host_utterances([np.zeros(w.shape[0], np.int16) for w in waves], "pcm16")
    eng.wait_host(eng.submit_host_packed(5, pcm, "pcm16", off, seeds, SR, ARGS, out=y))
    assert eng.last_host_traffic() == (2 * total + meta, 4 * total)
    sink = torch.zeros((B, ld_for(waves)), dtype=torch.float32, device=eng.device)
    eng.wait_host(eng.submit_host_packed(5, pcm, "pcm16", off, seeds, SR, ARGS, out=sink))
    assert eng.last_host_traffic() == (2 * total + meta, 0)


@pytest.mark.gpu
def test_packed_argument_checks(eng):
    from scl_deepfake_audio_detection_b200 import _lib
    lib, ctx = eng.lib, eng._host_ctx()
    a = _lib.args_struct(ARGS, SR)
    x = np.zeros(64, np.float32)
    y = np.zeros(64, np.float32)
    seeds = np.zeros(4, np.uint32)
    dev = torch.zeros((4, 32), dtype=torch.float32, device=eng.device)
    t = C.c_uint64(7)

    def call(off, x_kind=_lib.RB_IO_HOST_F32, y_kind=_lib.RB_IO_HOST_F32, ld=0, xp=x.ctypes.data, yp=y.ctypes.data,
             op=None, B=4):
        off = np.ascontiguousarray(off, dtype=np.int64)
        return lib.rb_submit_seeded_packed(ctx, 5, C.byref(a), C.c_void_p(xp), x_kind, C.c_void_p(off.ctypes.data if op is None else op),
                                           C.c_void_p(seeds.ctypes.data), B, ld, C.c_void_p(yp), y_kind, None, 0, C.byref(t))

    INVALID, ALIGN = -1, -2
    good = [0, 10, 10, 30, 60]
    assert call([0, 10, 9, 30, 60]) == INVALID and t.value == 0   # decreasing
    assert call([1, 10, 10, 30, 60]) == INVALID                   # off[0] != 0
    assert call([0, 10, 10, 30, 2 ** 31 + 40]) == INVALID         # a length past INT32_MAX
    assert call(good, xp=0) == INVALID and call(good, yp=0) == INVALID and call(good, op=0) == INVALID
    assert call(good, x_kind=_lib.RB_IO_DEVICE_F32) == INVALID and call(good, x_kind=7) == INVALID
    assert call(good, y_kind=_lib.RB_IO_HOST_PCM16) == INVALID
    dp = dev.data_ptr()
    assert call(good, y_kind=_lib.RB_IO_DEVICE_F32, yp=dp, ld=28) == INVALID   # below the longest utterance
    assert call(good, y_kind=_lib.RB_IO_DEVICE_F32, yp=dp, ld=0) == INVALID    # a device sink needs its stride
    assert call(good, y_kind=_lib.RB_IO_DEVICE_F32, yp=dp, ld=30) == ALIGN     # not a multiple of 4
    assert call(good, y_kind=_lib.RB_IO_DEVICE_F32, yp=dp + 4, ld=32) == ALIGN  # row base not 16-byte aligned
    assert call(good, ld=29) == INVALID and call(good, ld=34) == ALIGN          # an explicit host-sink stride
    assert call(good, B=-1) == INVALID
    assert call(good, B=0) == 0 and t.value == 0
    assert call([0, 0, 0, 0, 0]) == 0 and t.value == 0            # only empty utterances: nothing to do
    assert call(good, y_kind=_lib.RB_IO_DEVICE_F32, yp=dp, ld=32) == 0 and t.value > 0
    eng.wait_host(t.value)
    with pytest.raises(ValueError):
        eng.submit_host_packed(5, x, "f32", np.array(good, np.int32), seeds, SR, ARGS, out=y)
    with pytest.raises(ValueError):
        eng.submit_host_packed(5, x[:50], "f32", np.array(good, np.int64), seeds, SR, ARGS, out=y)
    with pytest.raises(ValueError):
        eng.submit_host_packed(5, x.astype(np.int16), "f16", np.array(good, np.int64), seeds, SR, ARGS, out=y)


@pytest.mark.gpu
@pytest.mark.parametrize("algo", [5, 2])
def test_packed_against_the_oracle(eng, algo):
    """A 16-utterance ragged sample against the float64 oracle: 1e-5 max-abs, ISD (algo 2) bit for bit."""
    lengths = [64600, 16000, 3, 48001, 2600, 33, 64600, 20000, 1, 9999, 4097, 31000, 64599, 12, 40000, 5000]
    waves = waves_for(lengths, 21)
    seeds = np.arange(4321, 4321 + len(lengths), dtype=np.uint32)
    from scl_deepfake_audio_detection_b200.engine import pack_host_utterances, split_packed
    flat, off = pack_host_utterances(waves)
    got = eng.process_host_packed(algo, flat, "f32", off, seeds, SR, ARGS)
    state = np.random.get_state()
    try:
        for u, (g, w) in enumerate(zip(split_packed(got, off), waves)):
            np.random.seed(int(seeds[u]))
            ref = np.asarray(orc.process(w, SR, ARGS, algo), dtype=np.float64)
            if algo == 2:
                assert np.array_equal(g.astype(np.float64), ref), u
            else:
                assert np.max(np.abs(g.astype(np.float64) - ref)) <= 1e-5, u
    finally:
        np.random.set_state(state)


# ---- without a GPU ----------------------------------------------------------------------------------------------------------
def test_pack_and_split_helpers_round_trip():
    from scl_deepfake_audio_detection_b200.engine import pack_host_utterances, split_packed
    waves = [np.arange(n, dtype=np.float32) + n for n in (3, 0, 5, 1)]
    flat, off = pack_host_utterances(waves, pin=False)
    assert off.dtype == np.int64 and off.tolist() == [0, 3, 3, 8, 9] and flat.dtype == np.float32 and flat.shape == (9,)
    for g, w in zip(split_packed(flat, off), waves):
        assert np.array_equal(g, w)
    pcm, off16 = pack_host_utterances([np.array([1, -2], np.int16), np.array([32767], np.int16)], "pcm16", pin=False)
    assert pcm.dtype == np.int16 and pcm.tolist() == [1, -2, 32767] and off16.tolist() == [0, 2, 3]
    with pytest.raises(ValueError):
        pack_host_utterances([np.zeros(3, np.float32)], "pcm16", pin=False)


def test_library_exports_the_packed_entry_and_the_header_compiles_as_c(tmp_path):
    from scl_deepfake_audio_detection_b200 import _lib
    lib = _lib.load()
    assert hasattr(lib, "rb_submit_seeded_packed") and "rb_submit_seeded_packed" in _lib.SYMBOLS
    src = tmp_path / "packed.c"
    src.write_text('#include "rawboost_b200.h"\n'
                   "int main(void) {\n"
                   "  int (*fn)(rb_ctx*, int, const rb_args*, const void*, int, const int64_t*, const uint32_t*, int, int, void*, int,\n"
                   "            void*, int, uint64_t*) = rb_submit_seeded_packed;\n"
                   "  return fn != 0 && RB_ABI_VERSION == 1 ? 0 : 1;\n"
                   "}\n")
    cc = os.environ.get("CC", "cc")
    r = subprocess.run([cc, "-std=c99", "-Wall", "-Werror", "-pedantic", "-fsyntax-only", "-I", os.path.join(ROOT, "include"),
                        str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr

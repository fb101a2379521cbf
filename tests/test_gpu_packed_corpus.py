"""Items from a packed corpus (rb_items_run_packed / rb_items_stream_run_packed, multiview.PackedCorpus).

A packed corpus holding the float values of a padded DeviceCorpus (k / 32768 for PCM16) must give the padded entries' results
bit for bit: out, out_len, labels and end states, for seeded items and running streams, float32 and PCM16, in device memory and
in page-locked host memory. Also: rows at the edges of the chunk and crop lengths, one item per storage form against the numpy
reference, a batch past the 65 535-row grid split, pointers the entries must refuse, malformed row tables, and the device
memory a host-resident corpus takes.
"""
import ctypes as C
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import rawboost_oracle as orc  # noqa: E402  (checker only)

ARGS = orc.make_args()
SR = 16000
FORMS = [(dtype, location) for dtype in ("float32", "pcm16") for location in ("device", "host")]


class PcmCorpus:
    """A synthetic corpus of 16-bit PCM values read as float32 k / 32768 (what librosa returns for 16-bit audio):
    ``<dir>/<name>`` and ``<dir>/<vocoder>_<name>``."""

    def __init__(self, lens, nvoc, seed=0, voc_lens=None):
        rs = np.random.RandomState(seed)
        self.ids = [f"u{k}.wav" for k in range(len(lens))]
        self.vocoders = [f"voc{v}" for v in range(nvoc)]
        self.waves = {}
        for k, name in enumerate(self.ids):
            self.waves[name] = self._pcm(rs, lens[k], 6000)
            for v, voc in enumerate(self.vocoders):
                L = voc_lens[k][v] if voc_lens is not None else max(1, lens[k] + int(rs.randint(-40, 41)))
                self.waves[voc + "_" + name] = self._pcm(rs, L, 30000 if v % 2 else 3000)

    @staticmethod
    def _pcm(rs, L, scale):
        k = np.clip(np.round(rs.standard_normal(L) * scale), -32768, 32767)
        k[:min(L, 2)] = [-32768, 32767][:min(L, 2)]
        return (k / 32768).astype(np.float32)

    def load(self, path):
        return self.waves[os.path.basename(path)]


@pytest.fixture(scope="module")
def eng():
    from scl_deepfake_audio_detection_b200.engine import Engine
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return Engine(0)


def _corpora(eng, c):
    """The padded reference and the four packed forms of the same corpus."""
    from scl_deepfake_audio_detection_b200 import multiview
    ref = multiview.DeviceCorpus(c.ids, "/data", c.load, c.vocoders, engine=eng)
    packed = {f: multiview.PackedCorpus(c.ids, "/data", c.load, c.vocoders, dtype=f[0], location=f[1], engine=eng) for f in FORMS}
    return ref, packed


def _seeded(eng, corpus, n_add, trim, indices, seeds, layout):
    from scl_deepfake_audio_detection_b200 import multiview
    bat = multiview.SeededItemBatcher(ARGS, corpus, num_additional_real=n_add, trim_length=trim)
    end = torch.empty((len(indices), 625), dtype=torch.int32, device=eng.device)
    _, data, labels, out_len = bat.items(indices, seeds, layout=layout, end_state=end)
    return data, out_len, labels, end


def _streams(eng, corpus, n_add, trim, index_lists, states, layout):
    from scl_deepfake_audio_detection_b200 import multiview
    bat = multiview.StreamItemBatcher(ARGS, corpus, num_additional_real=n_add, trim_length=trim)
    _, data, labels, out_len, end = bat.items_streams(index_lists, states, layout=layout)
    return data, out_len, labels, end


def _assert_same(got, want, what):
    for name, a, b in zip(("out", "out_len", "labels", "end_state"), got, want):
        assert torch.equal(a, b), (what, name)


@pytest.fixture(scope="module")
def matrix_corpora(eng):
    c = PcmCorpus([1200, 2500, 1, 3000, 900, 1001, 7, 1999], 2, seed=11)
    return c, _corpora(eng, c)


@pytest.mark.gpu
@pytest.mark.parametrize("walk", ["seeded", "one_stream", "three_streams"])
@pytest.mark.parametrize("form", FORMS, ids=[f"{d}-{l}" for d, l in FORMS])
@pytest.mark.parametrize("layout", [0, 1])
@pytest.mark.parametrize("n_add", [0, 2])
def test_packed_equals_padded(eng, matrix_corpora, walk, form, layout, n_add):
    c, (ref, packed) = matrix_corpora
    N, trim = len(c.ids), 1000
    rs = np.random.RandomState(layout * 10 + n_add)
    indices = [0, N - 1] + list(rs.randint(0, N, 22))
    if walk == "seeded":
        seeds = [0, 2 ** 32 - 1] + [int(s) for s in rs.randint(0, 2 ** 32, 22, dtype=np.int64)]
        run = lambda corpus: _seeded(eng, corpus, n_add, trim, indices, seeds, layout)  # noqa: E731
    else:
        cuts = [0, 24] if walk == "one_stream" else [0, 5, 5, 24]  # three streams, one of them empty
        lists = [indices[a:b] for a, b in zip(cuts[:-1], cuts[1:])]
        states = [np.random.RandomState(100 + q).get_state() for q in range(len(lists))]
        run = lambda corpus: _streams(eng, corpus, n_add, trim, lists, states, layout)  # noqa: E731
    want = run(ref)
    got = run(packed[form])
    torch.cuda.synchronize()
    _assert_same(got, want, (walk, form))


@pytest.mark.gpu
def test_packed_row_lengths_at_the_chunk_and_crop_edges(eng):
    """Rows of 1, 3, 7, 8, 9 samples (a PCM16 chunk holds 8, a float32 one 4), trim - 1, trim, trim + 1, and long rows
    (65 536, 65 537, 70 001, 211 000): every form equals the padded corpus, seeded and streamed."""
    trim = 64000
    lens = [1, 3, 7, 8, 9, trim - 1, trim, trim + 1, 65536, 65537, 70001, 211000]
    voc = [[lens[(k + 5) % len(lens)]] for k in range(len(lens))]
    c = PcmCorpus(lens, 1, seed=3, voc_lens=voc)
    ref, packed = _corpora(eng, c)
    N = len(lens)
    indices = list(range(N)) + list(range(N - 1, -1, -1))
    seeds = [31 * g + 5 for g in range(len(indices))]
    want = _seeded(eng, ref, 2, trim, indices, seeds, 1)
    want_s = _streams(eng, ref, 2, trim, [indices[:7], indices[7:]], [np.random.RandomState(9).get_state()] * 2, 0)
    for form, pc in packed.items():
        assert pc.ld == ref.ld and torch.equal(pc.lengths, ref.lengths)
        _assert_same(_seeded(eng, pc, 2, trim, indices, seeds, 1), want, form)
        _assert_same(_streams(eng, pc, 2, trim, [indices[:7], indices[7:]], [np.random.RandomState(9).get_state()] * 2, 0),
                     want_s, form)


def _same_stream(end_row, state):
    a, b = np.random.RandomState(), np.random.RandomState()
    a.set_state(("MT19937", np.asarray(end_row[:624]).view(np.uint32), int(end_row[624])))
    b.set_state(state)
    return np.array_equal(a.random_sample(700), b.random_sample(700))


@pytest.mark.gpu
@pytest.mark.parametrize("form", FORMS, ids=[f"{d}-{l}" for d, l in FORMS])
def test_packed_item_against_the_reference(eng, form):
    """One item per storage form against np.random.seed(s); oracle.dataset_item(...): views within 1e-5, the copied views
    bit for bit, labels exactly, the stream state after the item equal to numpy's."""
    from scl_deepfake_audio_detection_b200 import multiview
    c = PcmCorpus([1500, 3100, 800, 2047, 1000], 3, seed=21)
    pc = multiview.PackedCorpus(c.ids, "/data", c.load, c.vocoders, dtype=form[0], location=form[1], engine=eng)
    n_add, trim, idx, seed = 2, 1000, 1, 2 ** 31 + 7
    data, out_len, labels, end = _seeded(eng, pc, n_add, trim, [idx], [seed], 0)
    np.random.seed(seed)
    _, ref, lab = orc.dataset_item(idx, c.ids, c.load, ARGS, c.vocoders, n_add, trim)
    n = ref.shape[0]
    got = data[0].cpu().numpy()
    assert int(out_len[0]) == n
    assert np.max(np.abs(got[:n].astype(np.float64) - ref)) <= 1e-5
    copies = [0] + list(range(2, 2 + n_add + len(c.vocoders)))
    assert np.array_equal(got[:n, copies], ref[:, copies])
    assert np.array_equal(labels[0].cpu().numpy(), lab)
    assert _same_stream(end[0].cpu().numpy(), np.random.get_state())


@pytest.mark.gpu
def test_packed_past_the_grid_split(eng):
    """G * (nvoc + 1 + n_add) = 66 000 gathered rows of short utterances: every form equals the padded corpus."""
    rs = np.random.RandomState(8)
    N, nvoc, n_add, G = 40, 3, 2, 11000
    c = PcmCorpus(list(rs.randint(8, 40, N)), nvoc, seed=6)
    ref, packed = _corpora(eng, c)
    indices = rs.randint(0, N, G)
    seeds = np.arange(G, dtype=np.int64) * 2654435761 % 2 ** 32
    want = _seeded(eng, ref, n_add, 16, indices, seeds, 1)
    for form, pc in packed.items():
        _assert_same(_seeded(eng, pc, n_add, 16, indices, seeds, 1), want, form)


def _raw_run(eng, pc, desc, G=4, n_add=1, trim=100):
    """rb_items_run_packed called directly with descriptor ``desc`` on pc's shape; returns (rc, kernels launched)."""
    from scl_deepfake_audio_detection_b200 import _lib
    nvoc = pc.nvoc
    a = _lib.args_struct(ARGS, SR)
    need = int(eng.lib.rb_items_workspace_bytes(C.byref(a), G, nvoc, n_add, pc.N, pc.ld))
    ws = torch.empty(need + 256, dtype=torch.uint8, device=eng.device)
    idx = torch.zeros(G, dtype=torch.int32, device=eng.device)
    out = torch.zeros((G, trim, 2 + n_add + 2 * nvoc), dtype=torch.float32, device=eng.device)
    torch.cuda.synchronize()
    before = eng.lib.rb_launch_count()
    rc = eng.lib.rb_items_run_packed(C.byref(a), G, nvoc, n_add, pc.N, pc.ld, trim, 1, 0, C.byref(desc), C.c_void_p(idx.data_ptr()),
                                     C.c_void_p(idx.data_ptr()), C.c_void_p(out.data_ptr()), None, None, None,
                                     C.c_void_p(eng._ws_ptr(ws)), need, C.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return rc, eng.lib.rb_launch_count() - before


@pytest.mark.gpu
def test_packed_refuses_pageable_and_unallocated_samples(eng):
    from scl_deepfake_audio_detection_b200 import _lib, multiview
    c = PcmCorpus([300, 500, 200], 1, seed=2)
    pc = multiview.PackedCorpus(c.ids, "/data", c.load, c.vocoders, dtype="pcm16", location="device", engine=eng)
    rc, launched = _raw_run(eng, pc, pc.descriptor)
    assert rc == 0 and launched > 0
    pageable = np.zeros(pc.nbytes + 16, dtype=np.uint8)
    p = (pageable.ctypes.data + 15) // 16 * 16
    for samples in (p, 1 << 46):  # pageable host memory; an address no allocation covers
        d = _lib.RbCorpus(samples=samples, kind=pc.descriptor.kind, rows=pc.descriptor.rows, chunks=pc.chunks,
                          start=pc.start.data_ptr(), len=pc.lengths.data_ptr())
        assert _raw_run(eng, pc, d) == (-1, 0), hex(samples)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["float32", "pcm16"])
def test_packed_malformed_tables_stay_in_bounds(eng, dtype):
    """start past chunks (and far past it, and negative) and len > ld on a device-resident corpus: the call completes, and the
    items whose rows the table describes correctly equal the padded corpus's."""
    from scl_deepfake_audio_detection_b200 import _lib, multiview
    c = PcmCorpus([1200, 2500, 1800, 3000, 900, 1500, 2200, 1300], 1, seed=12)
    ref = multiview.DeviceCorpus(c.ids, "/data", c.load, c.vocoders, engine=eng)
    pc = multiview.PackedCorpus(c.ids, "/data", c.load, c.vocoders, dtype=dtype, location="device", engine=eng)
    # rows 3: bona fide 3; 9, 11: the vocoded copies of 1 and 3; 12: the vocoded copy of 4 (N = 8, one vocoder)
    bad = {3: ("start", pc.chunks + 5), 9: ("start", 1 << 62), 11: ("start", -7), 12: ("len", pc.ld + 100)}
    start, lengths = pc.start.clone(), pc.lengths.clone()
    for r, (what, v) in bad.items():
        (start if what == "start" else lengths)[r] = v
    desc = _lib.RbCorpus(samples=pc.samples.data_ptr(), kind=pc.descriptor.kind, rows=pc.descriptor.rows, chunks=pc.chunks,
                         start=start.data_ptr(), len=lengths.data_ptr())
    rs = np.random.RandomState(3)
    G, n_add, trim = 64, 2, 1000
    indices = rs.randint(0, len(c.ids), G)
    seeds = rs.randint(0, 2 ** 32, G, dtype=np.int64)
    want = _seeded(eng, ref, n_add, trim, indices, seeds, 0)
    got = eng.items_run_packed(ARGS, SR, desc, pc.ld, pc.nvoc, n_add, trim, indices, seeds, True, 0)
    torch.cuda.synchronize()
    bat = multiview.SeededItemBatcher(ARGS, ref, num_additional_real=n_add, trim_length=trim)
    rows = bat.draw(indices, seeds)["src_row"].cpu().numpy()
    per = pc.nvoc + 1
    touched = set()
    for g in range(G):
        mine = list(rows[g * per:(g + 1) * per]) + list(rows[G * per + g * n_add:G * per + (g + 1) * n_add])
        if any(int(r) in bad for r in mine):
            touched.add(g)
    clean = [g for g in range(G) if g not in touched]
    assert touched and len(clean) >= 8
    for a, b in zip(got, want[:3]):
        assert torch.equal(a[clean], b[clean])


@pytest.mark.gpu
def test_host_corpus_takes_only_its_tables_on_the_device(eng):
    from scl_deepfake_audio_detection_b200 import multiview
    c = PcmCorpus([40000, 61000, 25000, 90000, 33000], 3, seed=4)
    R = len(c.ids) * 4
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated(eng.device)
    pc = multiview.PackedCorpus(c.ids, "/data", c.load, c.vocoders, dtype="pcm16", location="host", engine=eng)
    torch.cuda.synchronize()
    grew = torch.cuda.memory_allocated(eng.device) - before
    assert pc.samples.device.type == "cpu" and pc.samples.is_pinned()
    assert pc.nbytes == pc.samples.numel() * 2 == sum(2 * ((w.shape[0] + 7) // 8 * 8) for w in c.waves.values())
    assert grew <= 12 * R + 2 * 512, grew

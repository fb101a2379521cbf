"""Dataset_for items that share numpy's running stream, on the device (rb_items_stream_draw / rb_items_stream_run,
multiview.StreamItemBatcher).

The items of one stream must equal ``np.random.set_state(start); for idx in items: oracle.dataset_item(idx, ...)``: the views
within 1e-5 (copies bit for bit), the labels exactly, the extra utterances, crop starts, tap counts, impulse positions and float64
gains bit for bit, the taps within 1 ulp, and the stream's state after its last item equal to numpy's. The first three tests need
no device: the argument checks and StreamItemBatcher's input checks run before any CUDA call.
"""
import ctypes as C
import types

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from conftest import stream_digest  # noqa: E402
from oracle import rawboost_oracle as orc  # noqa: E402  (checker only)
from test_gpu_items import EDGES, SR, Corpus, _rows_reference, _same_stream  # noqa: E402

ARGS = orc.make_args()


def _lib_and_args(**kw):
    from scl_deepfake_audio_detection_b200 import _lib
    return _lib.load(), _lib.args_struct(orc.make_args(**kw), SR)


def test_stream_items_argument_checks():
    from scl_deepfake_audio_detection_b200 import _lib
    lib, a = _lib_and_args()
    ws = 1 << 40
    draw = lambda S=2, G=4, N=10, ld=64, off=16, st=16, ptr=16, w=256, wbytes=ws, args=a, plan=True: lib.rb_items_stream_draw(  # noqa: E731
        C.byref(args), S, off, G, 3, 2, N, ld, 16, ptr, ptr, st, ptr, ptr, ptr, None, w, wbytes,
        C.byref(_lib.RbPlan()) if plan else None, None)
    assert draw(off=None) == -1 and draw(st=None) == -1 and draw(ptr=None) == -1 and draw(plan=False) == -1
    assert draw(S=-1) == -1 and draw(S=0) == -1
    assert draw(G=-1) == -1 and draw(N=0) == -1
    assert draw(ld=66) == -2 and draw(w=128) == -2
    assert draw(w=None) == -3 and draw(wbytes=100) == -3
    assert draw(args=_lib_and_args(nBands=12, maxCoeff=200)[1]) == -6
    assert draw(G=0, off=None, st=None, ptr=None) == 0      # no item: nothing is launched
    assert draw(S=0, G=0) == 0 and draw(S=-1, G=0) == -1
    run = lambda S=2, G=4, off=16, st=16, corpus=16, out=16, layout=0, w=256, wbytes=ws: lib.rb_items_stream_run(  # noqa: E731
        C.byref(a), S, off, G, 3, 2, 10, 64, 16, 1, layout, corpus, 16, 16, st, out, None, None, None, w, wbytes, None)
    assert run(off=None) == -1 and run(st=None) == -1 and run(corpus=None) == -1 and run(out=None) == -1
    assert run(S=-1) == -1 and run(S=0) == -1 and run(layout=2) == -1
    assert run(corpus=8) == -2 and run(w=128) == -2
    assert run(w=None) == -3 and run(wbytes=100) == -3
    assert run(G=0, off=None, st=None, corpus=None, out=None) == 0
    assert run(S=7, G=0) == 0                               # more streams than items is legal


def test_stream_items_workspace_is_the_items_workspace():
    """The running-stream entries need what rb_items_workspace_bytes returns for the same shape (no separate query): one byte
    less is refused by the run entry, and the draw entry needs less than the run entry."""
    from scl_deepfake_audio_detection_b200 import _lib
    lib, a = _lib_and_args()
    for G, nvoc, n_add, N, ld in ((8192, 3, 2, 2580, 64600), (5, 0, 0, 1, 4), (3, 1, 2, 70000, 128)):
        need = lib.rb_items_workspace_bytes(C.byref(a), G, nvoc, n_add, N, ld)
        assert need > 0
        rc = lib.rb_items_stream_run(C.byref(a), 2, 16, G, nvoc, n_add, N, ld, 1, 1, 0, 16, 16, 16, 16, 16, None, None, None, 256,
                                     need - 1, None)
        assert rc == -3
        rc = lib.rb_items_stream_draw(C.byref(a), 2, 16, G, nvoc, n_add, N, ld, 1, 16, 16, 16, 16, 16, 16, None, 256, 4096,
                                      C.byref(_lib.RbPlan()), None)
        assert rc == -3


def test_stream_item_batcher_rejects_malformed_input_before_any_launch():
    """States that are not numpy MT19937 states, and indices outside [0, N), raise before anything reaches the device, and
    numpy's global stream is left where it was."""
    from scl_deepfake_audio_detection_b200 import multiview

    def no_device(*_a, **_k):
        raise AssertionError("reached the device")

    corpus = types.SimpleNamespace(N=5, nvoc=1, list_ids=[f"u{k}" for k in range(5)],
                                   eng=types.SimpleNamespace(items_stream_run=no_device, device="cpu"))
    bat = multiview.StreamItemBatcher(ARGS, corpus, num_additional_real=2, trim_length=100)
    with pytest.raises(ValueError):
        multiview.StreamItemBatcher(ARGS, corpus, num_additional_real=5)
    np.random.seed(3)
    np.random.rand(7)
    before = stream_digest()
    good = np.random.get_state()
    with pytest.raises(IndexError):
        bat.items([0, 5])
    with pytest.raises(IndexError):
        bat.items([-1])
    with pytest.raises(IndexError):
        bat.items_streams([[1], [2, 9]], [good, good])
    bad_states = [
        ("PCG64", good[1], good[2]),
        ("MT19937", good[1][:623], good[2]),
        ("MT19937", good[1], 625),
        ("MT19937", good[1], -1),
        ("MT19937", good[1].astype(np.float64), good[2]),
        "MT19937",
    ]
    for bad in bad_states:
        with pytest.raises(ValueError):
            bat.items_streams([[1], [2]], [good, bad])
    with pytest.raises(ValueError):
        bat.items_streams([[1], [2]], [good])              # one state per stream
    with pytest.raises(ValueError):
        bat.items_streams([[1], [2]], torch.zeros((2, 625), dtype=torch.float32))  # state words are 32-bit integers
    assert stream_digest() == before


# ---------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def eng():
    from scl_deepfake_audio_detection_b200.engine import Engine
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return Engine(0)


def _batcher(eng, c, n_add, trim, repeat_pad=True):
    from scl_deepfake_audio_detection_b200 import multiview
    dc = multiview.DeviceCorpus(c.ids, "/data", c.load, c.vocoders, engine=eng)
    return multiview.StreamItemBatcher(ARGS, dc, num_additional_real=n_add, trim_length=trim, repeat_pad=repeat_pad)


def _seeded_state(seed, skip=0):
    """numpy's state after np.random.seed(seed) and `skip` uniform draws (2*skip words)."""
    rs = np.random.RandomState(seed)
    rs.random_sample(skip)
    return rs.get_state()


def _reference_streams(c, index_lists, states, n_add, trim, repeat_pad):
    """Per stream, the items of the numpy reference called one after another from its start state, numpy's own draws of the
    same items (plans, extra utterances, crop starts) and the state after the last item."""
    from scl_deepfake_audio_detection_b200 import plans
    saved = np.random.get_state()
    items, ref_plans, extras, starts, ends = [], [], [], [], []
    try:
        for ix, st in zip(index_lists, states):
            np.random.set_state(st)
            for idx in ix:
                items.append(orc.dataset_item(idx, c.ids, c.load, ARGS, c.vocoders, n_add, trim, repeat_pad=repeat_pad))
            ends.append(np.random.get_state())
            np.random.set_state(st)
            for idx in ix:
                L = [c.waves[v + "_" + c.ids[idx]].shape[0] for v in c.vocoders] + [c.waves[c.ids[idx]].shape[0]]
                ref_plans += [plans.draw_for_algo(n_, SR, ARGS, 5) for n_ in L]
                others = [k for k in range(len(c.ids)) if k != idx]
                extras.append(np.random.choice(others, n_add, replace=False))
                starts.append(int(np.random.rand() * (L[-1] - trim)) if L[-1] >= trim else 0)
    finally:
        np.random.set_state(saved)
    return items, ref_plans, extras, starts, ends


def _check_items(got, items, n_add, nvoc):
    ids, data, labels, out_len = got
    data, labels, out_len = data.cpu().numpy(), labels.cpu().numpy(), out_len.cpu().numpy()
    assert len(ids) == len(items) == data.shape[0]
    for g, (utt, ref, lab) in enumerate(items):
        n = ref.shape[0]
        assert ids[g] == utt and int(out_len[g]) == n, g
        assert np.max(np.abs(data[g][:n].astype(np.float64) - ref), initial=0.0) <= 1e-5, g
        copies = [0] + list(range(2, 2 + n_add + nvoc))
        assert np.array_equal(data[g][:n, copies], ref[:, copies]), g
        assert not np.any(data[g][n:]), "nothing is written past out_len"
        assert np.array_equal(labels[g], lab), g


def _check_streams(bat, c, index_lists, states, n_add, trim, repeat_pad=True, check_plan=True):
    """Run the streams in one call (items_streams) and compare every item, every stream's end state and (optionally) the plan
    with the numpy reference; numpy's global stream must stay where it was."""
    from scl_deepfake_audio_detection_b200 import plans
    nvoc = len(c.vocoders)
    before = stream_digest()
    got = bat.items_streams(index_lists, states)
    torch.cuda.synchronize()
    assert stream_digest() == before, "items_streams must leave numpy's stream alone"
    items, ref_plans, extras, starts, ends = _reference_streams(c, index_lists, states, n_add, trim, repeat_pad)
    _check_items(got[:4], items, n_add, nvoc)
    end = got[4].cpu().numpy()
    assert end.shape == (len(index_lists), 625)
    for q, e in enumerate(ends):
        assert 0 <= int(end[q, 624]) <= 623, "end states are stored with pos 0..623"
        assert _same_stream(end[q], e), q
    if not check_plan:
        return got
    idx = [i for ix in index_lists for i in ix]
    G = len(idx)
    dc, eng = bat.corpus, bat.corpus.eng
    off = np.concatenate([[0], np.cumsum([len(ix) for ix in index_lists])])
    from scl_deepfake_audio_detection_b200.multiview import _state_words
    words = np.stack([_state_words(s) for s in states])
    drawn = eng.items_stream_draw(ARGS, SR, dc.lengths, nvoc, n_add, dc.ld, trim, idx, off, words, end_state=True)
    torch.cuda.synchronize()
    assert np.array_equal(drawn["end_state"].cpu().numpy(), end)
    gp = eng.download_plan(drawn["plan"])
    rp = plans.pack(ref_plans, ld=dc.ld)
    for name in ("lnl_tap_off", "isd_off", "isd_idx", "isd_fr"):
        assert np.array_equal(getattr(rp, name), getattr(gp, name)), name
    rt = np.asarray(rp.lnl_taps, np.float32)
    err = np.abs(gp.lnl_taps.astype(np.float64) - rt) / np.spacing(np.maximum(np.abs(rt), np.float32(1e-30)))
    assert float(np.max(err, initial=0.0)) <= 1.0, "taps more than 1 ulp(fp32) from numpy"
    assert np.array_equal(drawn["start"].cpu().numpy(), starts)
    want_rows = _rows_reference(idx, len(c.ids), nvoc, np.array(extras, dtype=np.int64).reshape(G, n_add))
    assert np.array_equal(drawn["src_row"].cpu().numpy(), want_rows)
    lens = np.array([c.waves[n_].shape[0] for n_ in c.ids] + [c.waves[v + "_" + n_].shape[0] for n_ in c.ids for v in c.vocoders])
    assert np.array_equal(drawn["row_len"].cpu().numpy(), lens[want_rows])
    return got


def _check_global(bat, c, indices, seed, n_add, trim, repeat_pad=True):
    """StreamItemBatcher.items on numpy's global stream == the reference called for the indices in order after the same
    seed, and numpy's stream ends exactly where the reference leaves it (Gaussian cache included)."""
    np.random.seed(seed)
    np.random.standard_normal()  # leaves a cached Gaussian, which the items must carry over
    start = np.random.get_state()
    got = bat.items(indices)
    after = np.random.get_state()
    items, _, _, _, ends = _reference_streams(c, [indices], [start], n_add, trim, repeat_pad)
    _check_items(got, items, n_add, len(c.vocoders))
    assert after[3:] == start[3:]
    row = np.append(after[1], np.uint32(after[2]))
    assert _same_stream(row, ends[0])


@pytest.mark.gpu
@pytest.mark.parametrize("idx", [0, 3])
def test_stream_items_match_reference_getitem(eng, golden2, idx):
    """Fixtures produced by the reference's own Dataset_for after np.random.seed(8000 + idx): the views, the labels and the
    digest of numpy's global state afterwards (the fixtures' pos is below 624, so the stored form compares directly)."""
    from scl_deepfake_audio_detection_b200 import multiview
    arrays, meta = golden2
    m = meta["getitem"][f"getitem{idx}"]
    dc = multiview.DeviceCorpus(orc.CORPUS_IDS, "/data", orc.corpus_wave, orc.CORPUS_VOCODERS, engine=eng)
    bat = multiview.StreamItemBatcher(orc.make_args(), dc, num_additional_real=m["num_additional_real"], trim_length=m["trim_length"])
    np.random.seed(m["seed"])
    ids, data, labels, out_len = bat.items([idx])
    assert stream_digest() == m["stream"], "draw order / count differs from Dataset_for.__getitem__"
    got = data[0].cpu().numpy()
    ref = arrays[f"getitem{idx}_data"]
    assert ids == [m["utt"]] and list(got.shape) == m["shape"] and int(out_len[0]) == m["shape"][0]
    assert np.max(np.abs(got.astype(np.float64) - ref)) <= 1e-5
    for col in (0, 2, 3, 4, 5, 6):
        assert np.array_equal(got[:, col], ref[:, col]), col
    assert np.array_equal(labels[0].cpu().numpy(), arrays[f"getitem{idx}_label"])


@pytest.mark.gpu
def test_stream_items_consecutive_sweep_and_plans(eng):
    """A hundred items on one stream in one call, indices including 0 and N-1, ragged lengths around the crop length: every
    item, its plan, extra utterances and crop start, and the stream's end, against the reference called item after item."""
    rs = np.random.RandomState(15)
    N, nvoc, n_add, trim = 13, 2, 2, 1500
    lens = [1500, 1499, 1, 3000, 700, 2047, 1501, 64, 2500, 1200, 1800, 4000, 999]
    c = Corpus(lens, nvoc, seed=1)
    bat = _batcher(eng, c, n_add, trim)
    indices = [0, N - 1] + [int(i) for i in rs.randint(0, N, 98)]
    _check_streams(bat, c, [indices], [_seeded_state(31)], n_add, trim)
    _check_global(bat, c, indices, 32, n_add, trim)


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(EDGES))
def test_stream_items_edge_cases(eng, case):
    lens, nvoc, n_add, trim, repeat_pad, voc = EDGES[case]
    c = Corpus(lens, nvoc, seed=len(case), voc_lens=voc)
    bat = _batcher(eng, c, n_add, trim, repeat_pad)
    N = len(lens)
    indices = [g % N for g in range(3 * N)]
    _check_streams(bat, c, [indices], [_seeded_state(7919 + N)], n_add, trim, repeat_pad)
    _check_global(bat, c, indices[::-1], 11 * N, n_add, trim, repeat_pad)


@pytest.mark.gpu
def test_stream_items_wide_choice(eng):
    """N - 1 > 65536: the choice's permutation is applied in global memory."""
    N = 70003
    rs = np.random.RandomState(2)
    c = Corpus(list(rs.randint(1, 9, N)), 0, seed=3)
    bat = _batcher(eng, c, 2, 4)
    _check_streams(bat, c, [[0, N - 1, 4242], [65537, 70000]], [_seeded_state(11), _seeded_state(12, 5)], 2, 4)


@pytest.mark.gpu
def test_stream_items_split_invariance(eng):
    """One stream run as two consecutive calls, the first call's end state fed to the second, equals one call bit for bit --
    through the device end state and through numpy's global stream."""
    c = Corpus([1200, 2500, 1800, 3000, 900], 3, seed=9)
    bat = _batcher(eng, c, 2, 1000)
    indices = [4, 0, 2, 2, 1, 3, 0, 4, 3]
    st = _seeded_state(77, 300)
    _, d, l, n, e = bat.items_streams([indices], [st])
    for k in (1, 4, 8):
        _, d1, l1, n1, e1 = bat.items_streams([indices[:k]], [st])
        _, d2, l2, n2, e2 = bat.items_streams([indices[k:]], e1)
        assert torch.equal(torch.cat([d1, d2]), d) and torch.equal(torch.cat([l1, l2]), l) and torch.equal(torch.cat([n1, n2]), n)
        assert torch.equal(e2, e)
    np.random.set_state(st)
    _, g1, _, _ = bat.items(indices[:3])
    _, g2, _, _ = bat.items(indices[3:])
    assert torch.equal(torch.cat([g1, g2]), d)
    assert _same_stream(e[0].cpu().numpy(), np.random.get_state())


@pytest.mark.gpu
def test_stream_items_many_streams(eng):
    """Ragged streams, one of them empty, from states right after np.random.seed (pos 624) and from the middle of a block;
    each stream equals the reference run from its own state, and the empty one returns its start state in the stored form."""
    c = Corpus([1100, 2400, 900, 3100, 1600, 2000], 2, seed=12)
    bat = _batcher(eng, c, 2, 1000)
    index_lists = [[5, 0, 3, 3, 1], [], [2], [4, 4, 0, 1, 2, 5, 3], [1, 2]]
    states = [_seeded_state(1, 100), _seeded_state(2), _seeded_state(3, 311), np.random.RandomState(4).get_state(), _seeded_state(5, 7)]
    assert [s[2] for s in states] == [200, 624, 622, 624, 14]
    got = _check_streams(bat, c, index_lists, states, 2, 1000)
    empty = got[4][1].cpu().numpy()
    assert int(empty[624]) == 0 and _same_stream(empty, states[1])  # pos 624 is stored as the next block at 0


@pytest.mark.gpu
def test_stream_items_one_item_per_stream_equals_seeded_items(eng):
    """S = G streams of one item each, from seeded states, give exactly SeededItemBatcher's items and end states."""
    from scl_deepfake_audio_detection_b200 import multiview
    c = Corpus([1200, 2500, 1800, 3000, 900], 3, seed=21)
    bat = _batcher(eng, c, 2, 1000)
    seeded = multiview.SeededItemBatcher(ARGS, bat.corpus, num_additional_real=2, trim_length=1000)
    indices, seeds = [3, 1, 0, 2, 4, 4, 1], [0, 1, 2 ** 31, 2 ** 32 - 1, 99, 12345, 7]
    end_seeded = torch.empty((len(indices), 625), dtype=torch.int32, device="cuda")
    want = seeded.items(indices, seeds, end_state=end_seeded)
    got = bat.items_streams([[i] for i in indices], [np.random.RandomState(s).get_state() for s in seeds])
    assert got[0] == want[0]
    for a, b in zip(got[1:4], want[1:4]):
        assert torch.equal(a, b)
    assert torch.equal(got[4], end_seeded)


@pytest.mark.gpu
def test_stream_items_device_inputs_on_a_side_stream_do_not_synchronise(eng):
    from scl_deepfake_audio_detection_b200 import multiview
    c = Corpus([1200, 2500, 1800, 3000], 2, seed=4)
    bat = _batcher(eng, c, 1, 1000)
    dc = bat.corpus
    index_lists = [[3, 1], [0, 2, 2], []]
    states = [_seeded_state(8), _seeded_state(9, 40), _seeded_state(10)]
    _, ref, ref_lab, ref_len, ref_end = bat.items_streams(index_lists, states, layout=multiview.LAYOUT_MODEL)
    di = torch.tensor([3, 1, 0, 2, 2], dtype=torch.int32, device="cuda")
    doff = torch.tensor([0, 2, 5, 5], dtype=torch.int32, device="cuda")
    words = np.stack([multiview._state_words(s) for s in states])
    dst = torch.from_numpy(words.view(np.int32)).cuda()
    end = torch.empty((3, 625), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    torch.cuda.set_sync_debug_mode("error")
    try:
        with torch.cuda.stream(side):
            data, out_len, labels = eng.items_stream_run(ARGS, SR, dc.data, dc.lengths, dc.nvoc, 1, 1000, di, doff, dst, True,
                                                         multiview.LAYOUT_MODEL, end_state=end)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    side.synchronize()
    assert torch.equal(data, ref) and torch.equal(labels, ref_lab) and torch.equal(out_len, ref_len) and torch.equal(end, ref_end)


@pytest.mark.gpu
def test_stream_items_past_the_grid_split(eng):
    """G*(nvoc+1) > 65535 RawBoost rows over four streams: the items around the split, and the first items of a stream,
    equal the same items run as a small batch from the same state, bit for bit, and the reference."""
    rs = np.random.RandomState(8)
    N, nvoc = 40, 3
    c = Corpus(list(rs.randint(8, 40, N)), nvoc, seed=6)
    bat = _batcher(eng, c, 1, 16)
    G = 16400  # 65600 RawBoost rows; row 65535 belongs to item 16383
    indices = rs.randint(0, N, G)
    off = [0, 6000, 16382, 16390, G]
    lists = [list(indices[off[q]:off[q + 1]]) for q in range(4)]
    states = [_seeded_state(100 + q, q) for q in range(4)]
    _, data, labels, out_len, end = bat.items_streams(lists, states)
    _, small, slab, slen, send = bat.items_streams([lists[2], lists[0][:3]], [states[2], states[0]])
    big = list(range(16382, 16390)) + [0, 1, 2]
    assert torch.equal(data[big], small) and torch.equal(labels[big], slab) and torch.equal(out_len[big], slen)
    assert torch.equal(send[0], end[2])
    _check_streams(bat, c, [lists[2]], [states[2]], 1, 16, check_plan=False)

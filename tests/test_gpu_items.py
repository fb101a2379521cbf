"""Per-item-seeded Dataset_for items on the device (rb_items_draw / rb_items_run, multiview.SeededItemBatcher).

Item g must equal ``np.random.seed(seeds[g]); oracle.dataset_item(indices[g], ...)``: the views within 1e-5 (copies bit for
bit), the labels exactly, the extra utterances, crop starts, tap counts, impulse positions and float64 gains bit for bit, the
taps within 1 ulp, and the stream state after the item equal to numpy's. The first two tests need no device: the argument
checks run before any CUDA call.
"""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import rawboost_oracle as orc  # noqa: E402  (checker only)

ARGS = orc.make_args()
SR = 16000


def _lib_and_args(**kw):
    from scl_deepfake_audio_detection_b200 import _lib
    return _lib.load(), _lib.args_struct(orc.make_args(**kw), SR)


def _plan_struct():
    from scl_deepfake_audio_detection_b200 import _lib
    return _lib.RbPlan()


def test_items_argument_checks_and_workspace_bound():
    lib, a = _lib_and_args()
    wb = lambda G, nvoc, n_add, N, ld: lib.rb_items_workspace_bytes(C.byref(a), G, nvoc, n_add, N, ld)  # noqa: E731
    assert wb(0, 3, 2, 2580, 64600) == 0
    assert wb(8, 3, 2, 2, 64600) == 0          # n_add > N - 1
    assert wb(8, 3, 2, 3, 64602) == 0          # ld % 4
    assert wb(8, 3, 2, 2580, 64600) > wb(4, 3, 2, 2580, 64600) > 0
    assert wb(8, 3, 2, 2580, 64600) > wb(8, 3, 0, 2580, 64600)
    for G, nvoc, n_add, N, ld in ((8192, 3, 2, 2580, 64600), (5, 0, 0, 1, 4), (3, 1, 2, 70000, 128)):
        batch = (G * (nvoc + 1 + n_add) + G * (nvoc + 1)) * ld * 4  # gathered rows + their RawBoost results
        assert wb(G, nvoc, n_add, N, ld) >= batch
    big = lib.rb_items_workspace_bytes(C.byref(_lib_and_args(nBands=12, maxCoeff=200)[1]), 8, 3, 2, 2580, 64600)
    assert big == 0                            # cascades beyond what the device planner designs
    ws = 1 << 40
    draw = lambda G=4, nvoc=3, n_add=2, N=10, ld=64, trim=16, ptr=16, w=256, wbytes=ws, args=a, plan=True: lib.rb_items_draw(  # noqa: E731
        C.byref(args), G, nvoc, n_add, N, ld, trim, ptr, ptr, ptr, ptr, ptr, ptr, None, w, wbytes,
        C.byref(_plan_struct()) if plan else None, None)
    assert draw(ptr=None) == -1
    assert draw(plan=False) == -1
    assert draw(n_add=10) == -1 and draw(N=0) == -1 and draw(trim=0) == -1 and draw(G=-1) == -1 and draw(nvoc=-1) == -1
    assert draw(ld=66) == -2
    assert draw(w=None) == -3 and draw(wbytes=100) == -3
    assert draw(w=128) == -2
    assert draw(args=_lib_and_args(nBands=12, maxCoeff=200)[1]) == -6
    assert draw(G=0, ptr=None) == 0
    run = lambda G=4, layout=0, corpus=16, out=16, labels=None, nvoc=3, n_add=2, w=256, wbytes=ws: lib.rb_items_run(  # noqa: E731
        C.byref(a), G, nvoc, n_add, 10, 64, 16, 1, layout, corpus, 16, 16, 16, out, None, labels, None, w, wbytes, None)
    assert run(out=None) == -1 and run(corpus=None) == -1
    assert run(layout=2) == -1
    assert run(labels=16, nvoc=126, n_add=5) == -1   # V = 259 views: more than the label broadcast holds
    assert run(corpus=8) == -2
    assert run(w=None) == -3 and run(wbytes=100) == -3
    assert run(G=0, corpus=None, out=None) == 0


def _rows_reference(indices, N, nvoc, extra):
    """The batch's corpus rows as ItemBatcher packs them: per item the vocoded copies, then the anchor; then every item's
    additional bona fide utterances."""
    rows = [N + i * nvoc + v if v < nvoc else i for i in indices for v in range(nvoc + 1)]
    return np.array(rows + list(np.asarray(extra, dtype=np.int64).reshape(-1)), dtype=np.int32)


def test_row_map_helpers():
    """The corpus-row map restated here and ItemBatcher's view table / labels, on which rb_items_run's assembly relies."""
    from scl_deepfake_audio_detection_b200 import multiview
    assert _rows_reference([2, 0], 5, 2, [[1, 4], [3, 2]]).tolist() == [5 + 4, 5 + 5, 2, 5, 5 + 1, 0, 1, 4, 3, 2]
    assert _rows_reference([1], 3, 0, np.zeros((1, 0))).tolist() == [1]
    vr = multiview.item_view_rows(2, 2, 6 + np.arange(4).reshape(2, 2))
    assert vr.tolist() == [[2, -3, 6, 7, 0, 1, -1, -2], [5, -6, 8, 9, 3, 4, -4, -5]]
    assert multiview.item_labels(2, 2).tolist() == [1, 1, 1, 1, 0, 0, 0, 0]
    assert multiview.item_view_rows(1, 0).tolist() == [[0, -1]] and multiview.item_labels(0, 0).tolist() == [1, 1]


# ---------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def eng():
    from scl_deepfake_audio_detection_b200.engine import Engine
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return Engine(0)


def _digest(key, pos):
    return {"pos": int(pos), "key_sha1": hashlib.sha1(np.asarray(key, dtype=np.uint32).tobytes()).hexdigest()}


def _same_stream(end_row, state):
    """A device end state (key[624], pos as int32 bit patterns) continues exactly like numpy's state ``state``."""
    a, b = np.random.RandomState(), np.random.RandomState()
    a.set_state(("MT19937", np.asarray(end_row[:624]).view(np.uint32), int(end_row[624])))
    b.set_state(state)
    return np.array_equal(a.random_sample(700), b.random_sample(700))


class Corpus:
    """A synthetic corpus: ``waves[name]`` for ``<dir>/<name>`` and ``<dir>/<vocoder>_<name>``."""

    def __init__(self, lens, nvoc, seed=0, voc_lens=None):
        rs = np.random.RandomState(seed)
        self.ids = [f"u{k}.wav" for k in range(len(lens))]
        self.vocoders = [f"voc{v}" for v in range(nvoc)]
        self.waves = {}
        for k, name in enumerate(self.ids):
            self.waves[name] = (0.2 * rs.standard_normal(lens[k])).astype(np.float32)
            for v, voc in enumerate(self.vocoders):
                L = voc_lens[k][v] if voc_lens is not None else max(1, lens[k] + int(rs.randint(-40, 41)))
                self.waves[voc + "_" + name] = ((0.9 if v % 2 else 0.1) * rs.uniform(-1, 1, L)).astype(np.float32)

    def load(self, path):
        return self.waves[os.path.basename(path)]


def _batcher(eng, c, n_add, trim, repeat_pad=True):
    from scl_deepfake_audio_detection_b200 import multiview
    dc = multiview.DeviceCorpus(c.ids, "/data", c.load, c.vocoders, engine=eng)
    return multiview.SeededItemBatcher(ARGS, dc, num_additional_real=n_add, trim_length=trim, repeat_pad=repeat_pad)


def _check_items(bat, c, indices, seeds, n_add, trim, repeat_pad=True, check_plan=False):
    """Run the batch once and compare every item with the numpy reference, its end state and (optionally) its plan."""
    from scl_deepfake_audio_detection_b200 import plans
    G = len(indices)
    end = torch.empty((G, 625), dtype=torch.int32, device="cuda")
    state = np.random.get_state()
    ids, data, labels, out_len = bat.items(indices, seeds, end_state=end)
    torch.cuda.synchronize()
    after = np.random.get_state()
    assert after[2] == state[2] and np.array_equal(after[1], state[1]), "the device path must leave numpy's stream alone"
    assert ids == [c.ids[i] for i in indices]
    data, labels, out_len, end = data.cpu().numpy(), labels.cpu().numpy(), out_len.cpu().numpy(), end.cpu().numpy()
    drawn = bat.draw(indices, seeds, end_state=True) if check_plan else None
    nvoc = len(c.vocoders)
    ref_plans, extras, starts = [], [], []
    for g, (idx, s) in enumerate(zip(indices, seeds)):
        np.random.seed(s)
        utt, ref, lab = orc.dataset_item(idx, c.ids, c.load, ARGS, c.vocoders, n_add, trim, repeat_pad=repeat_pad)
        ref_state = np.random.get_state()
        n = ref.shape[0]
        assert int(out_len[g]) == n, g
        got = data[g]
        assert np.max(np.abs(got[:n].astype(np.float64) - ref), initial=0.0) <= 1e-5, (g, idx, s)
        copies = [0] + list(range(2, 2 + n_add + nvoc))
        assert np.array_equal(got[:n, copies], ref[:, copies]), (g, idx, s)
        assert not np.any(got[n:]), "nothing is written past out_len"
        assert np.array_equal(labels[g], lab)
        assert _same_stream(end[g], ref_state), (g, idx, s)
        if check_plan:  # numpy's own draws for this item: the planner's calls, then choice and crop
            np.random.seed(s)
            L = [c.waves[v + "_" + c.ids[idx]].shape[0] for v in c.vocoders] + [c.waves[c.ids[idx]].shape[0]]
            ref_plans += [plans.draw_for_algo(n_, SR, ARGS, 5) for n_ in L]
            others = [k for k in range(len(c.ids)) if k != idx]
            extras.append(np.random.choice(others, n_add, replace=False))
            starts.append(int(np.random.rand() * (L[-1] - trim)) if L[-1] >= trim else 0)
    if check_plan:
        torch.cuda.synchronize()
        eng = bat.corpus.eng
        got = eng.download_plan(drawn["plan"])
        ref = plans.pack(ref_plans, ld=bat.corpus.ld)
        for name in ("lnl_tap_off", "isd_off", "isd_idx", "isd_fr"):
            assert np.array_equal(getattr(ref, name), getattr(got, name)), name
        rt = np.asarray(ref.lnl_taps, np.float32)
        err = np.abs(got.lnl_taps.astype(np.float64) - rt) / np.spacing(np.maximum(np.abs(rt), np.float32(1e-30)))
        assert float(np.max(err)) <= 1.0, "taps more than 1 ulp(fp32) from numpy"
        assert np.array_equal(drawn["start"].cpu().numpy(), starts)
        N = len(c.ids)
        want_rows = _rows_reference(indices, N, nvoc, np.array(extras).reshape(G, n_add))
        assert np.array_equal(drawn["src_row"].cpu().numpy(), want_rows)
        lens = np.array([c.waves[n_].shape[0] for n_ in c.ids] + [c.waves[v + "_" + n_].shape[0] for n_ in c.ids for v in c.vocoders])
        assert np.array_equal(drawn["row_len"].cpu().numpy(), lens[want_rows])
        assert np.array_equal(drawn["end_state"].cpu().numpy(), end)


@pytest.mark.gpu
@pytest.mark.parametrize("idx", [0, 3])
def test_items_match_reference_getitem(eng, golden2, idx):
    """Fixtures produced by the reference's own Dataset_for with np.random.seed(8000 + idx) before __getitem__(idx): the views,
    the labels and the digest of the stream state after the item (which pins the chained walk's word count)."""
    from scl_deepfake_audio_detection_b200 import multiview
    arrays, meta = golden2
    g = meta["getitem"]
    m = g[f"getitem{idx}"]
    dc = multiview.DeviceCorpus(orc.CORPUS_IDS, "/data", orc.corpus_wave, orc.CORPUS_VOCODERS, engine=eng)
    bat = multiview.SeededItemBatcher(orc.make_args(), dc, num_additional_real=m["num_additional_real"], trim_length=m["trim_length"])
    end = torch.empty((1, 625), dtype=torch.int32, device="cuda")
    np.random.seed(123)
    before = np.random.get_state()
    ids, data, labels, out_len = bat.items([idx], [m["seed"]], end_state=end)
    got = data[0].cpu().numpy()
    after = np.random.get_state()
    assert after[2] == before[2] and np.array_equal(after[1], before[1])
    ref = arrays[f"getitem{idx}_data"]
    assert ids == [m["utt"]] and list(got.shape) == m["shape"] and int(out_len[0]) == m["shape"][0]
    assert np.max(np.abs(got.astype(np.float64) - ref)) <= 1e-5
    for col in (0, 2, 3, 4, 5, 6):
        assert np.array_equal(got[:, col], ref[:, col]), col
    assert np.array_equal(labels[0].cpu().numpy(), arrays[f"getitem{idx}_label"])
    e = end[0].cpu().numpy().view(np.uint32)
    assert _digest(e[:624], e[624]) == {k: m["stream"][k] for k in ("pos", "key_sha1")}


@pytest.mark.gpu
def test_items_oracle_sweep_and_plans(eng):
    """A few hundred items in one call, seeds across the uint32 range, indices including 0 and N-1, ragged lengths around
    the crop length: every item, its plan, its extra utterances, crop start and end state against numpy."""
    rs = np.random.RandomState(5)
    N, nvoc, n_add, trim = 13, 2, 2, 1500
    lens = [1500, 1499, 1, 3000, 700, 2047, 1501, 64, 2500, 1200, 1800, 4000, 999]
    c = Corpus(lens, nvoc, seed=1)
    bat = _batcher(eng, c, n_add, trim)
    G = 300
    indices = [0, N - 1] + list(rs.randint(0, N, G - 2))
    seeds = [0, 1, 2 ** 31, 2 ** 32 - 1] + [int(s) for s in rs.randint(0, 2 ** 32, G - 4, dtype=np.int64)]
    _check_items(bat, c, indices, seeds, n_add, trim, check_plan=True)


EDGES = {
    # name: (bona fide lengths, nvoc, n_add, trim, repeat_pad, explicit vocoded lengths or None)
    "short_anchor_repeat": ([300, 1200, 90], 2, 1, 1000, True, None),
    "short_anchor_zero": ([300, 1200, 90], 2, 1, 1000, False, None),
    "anchor_equals_trim": ([1000, 1000, 999, 1001], 1, 2, 1000, True, None),
    "no_vocoders": ([800, 1600, 2400], 0, 2, 1000, True, None),
    "no_extras": ([800, 1600, 2400], 2, 0, 1000, True, None),
    "two_utterances": ([1700, 600], 1, 1, 1000, True, None),
    "long_rows": ([70001, 66000, 3000], 1, 1, 64000, True, [[65537], [80000], [2000]]),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(EDGES))
def test_items_edge_cases(eng, case):
    lens, nvoc, n_add, trim, repeat_pad, voc = EDGES[case]
    c = Corpus(lens, nvoc, seed=len(case), voc_lens=voc)
    bat = _batcher(eng, c, n_add, trim, repeat_pad)
    N = len(lens)
    indices = [g % N for g in range(3 * N)]
    seeds = [7919 * g + 3 for g in range(3 * N)]
    _check_items(bat, c, indices, seeds, n_add, trim, repeat_pad, check_plan=True)


@pytest.mark.gpu
def test_items_wide_choice(eng):
    """N - 1 > 65536: the choice's permutation no longer fits the shared-memory path and is applied in global memory."""
    N = 70003
    rs = np.random.RandomState(2)
    c = Corpus(list(rs.randint(1, 9, N)), 0, seed=3)
    bat = _batcher(eng, c, 2, 4)
    _check_items(bat, c, [0, N - 1, 4242, 65537, 70000], [11, 12, 13, 14, 2 ** 32 - 1], 2, 4, check_plan=True)


@pytest.mark.gpu
def test_items_batch_independent_and_repeatable(eng):
    """An item is the same bit for bit alone or inside a batch, and two runs give the same result."""
    c = Corpus([1200, 2500, 1800, 3000, 900], 3, seed=9)
    bat = _batcher(eng, c, 2, 1000)
    indices, seeds = [4, 0, 2, 2, 1, 3], [5, 6, 7, 8, 9, 10]
    _, d1, l1, n1 = bat.items(indices, seeds)
    _, d2, l2, n2 = bat.items(indices, seeds)
    assert torch.equal(d1, d2) and torch.equal(l1, l2) and torch.equal(n1, n2)
    for g in (0, 3, 5):
        _, da, la, na = bat.items([indices[g]], [seeds[g]])
        assert torch.equal(da[0], d1[g]) and torch.equal(la[0], l1[g]) and torch.equal(na[0], n1[g])


@pytest.mark.gpu
def test_items_device_inputs_on_a_side_stream_do_not_synchronise(eng):
    from scl_deepfake_audio_detection_b200 import multiview
    c = Corpus([1200, 2500, 1800, 3000], 2, seed=4)
    bat = _batcher(eng, c, 1, 1000)
    indices, seeds = [3, 1, 0, 2], [2 ** 32 - 2, 0, 99, 1234]
    _, ref, ref_lab, _ = bat.items(indices, seeds, layout=multiview.LAYOUT_MODEL)  # also sizes the engine's workspace
    di = torch.tensor(indices, dtype=torch.int32, device="cuda")
    ds = torch.tensor(np.array(seeds, dtype=np.uint32).view(np.int32), device="cuda")
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    torch.cuda.set_sync_debug_mode("error")
    try:
        with torch.cuda.stream(side):
            ids, data, labels, out_len = bat.items(di, ds, layout=multiview.LAYOUT_MODEL)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    side.synchronize()
    assert ids is di
    assert torch.equal(data, ref) and torch.equal(labels, ref_lab)


@pytest.mark.gpu
def test_items_past_the_grid_split(eng):
    """G*(nvoc+1) > 65535 RawBoost rows: the items around the split equal the same items run as a small batch, bit for bit,
    and the numpy reference."""
    rs = np.random.RandomState(8)
    N, nvoc = 40, 3
    c = Corpus(list(rs.randint(8, 40, N)), nvoc, seed=6)
    bat = _batcher(eng, c, 1, 16)
    G = 16400  # 65600 RawBoost rows
    indices = rs.randint(0, N, G)
    seeds = np.arange(G, dtype=np.int64) * 2654435761 % 2 ** 32
    _, data, labels, out_len = bat.items(indices, seeds)
    around = [0, 16382, 16383, 16384, 16385, G - 1]
    _, small, slab, slen = bat.items(indices[around], seeds[around])
    assert torch.equal(data[around], small) and torch.equal(labels[around], slab) and torch.equal(out_len[around], slen)
    _check_items(bat, c, list(indices[around]), list(seeds[around]), 1, 16)

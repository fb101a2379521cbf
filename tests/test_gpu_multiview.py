"""GPU parity of the step after the path (SURVEY.md 8f-1/f-2): batch_pad_for_multiview + view assembly on the device, against
outputs of the unmodified reference (tests/golden/multiview_golden.*, made by oracle/make_golden.py --multiview)."""
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from conftest import GOLDEN_DIR, stream_digest  # noqa: E402
from oracle import golden_files, rawboost_oracle as orc  # noqa: E402  (checker only)


@pytest.fixture(scope="module")
def mv():
    arrays = np.load(os.path.join(GOLDEN_DIR, "multiview_golden.npz"))
    with open(os.path.join(GOLDEN_DIR, "multiview_golden.json")) as f:
        return arrays, json.load(f)


@pytest.fixture(scope="module")
def eng():
    from scl_deepfake_audio_detection_b200.engine import Engine
    assert torch.cuda.is_available()
    return Engine(0)


def test_batch_pad_for_multiview_golden(eng, mv):
    """Every branch of the reference function, bit for bit (samples are copied, indices are integers), and the same draws."""
    from scl_deepfake_audio_detection_b200 import multiview
    arrays, meta = mv
    for key, m in meta["pad"].items():
        flat = arrays[m["input"]]
        views, o = [], 0
        for n in m["lens"]:
            views.append(flat[o:o + n].reshape(n, 1))
            o += n
        np.random.seed(m["seed"])
        out = multiview.batch_pad_for_multiview(views, 16000, m["length"], random_trim_nosil=m["trim"], repeat_pad=m["repeat_pad"])
        assert stream_digest() == m["stream"], key
        got = np.concatenate(out, axis=1)
        assert got.shape == arrays[key].shape, key
        assert np.array_equal(got, arrays[key].astype(np.float32)), key


@pytest.mark.parametrize("layout", [0, 1])
def test_assemble_layouts_and_batching(eng, layout):
    """Several items in one launch, both output layouts, against the oracle's index map."""
    from scl_deepfake_audio_detection_b200 import multiview
    rs = np.random.RandomState(3 + layout)
    G, V, length = 5, 4, 300
    lens = rs.randint(1, 700, size=(G, V))
    lens[1, 0] = 120   # first view shorter than the crop
    lens[3, 0] = 300   # exactly the crop
    waves = [rs.standard_normal(n).astype(np.float32) for n in lens.reshape(-1)]
    x, ln = eng.pack_waveforms(waves)
    for repeat_pad in (False, True):
        starts = [0 if lens[g, 0] < length else int(rs.randint(0, lens[g, 0] - length + 1)) for g in range(G)]
        out, out_len = multiview.assemble(eng, x, ln, V, starts, length, repeat_pad, layout)
        out, out_len = out.cpu().numpy(), out_len.cpu().numpy()
        for g in range(G):
            first = int(lens[g, 0])
            wrap = first < length and repeat_pad
            olen = first if (first < length and not repeat_pad) else length
            assert out_len[g] == olen
            ref = orc.multiview_gather(waves[g * V:(g + 1) * V], first, starts[g], olen, wrap, repeat_pad)
            got = out[g, :olen, :] if layout == 0 else out[g, :, :olen].T
            assert np.array_equal(got, ref.astype(np.float32)), (g, repeat_pad)


def test_item_views_match_reference_item(eng, mv):
    """A whole Dataset item (RawBoost12 on 3 vocoded copies + the anchor, shared crop) in the loader's RNG order."""
    from scl_deepfake_audio_detection_b200 import multiview
    arrays, meta = mv
    args = orc.make_args()
    for key, m in meta["item"].items():
        waves = [orc.synth_utterance(m["first_wave"] + k, m["L"] + 37 * k, bool(k % 2)) for k in range(4)]
        np.random.seed(m["seed"])
        out, out_len = multiview.item_views(eng, [(waves[0], waves[1:])], args, 16000, m["trim"], repeat_pad=True,
                                            random_trim_nosil=True, layout=multiview.LAYOUT_ITEM)
        assert stream_digest() == m["stream"], "draw order / count differs from Dataset_for.__getitem__"
        got = out[0].cpu().numpy()
        assert list(got.shape) == m["shape"] and int(out_len[0]) == m["shape"][0]
        assert np.max(np.abs(got.astype(np.float64) - arrays[key])) <= 1e-5
        # the untouched views (anchor, vocoded copies) are pure copies
        for col in (0, 2, 3, 4):
            assert np.array_equal(got[:, col], arrays[key][:, col])


@pytest.mark.parametrize("L,K", [(64600, 8000), (16000, 1), (5000, 513), (300, 2049), (1, 700)])
def test_reverb_view_matches_reference_arithmetic(eng, L, K):
    """SURVEY.md 8f-4: np.convolve(data, rir) + peak normalisation (audio_augmentor/reverb.py:39-42) on the FIR machinery."""
    from scl_deepfake_audio_detection_b200 import reverb
    rs = np.random.RandomState(L + K)
    x = (0.2 * rs.standard_normal(L)).astype(np.float32)
    rir = (rs.standard_normal(K) * np.exp(-np.arange(K) / max(1.0, K / 6.0))).astype(np.float32)
    y = reverb.reverb_convolve(x, rir)
    ref = orc.reverb_convolve(x, rir)
    assert y.dtype == np.float32 and y.shape == ref.shape == (L + K - 1,)
    assert np.max(np.abs(y.astype(np.float64) - ref)) <= 1e-5
    assert abs(float(np.max(np.abs(y))) - 1.0) <= 1e-6


# ---------------------------------------------------------------------------------------------------------
# round 2: in-place assembly, the loader-level batcher, reduced-traffic streaming forms
# ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def g2():
    arrays = golden_files.load(GOLDEN_DIR, "round2_golden")
    with open(os.path.join(GOLDEN_DIR, "round2_golden.json")) as f:
        return arrays, json.load(f)


def test_assemble_ex_reads_views_in_place(eng):
    """The row-table form equals the regrouped form bit for bit, for both sources, both layouts, with labels."""
    from scl_deepfake_audio_detection_b200 import multiview
    rs = np.random.RandomState(8)
    G, nvoc, length = 3, 3, 500
    per, V = nvoc + 1, 2 * (nvoc + 1)
    lens = rs.randint(200, 900, size=G * per)
    xs = [rs.standard_normal(n).astype(np.float32) for n in lens]
    ys = [rs.standard_normal(n).astype(np.float32) for n in lens]
    x, ln = eng.pack_waveforms(xs)
    y, _ = eng.pack_waveforms(ys, ld=x.shape[1])
    rows = multiview.item_view_rows(G, nvoc)
    starts = [int(max(0, lens[g * per + nvoc] - length) // 2) for g in range(G)]
    for layout in (0, 1):
        for repeat_pad in (False, True):
            regrouped, rl = [], []
            for r in rows.reshape(-1):
                regrouped.append(xs[r] if r >= 0 else ys[-1 - r])
            v, vl = eng.pack_waveforms(regrouped, ld=x.shape[1])
            want, want_len = multiview.assemble(eng, v, vl, V, starts, length, repeat_pad, layout)
            got, got_len, labels = multiview.assemble_ex(eng, x, y, torch.from_numpy(rows.reshape(-1)).cuda(), ln, V, starts, length,
                                                         repeat_pad, layout, view_label=torch.from_numpy(multiview.item_labels(nvoc)))
            assert torch.equal(got, want) and torch.equal(got_len, want_len)
            assert labels.cpu().numpy().tolist() == [multiview.item_labels(nvoc).tolist()] * G


@pytest.mark.parametrize("planner", ["numpy", "native"])
def test_item_batcher_matches_reference_getitem(eng, g2, planner):
    """The whole ``Dataset_for.__getitem__`` (asvspoof_2019_augall_3.py:103-146) against fixtures produced by the reference's
    own class on a synthetic corpus: views, view order, labels and the state of the numpy stream afterwards."""
    from scl_deepfake_audio_detection_b200 import multiview
    arrays, meta = g2
    g = meta["getitem"]
    for idx in (0, 3):
        m = g[f"getitem{idx}"]
        bat = multiview.ItemBatcher(orc.make_args(), g["ids"], "/data", orc.corpus_wave, vocoders=m["vocoders"],
                                    num_additional_real=m["num_additional_real"], trim_length=m["trim_length"], engine=eng, planner=planner)
        np.random.seed(m["seed"])
        ids, data, labels, out_len = bat.items([idx])
        assert stream_digest() == m["stream"], "draw order / count differs from Dataset_for.__getitem__"
        assert ids == [m["utt"]] and list(data.shape[1:]) == m["shape"] and int(out_len[0]) == m["shape"][0]
        ref = arrays[f"getitem{idx}_data"]
        got = data[0].cpu().numpy()
        assert np.max(np.abs(got.astype(np.float64) - ref)) <= 1e-5
        for col in (0, 2, 3, 4, 5, 6):  # anchor, additional bona fide and vocoded copies are pure copies
            assert np.array_equal(got[:, col], ref[:, col]), col
        assert np.array_equal(labels[0].cpu().numpy(), arrays[f"getitem{idx}_label"])


def test_item_batcher_batches_like_consecutive_getitems(eng, g2):
    """Several indices in ONE device pass == the reference's __getitem__ called for them one after another on one stream."""
    from scl_deepfake_audio_detection_b200 import multiview
    _, meta = g2
    g = meta["getitem"]
    m = g["getitem0"]
    bat = multiview.ItemBatcher(orc.make_args(), g["ids"], "/data", orc.corpus_wave, vocoders=m["vocoders"], num_additional_real=2,
                                trim_length=m["trim_length"], engine=eng)
    idxs = [4, 1, 5]
    np.random.seed(77)
    ids, data, labels, _ = bat.items(idxs, layout=multiview.LAYOUT_MODEL)
    after = stream_digest()
    np.random.seed(77)
    for k, idx in enumerate(idxs):
        utt, ref, lab = orc.dataset_item(idx, g["ids"], orc.corpus_wave, orc.make_args(), m["vocoders"], 2, m["trim_length"])
        assert ids[k] == utt and np.array_equal(labels[k].cpu().numpy(), lab)
        assert np.max(np.abs(data[k].cpu().numpy().T.astype(np.float64) - ref)) <= 1e-5
    assert stream_digest() == after


def test_streaming_forms_pcm16_and_device_sink(eng):
    """rb_submit_seeded_ex: 16-bit PCM in == float32 in on the same samples; a device sink holds what the host sink receives;
    device in / device out (plans overlapped with the filtering) == the resident path with a device-drawn plan."""
    from scl_deepfake_audio_detection_b200 import workload
    args = workload.default_args()
    B, L = 24, 20000
    rs = np.random.RandomState(0)
    pcm = rs.randint(-20000, 20000, size=(B, L)).astype(np.int16)
    pcm[3] = np.clip(pcm[3].astype(np.int32) * 2, -32768, 32767).astype(np.int16)
    x = (pcm.astype(np.float32) / 32768.0).astype(np.float32)
    lengths = np.array([L - 17 * u for u in range(B)], dtype=np.int32)
    seeds = np.arange(100, 100 + B, dtype=np.uint32)
    for algo in (5, 2, 3):
        want = eng.process_host_seeded(algo, x, lengths, seeds, 16000, args)
        got = np.zeros_like(x)
        eng.wait_host(eng.submit_host_ex(algo, pcm, "pcm16", lengths, seeds, 16000, args, out=got))
        sink = torch.zeros((B, L), dtype=torch.float32, device="cuda")
        eng.wait_host(eng.submit_host_ex(algo, pcm, "pcm16", lengths, seeds, 16000, args, out=sink))
        sink2 = torch.zeros((B, L), dtype=torch.float32, device="cuda")
        eng.wait_host(eng.submit_host_ex(algo, x, "f32", lengths, seeds, 16000, args, out=sink2))
        xd, ld_, sd = torch.from_numpy(x).cuda(), torch.from_numpy(lengths).cuda(), torch.from_numpy(seeds.view(np.int32)).cuda()
        yd = eng.process_device_seeded(algo, xd, ld_, sd, 16000, args)
        torch.cuda.synchronize()
        for u in range(B):
            n = int(lengths[u])
            assert np.array_equal(got[u, :n], want[u, :n]), (algo, u)
            assert np.array_equal(sink[u, :n].cpu().numpy(), want[u, :n]) and np.array_equal(sink2[u, :n].cpu().numpy(), want[u, :n])
            assert np.array_equal(yd[u, :n].cpu().numpy(), want[u, :n]), (algo, u)
    eng.wait_host(eng.submit_host_ex(5, pcm, "pcm16", lengths, seeds, 16000, args, out=sink))
    h2d, d2h = eng.last_host_traffic()
    assert d2h == 0 and pcm.nbytes <= h2d < x.nbytes  # half the input bytes, nothing copied back

"""DeviceLoader (loader.py) against the real DataLoader it replaces.

The reference side is a real forked ``DataLoader`` over a dataset that runs ``oracle.dataset_item`` (``Dataset_for.__getitem__``
with RawBoost12) in its workers, with torch's own seeding after the same ``torch.manual_seed``. The ids, labels, batch order
and collated structure must be exact and the data within 1e-5, for a ragged 13-utterance corpus held as a ``DeviceCorpus`` and
as both ``PackedCorpus`` dtypes, in both layouts, with and without workers, over two epochs, with a ``chunk_batches`` that
does not divide the epoch. numpy's global stream must end where the real loader leaves it, its cached Gaussian included
(without workers the items draw on it; with workers it is not touched); every batch of
both epochs is held to the end before it is compared (nothing overwritten); torch's RNG must stand where the real loader
leaves it after each ``iter()`` and each epoch; consumption on a non-default stream must give the same batches; and with
workers, building the chunks must make no synchronising CUDA call.
"""
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import rawboost_oracle as orc  # noqa: E402  (checker only)

pytestmark = pytest.mark.gpu

ARGS = orc.make_args()
N_ADD, TRIM = 2, 1000
LENS = [1500, 1499, 700, 3000, 900, 2047, 1501, 64, 2500, 1200, 1800, 4000, 999]
CHUNK = 4  # divides none of the epochs below (13, 7 or 6 batches)


class PcmCorpus:
    """13 ragged bona fide utterances and two vocoded copies each, every sample k / 32768 (16-bit audio as librosa.load gives
    it), so that one set of waveforms feeds the padded corpus, both packed dtypes and the reference."""

    def __init__(self, seed=3):
        rs = np.random.RandomState(seed)
        self.ids = [f"u{k}.wav" for k in range(len(LENS))]
        self.vocoders = ["voc0", "voc1"]
        self.waves = {}
        for k, name in enumerate(self.ids):
            names = [name] + [v + "_" + name for v in self.vocoders]
            for j, nm in enumerate(names):
                L = LENS[k] if j == 0 else max(1, LENS[k] + int(rs.randint(-40, 41)))
                x = (0.9 if j == 2 else 0.1) * rs.uniform(-1, 1, L)
                self.waves[nm] = (np.round(x * 32768).clip(-32768, 32767) / 32768).astype(np.float32)

    def load(self, path):
        return self.waves[os.path.basename(path)]


CORPUS = PcmCorpus()


class RefDataset(torch.utils.data.Dataset):
    """Dataset_for.__getitem__ (RawBoost12, online_aug) as the oracle computes it, run by the real loader's workers."""

    def __init__(self, repeat_pad=True):
        self.repeat_pad = repeat_pad

    def __len__(self):
        return len(CORPUS.ids)

    def __getitem__(self, idx):
        uid, data, label = orc.dataset_item(idx, CORPUS.ids, CORPUS.load, ARGS, CORPUS.vocoders, N_ADD, TRIM,
                                            repeat_pad=self.repeat_pad)
        return uid, torch.from_numpy(data), torch.from_numpy(label)


def _epochs(make, epochs=2):
    """Two epochs of ``make()`` after torch.manual_seed and np.random.seed: (batches, rng after each iter(), rng after each
    epoch, numpy's state at the end)."""
    torch.manual_seed(308)
    np.random.seed(379)
    np.random.standard_normal()  # leaves a cached Gaussian: the items never use it, so it must survive the epochs
    dl = make()
    out, after_iter, after_epoch = [], [], []
    for _ in range(epochs):
        it = iter(dl)
        after_iter.append(torch.get_rng_state())
        out.append(list(it))
        after_epoch.append(torch.get_rng_state())
    return out, after_iter, after_epoch, np.random.get_state(), len(dl)


_REF = {}


def reference(workers, batch_size, drop_last, persistent, repeat_pad=True):
    key = (workers, batch_size, drop_last, persistent, repeat_pad)
    if key not in _REF:
        _REF[key] = _epochs(lambda: torch.utils.data.DataLoader(
            RefDataset(repeat_pad), batch_size=batch_size, shuffle=True, num_workers=workers, drop_last=drop_last,
            persistent_workers=persistent, multiprocessing_context="fork" if workers else None))
    return _REF[key]


_CORPORA = {}


def corpus(kind):
    from scl_deepfake_audio_detection_b200 import multiview
    if kind not in _CORPORA:
        if kind == "device":
            _CORPORA[kind] = multiview.DeviceCorpus(CORPUS.ids, "/data", CORPUS.load, CORPUS.vocoders)
        else:
            _CORPORA[kind] = multiview.PackedCorpus(CORPUS.ids, "/data", CORPUS.load, CORPUS.vocoders, dtype=kind)
    return _CORPORA[kind]


def device_loader(kind, workers, batch_size, drop_last, persistent, layout, repeat_pad=True):
    from scl_deepfake_audio_detection_b200 import loader
    return loader.DeviceLoader(corpus(kind), ARGS, num_additional_real=N_ADD, trim_length=TRIM, repeat_pad=repeat_pad,
                               batch_size=batch_size, shuffle=True, num_workers=workers, drop_last=drop_last,
                               persistent_workers=persistent, layout=layout, chunk_batches=CHUNK)


def _same_stream(a, b):
    """Two numpy states continue alike: the Gaussian cache (compared exactly) and the MT19937 stream."""
    if tuple(a[3:]) != tuple(b[3:]):
        return False
    x, y = np.random.RandomState(), np.random.RandomState()
    x.set_state(a)
    y.set_state(b)
    return np.array_equal(x.standard_normal(3), y.standard_normal(3)) and np.array_equal(x.random_sample(700), y.random_sample(700))


def compare(got, want, layout, workers):
    from scl_deepfake_audio_detection_b200 import multiview
    batches, it_rng, ep_rng, np_end, length = got
    w_batches, w_it_rng, w_ep_rng, w_np_end, w_length = want
    assert length == w_length
    for e in range(len(w_batches)):
        assert torch.equal(it_rng[e], w_it_rng[e]) and torch.equal(ep_rng[e], w_ep_rng[e]), e
        assert len(batches[e]) == len(w_batches[e]), e
        for j, (b, w) in enumerate(zip(batches[e], w_batches[e])):
            assert isinstance(b, list) and len(b) == 3, (e, j)
            ids, data, label = b
            assert isinstance(ids, list) and all(isinstance(u, str) for u in ids) and ids == list(w[0]), (e, j)
            assert data.is_cuda and label.is_cuda and data.dtype == torch.float32 and label.dtype == torch.float32
            ref = w[1].double()
            if layout == multiview.LAYOUT_MODEL:
                ref = ref.transpose(1, 2)
            assert tuple(data.shape) == tuple(ref.shape), (e, j)
            assert float((data.double().cpu() - ref).abs().max()) <= 1e-5, (e, j)
            assert torch.equal(label.cpu(), w[2]), (e, j)
    assert _same_stream(np_end, w_np_end), "numpy's global stream must end where the real loader leaves it"
    if workers:  # the main process's stream is not involved at all
        assert np.array_equal(np_end[1], w_np_end[1]) and np_end[2] == w_np_end[2]


CASES = [(w, bs, dl, p) for w in (0, 3) for bs in (1, 2) for dl in (False, True) for p in (False, True) if not (p and w == 0)]


@pytest.mark.parametrize("workers,batch_size,drop_last,persistent", CASES)
@pytest.mark.parametrize("kind", ["device", "pcm16", "float32"])
@pytest.mark.parametrize("layout", [0, 1])
def test_device_loader_matches_the_real_loader(kind, layout, workers, batch_size, drop_last, persistent):
    want = reference(workers, batch_size, drop_last, persistent)
    got = _epochs(lambda: device_loader(kind, workers, batch_size, drop_last, persistent, layout))
    torch.cuda.synchronize()
    compare(got, want, layout, workers)


@pytest.mark.parametrize("workers", [0, 3])
def test_device_loader_on_a_side_stream(workers):
    """Batches consumed under a non-default stream, and read there, equal the real loader's."""
    want = reference(workers, 2, False, False)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        got = _epochs(lambda: device_loader("pcm16", workers, 2, False, False, 1))
        # work queued on the consumer's stream after each batch arrives, as a training step would
        scaled = [[[b[0], b[1] * 2.0, b[2]] for b in ep] for ep in got[0]]
    side.synchronize()
    halves = [[[b[0], b[1] / 2.0, b[2]] for b in ep] for ep in scaled]
    compare((halves,) + got[1:], want, 1, workers)


@pytest.mark.parametrize("workers", [0, 3])
def test_device_loader_without_repeat_pad(workers):
    """repeat_pad=False: an item whose anchor is shorter than the crop is as long as its anchor, as in the reference."""
    want = reference(workers, 1, False, False, repeat_pad=False)
    got = _epochs(lambda: device_loader("float32", workers, 1, False, False, 0, repeat_pad=False))
    assert any(b[1].shape[1] < TRIM for b in got[0][0]), "the corpus has anchors shorter than the crop"
    compare(got, want, 0, workers)


def test_device_loader_production_does_not_synchronise():
    """Building the chunks makes no synchronising CUDA call (no copy from pageable memory, no read-back) with workers and
    repeat_pad: the host only enqueues, and the batches still equal the real loader's."""
    want = reference(3, 1, False, False)
    corpus("pcm16")  # built, with its uploads, before the check
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        got = _epochs(lambda: device_loader("pcm16", 3, 1, False, False, 0))
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    compare(got, want, 0, 3)

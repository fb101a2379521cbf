"""DeviceLoader (loader.py) with a caller's sampler, batch_sampler and worker_init_fn, against the real DataLoader.

As in test_gpu_device_loader.py, the reference is a real forked ``DataLoader`` over ``oracle.dataset_item`` (``Dataset_for``
with RawBoost12) after the same ``torch.manual_seed`` / ``np.random.seed``, and the device side a ``DeviceLoader`` on the
13-utterance ragged PCM16 corpus with ``chunk_batches=4``, which divides none of the epochs below. ids, labels and collated
structure must be exact, data within 1e-5, and torch's RNG and numpy's global stream must end where the real loader leaves
them. Covered: two ``DistributedSampler`` ranks, each with its own loader on the one GPU (their ids together make the sampler's
padded epoch); ``WeightedRandomSampler`` with replacement, so that a chunk holds one item more than once; an uneven plain-list
``batch_sampler``; the reproducibility notes' ``seed_worker``; production that makes no synchronising CUDA call; indices
refused before anything is enqueued; and, where two GPUs are visible, ranks on devices 0 and 1 iterated while the other
device is current.
"""
import collections
import random

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from torch.utils.data import DistributedSampler, WeightedRandomSampler  # noqa: E402

from test_gpu_device_loader import ARGS, CHUNK, CORPUS, N_ADD, TRIM, RefDataset, compare, corpus  # noqa: E402

pytestmark = pytest.mark.gpu

N = len(CORPUS.ids)
UNEVEN = [[0, 5, 5], [12], [3, 4], [7, 8, 9, 10], [1], [2, 11], [6, 6, 6, 6, 6]]


def seed_worker(worker_id):
    """The recipe of PyTorch's reproducibility notes."""
    worker_seed = torch.initial_seed() % 2 ** 32
    np.random.seed(worker_seed)
    random.seed(worker_seed)


def _epochs(make, epochs=2):
    """``epochs`` epochs of the loader ``make()`` returns with its per-epoch hook, after torch.manual_seed and np.random.seed:
    (batches, rng after each iter(), rng after each epoch, numpy's state at the end, len)."""
    torch.manual_seed(308)
    np.random.seed(379)
    np.random.standard_normal()  # a cached Gaussian the items never use
    dl, hook = make()
    out, after_iter, after_epoch = [], [], []
    for e in range(epochs):
        hook(e)
        it = iter(dl)
        after_iter.append(torch.get_rng_state())
        out.append(list(it))
        after_epoch.append(torch.get_rng_state())
    return out, after_iter, after_epoch, np.random.get_state(), len(dl)


def _no_hook(e):
    pass


def _loader_kw(case):
    """Fresh DataLoader keyword arguments (new sampler objects) and the per-epoch hook of one case."""
    kind, workers, batch_size = case[:3]
    kw = dict(num_workers=workers)
    hook = _no_hook
    if kind == "distributed":
        s = DistributedSampler(range(N), num_replicas=2, rank=case[3], shuffle=True, seed=23)
        kw.update(batch_size=batch_size, sampler=s)
        hook = s.set_epoch
    elif kind == "weighted":
        kw.update(batch_size=batch_size, sampler=WeightedRandomSampler([1.0 + (k % 3) for k in range(N)], N + 7, replacement=True))
    elif kind == "uneven":
        kw.update(batch_sampler=[list(b) for b in UNEVEN])
    elif kind == "seed_worker":
        kw.update(batch_size=batch_size, shuffle=True, worker_init_fn=seed_worker, persistent_workers=case[3])
    elif kind == "distributed+init":
        s = DistributedSampler(range(N), num_replicas=2, rank=1, shuffle=True, seed=5)
        kw.update(batch_size=batch_size, sampler=s, worker_init_fn=seed_worker)
        hook = s.set_epoch
    return kw, hook


_REF = {}


def reference(case):
    if case not in _REF:
        def make():
            kw, hook = _loader_kw(case)
            return torch.utils.data.DataLoader(RefDataset(), multiprocessing_context="fork" if kw["num_workers"] else None,
                                               **kw), hook
        _REF[case] = _epochs(make)
    return _REF[case]


def device_loader(case, corpus_=None):
    from scl_deepfake_audio_detection_b200 import loader
    kw, hook = _loader_kw(case)
    return loader.DeviceLoader(corpus_ or corpus("pcm16"), ARGS, num_additional_real=N_ADD, trim_length=TRIM,
                               chunk_batches=CHUNK, **kw), hook


DIST = [("distributed", w, bs, r) for w in (0, 3) for bs in (1, 2) for r in (0, 1)]


@pytest.mark.parametrize("case", DIST, ids=str)
def test_distributed_sampler_rank(case):
    want = reference(case)
    got = _epochs(lambda: device_loader(case))
    torch.cuda.synchronize()
    compare(got, want, 0, case[1])


@pytest.mark.parametrize("workers", [0, 3])
@pytest.mark.parametrize("batch_size", [1, 2])
def test_distributed_ranks_make_the_padded_epoch(workers, batch_size):
    """Each epoch, the two ranks' ids together are the sampler's padded epoch: every utterance, and one twice (13 = 2 * 7 - 1)."""
    ranks = [[[u for b in ep for u in b[0]] for ep in _epochs(lambda: device_loader(("distributed", workers, batch_size, r)))[0]]
             for r in (0, 1)]
    for e in range(2):
        count = collections.Counter(ranks[0][e] + ranks[1][e])
        assert set(count) == set(CORPUS.ids) and sorted(count.values()) == [1] * 12 + [2], e
    assert ranks[0][0] != ranks[0][1], "set_epoch reshuffles"


@pytest.mark.parametrize("workers", [0, 3])
def test_weighted_sampler_repeats_items_in_a_chunk(workers):
    case = ("weighted", workers, 2)
    want = reference(case)
    chunk_ids = [[u for b in want[0][0][k:k + CHUNK] for u in b[0]] for k in range(0, len(want[0][0]), CHUNK)]
    assert any(len(set(c)) < len(c) for c in chunk_ids), "some chunk holds one item twice"
    got = _epochs(lambda: device_loader(case))
    torch.cuda.synchronize()
    compare(got, want, 0, workers)


@pytest.mark.parametrize("workers", [0, 3])
def test_uneven_batch_sampler(workers):
    case = ("uneven", workers, 1)
    want = reference(case)
    got = _epochs(lambda: device_loader(case))
    torch.cuda.synchronize()
    assert [len(b[0]) for b in got[0][0]] == [len(b) for b in UNEVEN]
    compare(got, want, 0, workers)


@pytest.mark.parametrize("persistent", [False, True])
def test_seed_worker(persistent):
    case = ("seed_worker", 3, 2, persistent)
    want = reference(case)
    got = _epochs(lambda: device_loader(case))
    torch.cuda.synchronize()
    compare(got, want, 0, 3)


def test_production_with_sampler_and_init_fn_does_not_synchronise():
    """A DistributedSampler, workers and a worker_init_fn: building the chunks makes no synchronising CUDA call (the init
    children are forked from this process, which holds a CUDA context, and make no CUDA call themselves)."""
    import multiprocessing
    case = ("distributed+init", 3, 1)
    want = reference(case)
    corpus("pcm16")
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        got = _epochs(lambda: device_loader(case))
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    compare(got, want, 0, 3)
    assert multiprocessing.active_children() == []


@pytest.mark.parametrize("workers", [0, 3])
def test_bad_index_raises_before_anything_is_enqueued(workers, monkeypatch):
    from scl_deepfake_audio_detection_b200 import loader
    dl = loader.DeviceLoader(corpus("pcm16"), ARGS, num_additional_real=N_ADD, trim_length=TRIM, num_workers=workers,
                             chunk_batches=1, batch_sampler=[[0], [1, 2], [N]])
    produced = []
    monkeypatch.setattr(dl, "_produce", lambda *a: produced.append(a))
    with pytest.raises(IndexError):
        next(iter(dl))
    assert produced == []


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_ranks_on_two_devices():
    """Rank r on device r, iterated while device 1 - r is current: the batches live on device r and equal the real loader's."""
    from scl_deepfake_audio_detection_b200 import multiview
    from scl_deepfake_audio_detection_b200.engine import Engine
    for r in (0, 1):
        case = ("distributed", 3, 2, r)
        want = reference(case)
        c = multiview.PackedCorpus(CORPUS.ids, "/data", CORPUS.load, CORPUS.vocoders, dtype="pcm16", engine=Engine(r))
        with torch.cuda.device(1 - r):
            got = _epochs(lambda: device_loader(case, c))
            assert all(b[1].device == torch.device("cuda", r) for ep in got[0] for b in ep)
        torch.cuda.synchronize(r)
        compare(got, want, 0, 3)

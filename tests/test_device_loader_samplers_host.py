"""loader.epoch_schedule with a caller's sampler, batch_sampler and worker_init_fn, against the installed torch's DataLoader,
without a GPU.

As in test_device_loader_host.py, a real ``DataLoader`` (the platform's default worker context) runs over a stub dataset of
13 items whose items report their index, the worker that built them and numpy's 625 state words at item start, then draw
``1 + i % 5`` values. ``epoch_schedule``, given fresh sampler objects built alike, must predict over three epochs: the batches
and their order, the worker of each batch and ``len()``; each worker's first state (after the ``worker_init_fn``, where one
is given); every later state, replayed on the host from the predicted start; and torch's global RNG state after each
``iter()`` and after each epoch. ``set_epoch(e)`` is called on a ``DistributedSampler`` before each epoch on both sides.
"""
import multiprocessing
import random

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from torch.utils.data import (DistributedSampler, SequentialSampler, SubsetRandomSampler, WeightedRandomSampler,  # noqa: E402
                              get_worker_info)

from scl_deepfake_audio_detection_b200 import loader, multiview  # noqa: E402

N = 13
EPOCHS = 3


class StateDataset(torch.utils.data.Dataset):
    def __len__(self):
        return N

    def __getitem__(self, i):
        info = get_worker_info()
        st = np.random.get_state()
        words = np.append(st[1], st[2]).astype(np.int64)
        np.random.random_sample(1 + i % 5)
        return i, (info.id if info else -1), words


def _words(rs):
    st = rs.get_state()
    return np.append(st[1], st[2]).astype(np.int64)


# -- worker_init_fn: module-level, so that a spawned child can unpickle them ----------------------------------------------------
def seed_worker(worker_id):
    """The recipe of PyTorch's reproducibility notes."""
    worker_seed = torch.initial_seed() % 2 ** 32
    np.random.seed(worker_seed)
    random.seed(worker_seed)


def draw_by_id(worker_id):
    np.random.random_sample(get_worker_info().id + 1)


def check_info(worker_id):
    info = get_worker_info()
    assert info.id == worker_id and info.num_workers == 3 and info.seed == torch.initial_seed(), info
    np.random.random_sample(info.seed % 7 + 1)


def fail_in_worker_1(worker_id):
    if worker_id == 1:
        raise ValueError("worker_init_fn failed on purpose")


# -- the cases: each returns fresh DataLoader keyword arguments and a hook called before every epoch --------------------------
def _no_hook(e):
    pass


def distributed(R, r, shuffle, drop_last, workers, persistent, batch_size):
    def make():
        s = DistributedSampler(StateDataset(), num_replicas=R, rank=r, shuffle=shuffle, seed=17, drop_last=drop_last)
        return dict(batch_size=batch_size, sampler=s, num_workers=workers, persistent_workers=persistent), s.set_epoch
    return make


def weighted(own_generator, workers):
    def make():
        g = torch.Generator().manual_seed(41) if own_generator else None
        s = WeightedRandomSampler([1.0 + (k % 4) for k in range(N)], N + 4, replacement=True, generator=g)
        return dict(batch_size=2, sampler=s, num_workers=workers), _no_hook
    return make


def subset(workers):
    def make():
        return dict(batch_size=2, sampler=SubsetRandomSampler([12, 0, 3, 4, 9, 7, 1, 11]), num_workers=workers), _no_hook
    return make


UNEVEN = [[0, 5, 5], [12], [3, 4], [7, 8, 9, 10], [1], [2, 11], [6, 6, 6, 6, 6]]


def uneven(workers):
    def make():
        return dict(batch_sampler=[list(b) for b in UNEVEN], num_workers=workers), _no_hook
    return make


def with_init(fn, persistent, context=None):
    def make():
        kw = dict(batch_size=2, shuffle=True, num_workers=3, persistent_workers=persistent, worker_init_fn=fn)
        if context is not None:
            kw["multiprocessing_context"] = context
        return kw, _no_hook
    return make


def real_epochs(make):
    torch.manual_seed(2024)
    np.random.seed(5)
    kw, hook = make()
    real = torch.utils.data.DataLoader(StateDataset(), **kw)
    epochs = []
    for e in range(EPOCHS):
        hook(e)
        it = iter(real)
        after_iter = torch.get_rng_state()
        batches = [(b[0].tolist(), b[1].tolist(), b[2].numpy()) for b in it]
        epochs.append((after_iter, batches, torch.get_rng_state(), np.random.get_state()))
    real_len = len(real)
    del it, real
    return epochs, real_len


def check_schedule(make, schedule_context=None):
    """The real loader's epochs of ``make()``'s arguments against epoch_schedule's prediction from a second ``make()``."""
    epochs, real_len = real_epochs(make)
    torch.manual_seed(2024)
    np.random.seed(5)
    kw, hook = make()
    if schedule_context is not None:
        kw["multiprocessing_context"] = schedule_context
    workers, persistent = kw.get("num_workers", 0), kw.get("persistent_workers", False)
    args = dict(batch_size=kw.get("batch_size", 1), shuffle=kw.get("shuffle", False), drop_last=kw.get("drop_last", False),
                sampler=kw.get("sampler"), batch_sampler=kw.get("batch_sampler"))
    assert len(loader.index_sampler(N, **args)) == real_len
    carried = None
    for e, (after_iter, batches, after_epoch, np_after) in enumerate(epochs):
        hook(e)
        if workers == 0:  # the base seed at iter(), the sampler's pass at the first next()
            it = iter(loader.index_sampler(N, **args))
            loader.draw_base_seed(None)
            assert torch.equal(torch.get_rng_state(), after_iter), e
            order = loader.checked_batches(it, N)
            s = loader.EpochSchedule(order, *loader.split_batches(order, 0), None, None)
        else:
            s = loader.epoch_schedule(N, num_workers=workers, persistent_workers=persistent, first_iter=e == 0,
                                      worker_init_fn=kw.get("worker_init_fn"),
                                      multiprocessing_context=kw.get("multiprocessing_context"), **args)
            assert torch.equal(torch.get_rng_state(), after_iter), e
            assert (s.worker_states is None) == (persistent and e > 0)
        assert torch.equal(torch.get_rng_state(), after_epoch), e
        assert [b[0] for b in batches] == s.batches, e
        assert [b[1] for b in batches] == [[w if workers else -1] * len(b[0]) for w, b in zip(s.batch_worker, batches)], e
        streams = []
        for w in range(max(1, workers)):
            items = [(i, words) for b in batches for i, wid, words in zip(*b) if wid == (w if workers else -1)]
            assert [i for i, _ in items] == s.worker_indices[w], (e, w)
            if workers == 0:
                rs = carried[0] if carried else np.random.RandomState(5)
            elif s.worker_states is not None:
                rs = np.random.RandomState()
                rs.set_state(multiview.numpy_state(s.worker_states[w]))
                if items:
                    assert np.array_equal(items[0][1], s.worker_states[w].astype(np.int64)), (e, w)
            else:
                rs = carried[w]
            for k, (i, words) in enumerate(items):
                assert np.array_equal(words, _words(rs)), (e, w, k)
                rs.random_sample(1 + i % 5)
            streams.append(rs)
        if workers == 0:
            assert np.array_equal(_words(streams[0]), np.append(np_after[1], np_after[2])), e
        carried = streams
    return epochs


DIST = [(R, r, sh, dl, w, p, bs) for R in (2, 3) for r in range(R) for sh in (False, True) for dl in (False, True)
        for w, p in ((0, False), (3, False), (3, True)) for bs in (1, 2)]


@pytest.mark.parametrize("R,rank,shuffle,drop_last,workers,persistent,batch_size", DIST)
def test_distributed_sampler(R, rank, shuffle, drop_last, workers, persistent, batch_size):
    epochs = check_schedule(distributed(R, rank, shuffle, drop_last, workers, persistent, batch_size))
    ids = [i for b in epochs[0][1] for i in b[0]]
    if not drop_last:  # 13 is divisible by neither R: the sampler pads with repeated indices
        assert len(ids) == -(-N // R)


@pytest.mark.parametrize("workers", [0, 3])
@pytest.mark.parametrize("own_generator", [False, True])
def test_weighted_random_sampler(own_generator, workers):
    epochs = check_schedule(weighted(own_generator, workers))
    ids = [i for b in epochs[0][1] for i in b[0]]
    assert len(ids) == N + 4 and len(set(ids)) < len(ids), "drawn with replacement: some index comes twice"


@pytest.mark.parametrize("workers", [0, 3])
def test_subset_random_sampler(workers):
    check_schedule(subset(workers))


@pytest.mark.parametrize("workers", [0, 3])
def test_uneven_batch_sampler_list(workers):
    epochs = check_schedule(uneven(workers))
    assert [b[0] for b in epochs[0][1]] == UNEVEN


@pytest.mark.parametrize("persistent", [False, True])
@pytest.mark.parametrize("fn", [seed_worker, draw_by_id, check_info], ids=lambda f: f.__name__)
def test_worker_init_fn(fn, persistent):
    check_schedule(with_init(fn, persistent))


def test_worker_init_fn_in_spawned_children():
    """The children start from the context given (here by name); what the function leaves does not depend on it."""
    check_schedule(with_init(draw_by_id, False), schedule_context="spawn")


def test_worker_init_fn_not_called_without_workers():
    calls = []
    s = loader.epoch_schedule(N, 2, worker_init_fn=calls.append)
    assert calls == [] and s.worker_states is None


def test_worker_init_fn_that_raises():
    torch.manual_seed(0)
    with pytest.raises(RuntimeError, match=r"worker process 1(.|\n)*worker_init_fn failed on purpose"):
        loader.epoch_schedule(N, 2, num_workers=3, worker_init_fn=fail_in_worker_1)
    assert multiprocessing.active_children() == []


# -- refusals: DataLoader's own, then the index checks, each before anything is built ------------------------------------------
def test_refuses_what_the_loader_refuses():
    seq = SequentialSampler(range(N))
    cases = [dict(sampler=seq, shuffle=True), dict(batch_sampler=[[0]], batch_size=2), dict(batch_sampler=[[0]], shuffle=True),
             dict(batch_sampler=[[0]], sampler=seq), dict(batch_sampler=[[0]], drop_last=True)]
    for kw in cases:
        with pytest.raises(ValueError) as real:
            torch.utils.data.DataLoader(StateDataset(), **kw)
        with pytest.raises(ValueError) as ours:
            loader.epoch_schedule(N, **kw)
        assert str(ours.value) == str(real.value), kw
    for ctx, err in (("no-such-method", ValueError), (object(), TypeError)):
        with pytest.raises(err):
            loader.epoch_schedule(N, num_workers=2, multiprocessing_context=ctx)
    with pytest.raises(ValueError):
        loader.epoch_schedule(N, multiprocessing_context="fork")  # a context needs workers


class _Unsized(torch.utils.data.Sampler):
    def __iter__(self):
        return iter(range(N))


def test_len_of_an_unsized_sampler_raises_as_torch_does():
    with pytest.raises(TypeError):
        len(torch.utils.data.DataLoader(StateDataset(), batch_size=2, sampler=_Unsized()))
    with pytest.raises(TypeError):
        len(loader.index_sampler(N, 2, sampler=_Unsized()))
    assert loader.epoch_schedule(N, 2, sampler=_Unsized()).batches == [[2 * k, 2 * k + 1] for k in range(6)] + [[12]]


@pytest.mark.parametrize("bad,err", [([[0, 1], [N]], IndexError), ([[0, 1], [-1]], IndexError), ([[0, 1.0]], TypeError),
                                     ([[0], ["3"]], TypeError), ([[0], [True]], TypeError), ([[0], []], ValueError)],
                         ids=["past the end", "negative", "float", "str", "bool", "empty batch"])
def test_bad_indices_raise_before_anything_is_built(bad, err, monkeypatch):
    def must_not_run(*a):
        raise AssertionError("worker start states computed for a refused epoch")
    monkeypatch.setattr(loader, "_init_states", must_not_run)
    monkeypatch.setattr(loader, "worker_start_states", must_not_run)
    with pytest.raises(err):
        loader.epoch_schedule(N, num_workers=2, batch_sampler=bad, worker_init_fn=seed_worker)
    with pytest.raises(err):
        loader.checked_batches(bad, N)


def test_checked_batches_keeps_repeats_and_integer_types():
    assert loader.checked_batches([[np.int64(3), 3], torch.tensor([12, 0]), (5,)], N) == [[3, 3], [12, 0], [5]]

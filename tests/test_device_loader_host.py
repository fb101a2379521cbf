"""The epoch schedule of loader.py against the installed torch's own DataLoader, and serve_items' routing, without a GPU.

A real ``DataLoader`` (default sampler and collate, the platform's default worker context) runs over a stub dataset whose
items report their index, the worker that built them and numpy's 625 state words at item start, then draw a number of values
that depends on the index, so that every later state depends on which worker got which index. ``epoch_schedule`` must
predict, over three epochs: the batches and their order, the worker of each batch and ``len()``; each worker's first state;
every later state, replayed on the host from the predicted start; and torch's global RNG state after each ``iter()`` and after
each epoch.
"""
import logging
import types

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from scl_deepfake_audio_detection_b200 import loader, multiview  # noqa: E402

N = 13


class StateDataset(torch.utils.data.Dataset):
    def __len__(self):
        return N

    def __getitem__(self, i):
        info = torch.utils.data.get_worker_info()
        st = np.random.get_state()
        words = np.append(st[1], st[2]).astype(np.int64)
        np.random.random_sample(1 + i % 5)
        return i, (info.id if info else -1), words


def _draw(rs, i):
    rs.random_sample(1 + i % 5)


def _words(rs):
    st = rs.get_state()
    return np.append(st[1], st[2]).astype(np.int64)


CONFIGS = [(w, sh, bs, dl, gen, pers) for w in (0, 1, 3, 8) for sh in (False, True) for bs in (1, 3) for dl in (False, True)
           for gen in (False, True) for pers in (False, True) if not (pers and w == 0)]


@pytest.mark.parametrize("workers,shuffle,batch_size,drop_last,seeded_generator,persistent", CONFIGS)
def test_schedule_matches_the_real_loader(workers, shuffle, batch_size, drop_last, seeded_generator, persistent):
    def gen():
        return torch.Generator().manual_seed(77) if seeded_generator else None

    # the real loader: three epochs after torch.manual_seed, numpy's global stream seeded for the no-worker case
    torch.manual_seed(2024)
    np.random.seed(5)
    real = torch.utils.data.DataLoader(StateDataset(), batch_size=batch_size, shuffle=shuffle, num_workers=workers,
                                       drop_last=drop_last, generator=gen(), persistent_workers=persistent)
    epochs = []
    for _ in range(3):
        it = iter(real)
        after_iter = torch.get_rng_state()
        batches = [(b[0].tolist(), b[1].tolist(), b[2].numpy()) for b in it]
        epochs.append((after_iter, batches, torch.get_rng_state(), np.random.get_state()))
    real_len = len(real)
    del it, real

    # the schedule, from the same seeds
    torch.manual_seed(2024)
    np.random.seed(5)
    g = gen()
    assert len(loader.batch_sampler(N, batch_size, shuffle, drop_last, g)) == real_len
    carried = None
    for e, (after_iter, batches, after_epoch, np_after) in enumerate(epochs):
        if workers == 0:  # the loader draws its base seed at iter() and starts the sampler's pass at the first next()
            loader.draw_base_seed(g)
            assert torch.equal(torch.get_rng_state(), after_iter), e
            order = [list(b) for b in loader.batch_sampler(N, batch_size, shuffle, drop_last, g)]
            s = loader.EpochSchedule(order, *loader.split_batches(order, 0), None, None)
        else:
            s = loader.epoch_schedule(N, batch_size, shuffle, workers, drop_last, g, persistent, first_iter=e == 0)
            assert torch.equal(torch.get_rng_state(), after_iter), e
            assert (s.worker_states is None) == (persistent and e > 0)
        assert torch.equal(torch.get_rng_state(), after_epoch), e
        assert [b[0] for b in batches] == s.batches, e
        assert [b[1] for b in batches] == [[w if workers else -1] * len(b[0]) for w, b in zip(s.batch_worker, batches)], e
        # numpy: each worker's first state, then every later state replayed on the host from the predicted start
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
                _draw(rs, i)
            streams.append(rs)
        if workers == 0:
            assert np.array_equal(_words(streams[0]), np.append(np_after[1], np_after[2])), e
        carried = streams


def test_epoch_schedule_refuses_what_the_loader_refuses():
    with pytest.raises(ValueError):
        loader.epoch_schedule(N, 1, num_workers=0, persistent_workers=True)
    with pytest.raises(ValueError):
        loader.epoch_schedule(N, 0)
    with pytest.raises(ValueError):
        loader.epoch_schedule(N, 1, num_workers=-1)
    with pytest.raises(ValueError):
        loader.epoch_schedule(0, 1, shuffle=True)   # RandomSampler refuses an empty dataset, as DataLoader does
    assert loader.epoch_schedule(0, 1).batches == []


# -- serve_items: routing and fallbacks, against a stand-in Dataset_for with the reference's signature -----------------------
class StandInDataset:
    """``Dataset_for``'s constructor signature (main.py passes the dataset kwargs of its YAML); like the reference, it sets
    ``args.online_aug``."""

    def __init__(self, args, list_IDs, labels, base_dir, vocoders=[], augmentation_methods=[], num_additional_real=2,
                 trim_length=64000, online_aug=False, aug_dir=None, repeat_pad=True):
        args.online_aug, args.aug_dir = online_aug, aug_dir
        self.list_IDs = list_IDs

    def __len__(self):
        return len(self.list_IDs)

    def __getitem__(self, i):
        return i


@pytest.fixture
def served(monkeypatch):
    """serve_items over a stand-in loader module; PackedCorpus and DeviceLoader record their arguments instead of touching a
    device."""
    made = {"corpora": [], "loaders": []}

    class FakeCorpus:
        def __init__(self, *a, **kw):
            made["corpora"].append((a, kw))

    class FakeLoader:
        def __init__(self, corpus, args, **kw):
            self.corpus, self.args, self.kw = corpus, args, kw
            made["loaders"].append(self)

    monkeypatch.setattr(multiview, "PackedCorpus", FakeCorpus)
    monkeypatch.setattr(loader, "DeviceLoader", FakeLoader)
    module = types.SimpleNamespace(Dataset_for=type("Dataset_for", (StandInDataset,), {}))
    real_init, real_loader = module.Dataset_for.__init__, torch.utils.data.DataLoader
    from scl_deepfake_audio_detection_b200 import dropin
    svc = dropin.serve_items(module, load_audio="reader", dtype="float32", location="host")
    try:
        yield module, svc, made, FakeLoader
    finally:
        svc.close()
    assert module.Dataset_for.__init__ is real_init and torch.utils.data.DataLoader is real_loader


def _dataset(module, ids=("a.wav", "b.wav", "c.wav"), **kw):
    args = types.SimpleNamespace()
    kw = {"vocoders": ["hifigan"], "augmentation_methods": ["RawBoost12"], "num_additional_real": 1, "trim_length": 1000,
          "online_aug": True, "aug_dir": "", "repeat_pad": False, **kw}
    return module.Dataset_for(args, list(ids), {}, "/data", **kw), args


def test_serve_items_routes_the_reference_call(served):
    module, svc, made, FakeLoader = served
    ds, args = _dataset(module)
    gen = torch.Generator()
    dl = torch.utils.data.DataLoader(ds, batch_size=2, shuffle=True, num_workers=8, pin_memory=True, drop_last=True,
                                     timeout=5, multiprocessing_context="fork", generator=gen, prefetch_factor=4,
                                     persistent_workers=True)
    assert isinstance(dl, FakeLoader) and dl.args is args
    factory = torch.utils.data.DataLoader
    assert factory.__wrapped__ is svc._real_loader and factory.__name__ == "DataLoader" and "__iter__" not in vars(factory)
    assert dl.kw == {"num_additional_real": 1, "trim_length": 1000, "repeat_pad": False, "batch_size": 2, "shuffle": True,
                     "num_workers": 8, "drop_last": True, "generator": gen, "persistent_workers": True}
    assert made["corpora"] == [((("a.wav", "b.wav", "c.wav"), "/data", "reader", ("hifigan",)),
                                {"dtype": "float32", "location": "host"})]
    # positional arguments as DataLoader takes them; the same corpus again is not built twice
    ds2, _ = _dataset(module, trim_length=500)
    dl2 = torch.utils.data.DataLoader(ds2, 1, False, None, None, 0)
    assert dl2.corpus is dl.corpus and dl2.kw["trim_length"] == 500 and dl2.kw["shuffle"] is False
    assert dl2.kw["batch_size"] == 1 and dl2.kw["num_workers"] == 0 and len(made["corpora"]) == 1
    ds3, _ = _dataset(module, ids=("a.wav", "b.wav"))
    torch.utils.data.DataLoader(ds3)
    assert len(made["corpora"]) == 2 and len(svc.corpora) == 2


@pytest.mark.parametrize("case", ["other dataset", "augmentation", "online_aug", "sampler", "batch_sampler", "worker_init_fn",
                                  "collate_fn", "batch_size None", "in_order"])
def test_serve_items_falls_back_to_the_real_loader(served, case, caplog):
    module, svc, made, FakeLoader = served
    ds, _ = _dataset(module, **({"augmentation_methods": ["RawBoost12", "background_noise"]} if case == "augmentation" else
                                {"online_aug": False} if case == "online_aug" else {}))
    kw = {"sampler": {"sampler": torch.utils.data.SequentialSampler(range(3))},
          "batch_sampler": {"batch_sampler": [[0, 1], [2]]},
          "worker_init_fn": {"worker_init_fn": print},
          "collate_fn": {"collate_fn": list},
          "batch_size None": {"batch_size": None},
          "in_order": {"in_order": False}}.get(case, {})
    if case == "other dataset":
        ds = torch.utils.data.TensorDataset(torch.arange(3))
    with caplog.at_level(logging.WARNING, logger=loader.__name__):
        dl = torch.utils.data.DataLoader(ds, **kw)
    assert type(dl) is svc._real_loader and not made["loaders"] and not made["corpora"]
    lines = [r for r in caplog.records if r.name == loader.__name__]
    assert len(lines) == 1 and lines[0].getMessage().startswith("serve_items: real DataLoader")
    assert len(list(dl)) >= 1


def test_serve_items_checks_its_arguments():
    from scl_deepfake_audio_detection_b200 import dropin
    module = types.SimpleNamespace(Dataset_for=StandInDataset)
    with pytest.raises(ValueError):
        dropin.serve_items(module, None, dtype="int8")
    with pytest.raises(ValueError):
        dropin.serve_items(module, None, location="disk")
    assert module.Dataset_for.__init__ is StandInDataset.__init__

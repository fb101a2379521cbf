"""The reference's DataLoader epochs built on the device, batch for batch, with no worker processes building items.

The reference trains with ``DataLoader(train_set, batch_size=1, shuffle=True, num_workers=8)`` after
``torch.manual_seed(args.seed)`` (main.py:308, 379): torch decides which indices each worker gets and seeds each worker's
numpy stream, and every ``Dataset_for.__getitem__`` draws on the stream of the worker that runs it.

* :func:`epoch_schedule` -- what the installed torch's ``DataLoader`` does for one epoch, on the host: the batches in yield
  order, the worker of each batch, each worker's index list and numpy start state. It consumes torch's RNG exactly as the
  loader does, through torch's own sampler classes (or the caller's ``sampler`` / ``batch_sampler``) and its worker seeding
  (``_generate_state``, ``WorkerInfo`` and the ``_worker_info`` global, private parts of ``torch.utils.data._utils.worker``,
  on purpose: tests/test_device_loader_host.py and tests/test_device_loader_samplers_host.py pin them against a real loader,
  so a torch release that changes the seeding fails the suite instead of silently changing the data). A ``worker_init_fn``
  runs in one short-lived child process per worker, after torch's worker seeding, and what it leaves in numpy's state is
  that worker's start state.
* :class:`DeviceLoader` -- the iterable ``main.py``'s loop consumes: each epoch's items built on the GPU by
  :meth:`multiview.StreamItemBatcher.items_streams`, one stream per worker, every draw from the stream that worker would have
  used; batches are ``[ids, data, label]`` as ``default_collate`` gives them, with ``data`` and ``label`` on the device.
* :func:`serve_items` -- runs an unmodified ``main.py`` on :class:`DeviceLoader` (``dropin.serve_items``).
"""
from __future__ import annotations

import functools
import inspect
import logging
import multiprocessing
import operator
import random
import traceback
import weakref
from dataclasses import dataclass
from typing import List, Optional

import numpy as np
import torch
import torch.multiprocessing
from torch.utils.data import BatchSampler, RandomSampler, SequentialSampler
from torch.utils.data._utils import worker as _worker
from torch.utils.data._utils.worker import WorkerInfo, _generate_state

from . import multiview as _mv
from .engine import Engine

log = logging.getLogger(__name__)


def draw_base_seed(generator: Optional[torch.Generator] = None) -> int:
    """The seed ``_BaseDataLoaderIter.__init__`` draws from the loader's generator (or torch's global one) at ``iter()``."""
    return int(torch.empty((), dtype=torch.int64).random_(generator=generator).item())


def batch_sampler(n: int, batch_size: int = 1, shuffle: bool = False, drop_last: bool = False,
                  generator: Optional[torch.Generator] = None) -> BatchSampler:
    """The loader's index sampler: torch's ``BatchSampler`` over ``RandomSampler`` / ``SequentialSampler`` as ``DataLoader``
    builds it. A ``RandomSampler`` without a generator draws its own seed from torch's global generator each time a pass over
    it starts (at the first index)."""
    return index_sampler(n, batch_size, shuffle, drop_last, generator)


def index_sampler(n: int, batch_size: int = 1, shuffle: bool = False, drop_last: bool = False,
                  generator: Optional[torch.Generator] = None, sampler=None, batch_sampler=None):
    """What ``DataLoader.__init__`` iterates for index batches, with its refusals: a given ``batch_sampler`` as it is (any
    iterable of index lists, a plain list included); else ``BatchSampler(sampler, batch_size, drop_last)`` over the given
    ``sampler``, or over ``RandomSampler`` / ``SequentialSampler`` of ``range(n)`` (see :func:`batch_sampler`)."""
    if sampler is not None and shuffle:
        raise ValueError("sampler option is mutually exclusive with shuffle")
    if batch_sampler is not None:
        if batch_size != 1 or shuffle or sampler is not None or drop_last:
            raise ValueError("batch_sampler option is mutually exclusive with batch_size, shuffle, sampler, and drop_last")
        return batch_sampler
    if sampler is None:
        sampler = RandomSampler(range(n), generator=generator) if shuffle else SequentialSampler(range(n))
    return BatchSampler(sampler, batch_size, drop_last)


def checked_batches(batches, n: int) -> List[List[int]]:
    """One pass of a batch sampler as lists of int, every index checked before any item is built: a non-integer index
    (``bool`` included) raises TypeError, one outside ``[0, n)`` IndexError -- a negative one too, although a dataset that
    indexes a Python list would take it -- and an empty batch ValueError. Repeated indices are kept."""
    out = []
    for j, b in enumerate(batches):
        row = []
        for i in b:
            if isinstance(i, (bool, np.bool_)):
                raise TypeError(f"batch {j}: index {i!r} is not an integer")
            try:
                k = operator.index(i)
            except TypeError:
                raise TypeError(f"batch {j}: index {i!r} is not an integer") from None
            if not 0 <= k < n:
                raise IndexError(f"batch {j}: index {k} lies outside [0, {n})")
            row.append(k)
        if not row:
            raise ValueError(f"batch {j} is empty")
        out.append(row)
    return out


def worker_context(num_workers: int, multiprocessing_context=None):
    """The multiprocessing context ``DataLoader`` starts its workers from, with the refusals of its
    ``multiprocessing_context`` setter: a start method's name or a context; None is ``torch.multiprocessing`` (the platform's
    default start method)."""
    if multiprocessing_context is None:
        return torch.multiprocessing
    if num_workers <= 0:
        raise ValueError("multiprocessing_context can only be used with multi-process loading (num_workers > 0), but got "
                         f"num_workers={num_workers}")
    if isinstance(multiprocessing_context, str):
        valid = torch.multiprocessing.get_all_start_methods()
        if multiprocessing_context not in valid:
            raise ValueError(f"multiprocessing_context option should specify a valid start method in {valid!r}, but got "
                             f"multiprocessing_context={multiprocessing_context!r}")
        multiprocessing_context = torch.multiprocessing.get_context(multiprocessing_context)
    if not isinstance(multiprocessing_context, multiprocessing.context.BaseContext):
        raise TypeError("multiprocessing_context option should be a valid context object or a string specifying the start "
                        f"method, but got multiprocessing_context={multiprocessing_context}")
    return multiprocessing_context


def _run_worker_init(init_fn, base_seed: int, worker_id: int, num_workers: int, conn) -> None:
    """Child process: the prologue of torch's ``_worker_loop`` up to and including ``init_fn(worker_id)``, then numpy's state
    to the parent. No CUDA call: in a child forked from a process with a CUDA context, ``torch.manual_seed`` only queues its
    CUDA part, as in torch's own workers."""
    try:
        torch.set_num_threads(1)
        seed = base_seed + worker_id
        random.seed(seed)
        torch.manual_seed(seed)
        np.random.seed(_generate_state(base_seed, worker_id))
        # DeviceLoader holds no dataset object: get_worker_info().dataset is None
        _worker._worker_info = WorkerInfo(id=worker_id, num_workers=num_workers, seed=seed, dataset=None)
        init_fn(worker_id)
        conn.send(("ok", np.random.get_state()))
    except Exception:
        conn.send(("error", traceback.format_exc()))
    finally:
        conn.close()


def _init_states(base_seed: int, num_workers: int, init_fn, context) -> np.ndarray:
    """uint32 [num_workers, 625]: each worker's numpy state after ``init_fn`` has run in a child process started from
    ``context``, all children at once. An exception in a child raises RuntimeError here naming the worker, with the child's
    traceback; every child is joined whatever happens."""
    procs, conns = [], []
    ok = False
    try:
        for w in range(num_workers):
            recv, send = context.Pipe(duplex=False)
            conns.append(recv)
            try:
                p = context.Process(target=_run_worker_init, args=(init_fn, base_seed, w, num_workers, send), daemon=True)
                p.start()
            finally:
                send.close()  # the child holds its own end: a child that dies before it answers shows up as EOFError
            procs.append(p)
        states = np.zeros((num_workers, 625), dtype=np.uint32)
        for w, (p, recv) in enumerate(zip(procs, conns)):
            try:
                kind, value = recv.recv()
            except EOFError:
                p.join()
                raise RuntimeError(f"DataLoader worker process {w} exited with code {p.exitcode} before its worker_init_fn "
                                   "returned") from None
            if kind != "ok":
                raise RuntimeError(f"worker_init_fn raised in DataLoader worker process {w}:\n{value}")
            states[w] = _mv._state_words(value)
        ok = True
        return states
    finally:
        for p in procs:
            if not ok and p.is_alive():
                p.terminate()
            p.join()
        for c in conns:
            c.close()


def worker_start_states(base_seed: int, num_workers: int) -> np.ndarray:
    """uint32 [num_workers, 625]: the numpy state (key[624], pos) each worker holds before its first item --
    ``np.random.seed(_generate_state(base_seed, worker_id))`` as torch's worker loop seeds it."""
    states = np.zeros((num_workers, 625), dtype=np.uint32)
    for w in range(num_workers):
        states[w] = _mv._state_words(np.random.RandomState(_generate_state(base_seed, w)).get_state())
    return states


@dataclass
class EpochSchedule:
    """One epoch of a ``DataLoader``.

    ``batches``: lists of dataset indices in yield order. ``batch_worker``: the worker that builds each batch (0, the main
    process, without workers). ``worker_indices``: each worker's items in the order it builds them (one list without workers).
    ``worker_states``: uint32 [W, 625] numpy start states, or None where the streams are not seeded at this epoch: without
    workers (the items draw on the main process's global numpy stream) and in the later epochs of persistent workers (each
    worker's stream carries on from where the previous epoch left it). ``base_seed``: the seed drawn at ``iter()``, None where
    none is drawn."""
    batches: List[List[int]]
    batch_worker: List[int]
    worker_indices: List[List[int]]
    worker_states: Optional[np.ndarray]
    base_seed: Optional[int]


def check_loader_args(n: int, batch_size: int, num_workers: int, persistent_workers: bool) -> None:
    """The refusals of ``DataLoader.__init__`` for the arguments :func:`epoch_schedule` takes."""
    if int(n) < 0:
        raise ValueError(f"the dataset length must be non-negative, not {n}")
    if int(num_workers) < 0:
        raise ValueError("num_workers option should be non-negative; use num_workers=0 to disable multiprocessing.")
    if persistent_workers and num_workers == 0:
        raise ValueError("persistent_workers option needs num_workers > 0")
    if isinstance(batch_size, bool) or not isinstance(batch_size, int) or batch_size <= 0:
        raise ValueError(f"batch_size should be a positive integer value, but got batch_size={batch_size}")


def split_batches(batches: List[List[int]], num_workers: int):
    """``(batch_worker, worker_indices)``: batch j goes to worker j mod W, as the loader's round-robin dispatch sends it (every
    epoch restarts at worker 0)."""
    W = max(1, num_workers)
    batch_worker = [j % W for j in range(len(batches))]
    worker_indices = [[i for j in range(w, len(batches), W) for i in batches[j]] for w in range(W)]
    return batch_worker, worker_indices


def epoch_schedule(n: int, batch_size: int = 1, shuffle: bool = False, num_workers: int = 0, drop_last: bool = False,
                   generator: Optional[torch.Generator] = None, persistent_workers: bool = False,
                   first_iter: bool = True, *, sampler=None, batch_sampler=None, worker_init_fn=None,
                   multiprocessing_context=None) -> EpochSchedule:
    """What ``iter(DataLoader(dataset_of_length_n, batch_size, shuffle, sampler, batch_sampler, num_workers, drop_last=...,
    worker_init_fn=..., multiprocessing_context=..., generator=..., persistent_workers=...))`` followed by a full pass does
    with the installed torch, for a map-style dataset with the default collate function. The index batches are those of
    :func:`index_sampler`, every index checked by :func:`checked_batches`.

    torch's RNG is consumed as the loader consumes it: the base seed from ``generator`` (or the global generator) -- only at
    the first ``iter()`` of persistent workers (``first_iter``) -- then the batch sampler's pass starts, and torch's own
    samplers make their draws there (a ``RandomSampler`` without a generator its own seed from the global generator;
    ``WeightedRandomSampler``, ``SubsetRandomSampler`` and ``DistributedSampler`` likewise at their first index). The loader
    with workers makes both inside ``iter()``; without workers the pass starts at the first ``next()`` (:class:`DeviceLoader`
    keeps that timing; this function makes both at once).

    Where torch seeds its workers (every epoch, or only the first one of persistent workers) and a ``worker_init_fn`` is
    given, it runs for each worker in a child process started from ``multiprocessing_context`` (a start method's name or a
    context; None is the platform's default), after torch's worker seeding, with ``get_worker_info()`` set (its ``dataset``
    None), and the numpy state it leaves is the worker's start state. An exception there raises RuntimeError naming the
    worker. Without workers it is not called, as torch does not call it then."""
    check_loader_args(n, batch_size, num_workers, persistent_workers)
    index_batches = index_sampler(n, batch_size, shuffle, drop_last, generator, sampler, batch_sampler)
    context = worker_context(num_workers, multiprocessing_context)
    seeded = num_workers == 0 or first_iter or not persistent_workers
    return _schedule(index_batches, n, num_workers, generator, seeded, worker_init_fn, context)


def _schedule(index_batches, n: int, num_workers: int, generator, seeded: bool, worker_init_fn, context) -> EpochSchedule:
    it = iter(index_batches)  # _BaseDataLoaderIter takes the sampler's iterator first, then draws the base seed
    seed = draw_base_seed(generator) if seeded else None
    batches = checked_batches(it, n)
    batch_worker, worker_indices = split_batches(batches, num_workers)
    states = None
    if num_workers and seed is not None:
        states = (_init_states(seed, num_workers, worker_init_fn, context) if worker_init_fn is not None else
                  worker_start_states(seed, num_workers))
    return EpochSchedule(batches, batch_worker, worker_indices, states, seed)


@dataclass
class _Chunk:
    """One production call: its outputs, the row of each of its batches, and the event its consumers wait on."""
    first: int            # index of its first batch in the epoch
    rows: List[int]       # row of each batch's first item
    ids: list
    data: torch.Tensor
    labels: torch.Tensor
    done: torch.cuda.Event
    out_len_host: Optional[torch.Tensor] = None
    end_host: Optional[torch.Tensor] = None


class DeviceLoader:
    """``DataLoader(Dataset_for(...), batch_size, shuffle, sampler, batch_sampler, num_workers, drop_last=...,
    worker_init_fn=..., multiprocessing_context=..., generator=..., persistent_workers=...)`` for
    ``augmentation_methods == ['RawBoost12']`` with ``online_aug``, every item built on the GPU.

    ``corpus``: a :class:`multiview.DeviceCorpus` or :class:`multiview.PackedCorpus` of the dataset's ``list_IDs`` and
    vocoders; ``args``, ``num_additional_real``, ``trim_length``, ``repeat_pad`` and ``wav_samp_rate`` as the ``Dataset_for``
    was given them. ``len()`` is the loader's length and every ``next()`` yields ``[ids, data, label]``: ``ids`` a list of
    str, ``data`` a device tensor [b, trim, V] (``layout`` LAYOUT_ITEM, what ``default_collate`` stacks) or [b, V, trim]
    (LAYOUT_MODEL), ``label`` a device tensor [b, V]. The batches, their order, and every draw of every item are those of the
    real loader after the same ``torch.manual_seed``: each worker's items come from the numpy stream torch would have seeded
    for that worker; without workers they come from numpy's global stream, which afterwards stands where the real loader
    leaves it (read when the epoch's first batch is built, written back when its last batch is yielded: one synchronisation).

    ``sampler`` / ``batch_sampler`` are taken as ``DataLoader`` takes them (:func:`index_sampler`), and every epoch iterates
    the same object, so ``DistributedSampler.set_epoch(e)`` before an epoch works as with torch. Each epoch's indices are
    checked on the host before anything is enqueued (:func:`checked_batches`): a negative index raises IndexError although a
    dataset indexing a Python list would take it. ``worker_init_fn`` runs where torch's workers run it, in a short-lived child
    process per worker started from ``multiprocessing_context``, and the numpy state it leaves is that worker's start state
    (:func:`epoch_schedule`); the child makes no CUDA call. One data-parallel rank per GPU builds its shard on its own device:
    the loader runs on ``corpus.eng.device``, whatever the current device is when it is iterated.

    Items are built ``chunk_batches`` loader batches at a time, one ``items_streams`` call per chunk with one stream per
    worker, on a side stream of the loader's own; a chunk's end states stay on the device and seed the next chunk's call (for
    persistent workers, the next epoch's). The next chunk is built while this one is consumed: every ``next()`` makes the
    caller's current stream wait for its chunk and records the yielded tensors on that stream, so a yielded batch stays
    valid, and is never overwritten, for as long as the caller holds it. With ``repeat_pad=False`` an item shorter than the
    crop is as long as its anchor, so each chunk's lengths are read back (with the end state above, the only read-backs); a
    batch of items of different lengths then raises as ``default_collate`` does.

    A yielded batch is a view of its chunk's output, so a batch kept beyond its epoch keeps the whole chunk's memory alive:
    at ASVspoof 2019 LA train's shape (trim 64 000, V = 10) and the default 256 batches of one item, about 655 MB. Keep a
    ``.clone()`` of what outlives the step instead.

    Differences from the real loader:
    * Without workers, the items of an epoch draw on numpy's global state as it stood at the epoch's first ``next()``, and
      the state after the epoch's last item is written back when its last batch is yielded. Draws the training loop itself
      makes on numpy's global stream during the epoch are therefore not seen by later items (the real single-process loader
      would interleave them) and are discarded at the epoch's end. With workers, as in the reference, the main process's
      stream is not involved.
    * An epoch left before its end leaves numpy's global stream where it was (no workers), and persistent workers' streams
      carry on from where production stopped (torch's workers would also have built the batches they had been sent).
    * Items are always built in the main process, whatever ``num_workers`` says.
    * The real loader pulls ``prefetch_factor * num_workers`` batches from the batch sampler ahead of the batches it yields;
      this loader pulls the whole epoch at ``iter()`` (at the first ``next()`` without workers). The samplers of torch make
      all their draws when their pass starts, so this changes nothing for them; a sampler that draws on torch's *global*
      generator lazily, index by index, sees those draws at another point relative to the training loop's own draws on it.
    * ``get_worker_info().dataset`` is None inside ``worker_init_fn``: the loader holds no dataset object."""

    def __init__(self, corpus, args, num_additional_real=2, trim_length=64000, repeat_pad=True, wav_samp_rate=16000,
                 batch_size=1, shuffle=False, num_workers=0, drop_last=False, generator=None, persistent_workers=False,
                 layout=_mv.LAYOUT_ITEM, chunk_batches=256, *, sampler=None, batch_sampler=None, worker_init_fn=None,
                 multiprocessing_context=None):
        n = int(corpus.N)
        check_loader_args(n, batch_size, num_workers, persistent_workers)
        index_batches = index_sampler(n, batch_size, shuffle, drop_last, generator, sampler, batch_sampler)
        self._context = worker_context(num_workers, multiprocessing_context)
        if int(chunk_batches) < 1:
            raise ValueError(f"chunk_batches must be at least 1, not {chunk_batches}")
        if layout not in (_mv.LAYOUT_ITEM, _mv.LAYOUT_MODEL):
            raise ValueError(f"layout must be LAYOUT_ITEM or LAYOUT_MODEL, not {layout!r}")
        self.corpus, self.n = corpus, n
        self.batch_size, self.shuffle, self.num_workers, self.drop_last = int(batch_size), bool(shuffle), int(num_workers), bool(drop_last)
        self.generator, self.persistent_workers = generator, bool(persistent_workers)
        self.layout, self.chunk_batches, self.repeat_pad = layout, int(chunk_batches), bool(repeat_pad)
        self.sampler, self.batch_sampler, self.worker_init_fn = sampler, index_batches, worker_init_fn
        self.device = corpus.eng.device
        # its own engine: its own workspace, so the side stream shares no scratch memory with other users of the corpus's engine
        self._eng = Engine(self.device)
        self._bat = _mv.StreamItemBatcher(args, corpus, num_additional_real, trim_length, repeat_pad, wav_samp_rate, engine=self._eng)
        self._side = torch.cuda.Stream(self.device)
        # where each stream stands after the last chunk enqueued: numpy state tuples at an epoch's start, then the device
        # [W, 625] end states of the last call
        self._states = None
        self._iterated = False

    def __len__(self) -> int:
        return len(self.batch_sampler)

    def __iter__(self):
        if self.num_workers == 0:
            it = iter(self.batch_sampler)
            draw_base_seed(self.generator)  # the sampler's own draws wait for the first next()
            return self._epoch(None, it)
        s = _schedule(self.batch_sampler, self.n, self.num_workers, self.generator,
                      not (self.persistent_workers and self._iterated), self.worker_init_fn, self._context)
        self._iterated = True
        if s.worker_states is not None:
            self._states = [_mv.numpy_state(row) for row in s.worker_states]
        return self._epoch(s.batches)

    def _epoch(self, batches, sampler_iter=None):
        gauss = None
        if batches is None:  # no workers: the first next() starts the sampler's pass, then the items draw on numpy's stream
            batches = checked_batches(sampler_iter, self.n)
            state = np.random.get_state()
            gauss = tuple(state[3:5])  # the items never use numpy's Gaussian cache: it carries over unchanged
            self._states = [state]
        C = self.chunk_batches
        nchunks = -(-len(batches) // C)
        chunk = self._produce(batches, 0, gauss is not None and nchunks == 1) if nchunks else None
        for k in range(nchunks):
            nxt = self._produce(batches, (k + 1) * C, gauss is not None and k + 2 == nchunks) if k + 1 < nchunks else None
            lens = None
            if chunk.out_len_host is not None or chunk.end_host is not None:
                chunk.done.synchronize()
                lens = chunk.out_len_host.numpy() if chunk.out_len_host is not None else None
            for j in range(chunk.first, min(chunk.first + C, len(batches))):
                if gauss is not None and j + 1 == len(batches):
                    np.random.set_state(_mv.numpy_state(chunk.end_host[0])[:3] + gauss)
                yield self._batch(chunk, j, len(batches[j]), lens)
            chunk = nxt

    def _produce(self, batches, first, read_end):
        """Enqueue the chunk of batches [first, first + chunk_batches) on the side stream."""
        part = batches[first:first + self.chunk_batches]
        W = max(1, self.num_workers)
        lists = [[] for _ in range(W)]
        starts = []
        for j, b in enumerate(part, start=first):
            w = j % W
            starts.append((w, len(lists[w])))
            lists[w] += b
        base = np.concatenate([[0], np.cumsum([len(ix) for ix in lists])])
        rows = [int(base[w]) + r for w, r in starts]
        with torch.cuda.stream(self._side):
            ids, data, labels, out_len, end = self._bat.items_streams(lists, self._states, self.layout)
            self._states = end
            out_len_host = end_host = None
            if not self.repeat_pad:
                out_len_host = torch.empty(out_len.shape, dtype=out_len.dtype, pin_memory=True)
                out_len_host.copy_(out_len, non_blocking=True)
            if read_end:
                end_host = torch.empty(end.shape, dtype=end.dtype, pin_memory=True)
                end_host.copy_(end, non_blocking=True)
            done = torch.cuda.Event()
            done.record(self._side)
        return _Chunk(first, rows, ids, data, labels, done, out_len_host, end_host)

    def _batch(self, chunk: _Chunk, j: int, b: int, lens):
        r = chunk.rows[j - chunk.first]
        data, labels = chunk.data[r:r + b], chunk.labels[r:r + b]
        if lens is not None:
            got = {int(x) for x in lens[r:r + b]}
            if len(got) != 1:
                raise RuntimeError(f"stack expects each tensor to be equal size, but the items of batch {j} have "
                                   f"{sorted(got)} samples per view")
            L = got.pop()
            data = data[:, :L] if self.layout == _mv.LAYOUT_ITEM else data[:, :, :L]
        cur = torch.cuda.current_stream(self.device)
        cur.wait_event(chunk.done)
        data.record_stream(cur)
        labels.record_stream(cur)
        return [chunk.ids[r:r + b], data, labels]


# -- the unmodified main.py ---------------------------------------------------------------------------------------------------
_DL_SIGNATURE = inspect.signature(torch.utils.data.DataLoader.__init__)


class ItemService:
    """Handle of :func:`serve_items`: ``close()`` (or leaving a ``with`` block) puts ``Dataset_for.__init__`` and
    ``torch.utils.data.DataLoader`` back; ``corpora`` holds the corpora built so far."""

    def __init__(self, loader_module, load_audio, dtype, location):
        self.loader_module, self.load_audio, self.dtype, self.location = loader_module, load_audio, dtype, location
        self.corpora = {}
        self._recorded = weakref.WeakKeyDictionary()
        self._real_init = loader_module.Dataset_for.__init__
        self._real_loader = torch.utils.data.DataLoader
        init_sig = inspect.signature(self._real_init)
        real_init, recorded = self._real_init, self._recorded

        @functools.wraps(real_init)
        def init(ds, *a, **kw):
            real_init(ds, *a, **kw)
            bound = init_sig.bind(ds, *a, **kw)
            bound.apply_defaults()
            recorded[ds] = dict(bound.arguments)

        def factory(dataset, *a, **kw):
            return self.make_loader(dataset, *a, **kw)

        # a function, not a class: ``isinstance(x, torch.utils.data.DataLoader)`` raises TypeError while the service runs
        factory.__name__ = factory.__qualname__ = "DataLoader"
        factory.__doc__ = ("torch.utils.data.DataLoader as serve_items replaces it: a DeviceLoader where the call can be one, "
                           "else the real DataLoader (documented at __wrapped__).")
        factory.__wrapped__ = self._real_loader

        loader_module.Dataset_for.__init__ = init
        torch.utils.data.DataLoader = factory

    def close(self) -> None:
        self.loader_module.Dataset_for.__init__ = self._real_init
        torch.utils.data.DataLoader = self._real_loader

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def refusal(self, dataset, call: dict) -> Optional[str]:
        """Why ``DataLoader(dataset, **call)`` cannot be a :class:`DeviceLoader` (None when it can)."""
        rec = self._recorded.get(dataset) if _weakrefable(dataset) else None
        if rec is None:
            return f"the dataset is a {type(dataset).__name__}, not a Dataset_for built after serve_items"
        if list(rec.get("augmentation_methods") or []) != ["RawBoost12"]:
            return f"augmentation_methods is {rec.get('augmentation_methods')!r}, not ['RawBoost12']"
        if not getattr(rec.get("args"), "online_aug", False):
            return "args.online_aug is not set"
        for name in ("sampler", "batch_sampler", "worker_init_fn", "collate_fn"):
            if call[name] is not None:
                return f"a {name} is given"
        if call["batch_size"] is None:
            return "batch_size is None"
        if not call["in_order"]:
            return "in_order is False"
        return None

    def make_loader(self, dataset, *a, **kw):
        """What the replaced ``torch.utils.data.DataLoader`` returns: a :class:`DeviceLoader` where the call can be one, else
        the real ``DataLoader`` (after one logged line saying why)."""
        bound = _DL_SIGNATURE.bind(None, dataset, *a, **kw)
        bound.apply_defaults()
        call = dict(bound.arguments)
        why = self.refusal(dataset, call)
        if why is not None:
            log.warning("serve_items: real DataLoader, %s", why)
            return self._real_loader(dataset, *a, **kw)
        rec = self._recorded[dataset]
        key = (tuple(rec["list_IDs"]), rec["base_dir"], tuple(rec.get("vocoders") or ()))
        corpus = self.corpora.get(key)
        if corpus is None:
            corpus = self.corpora[key] = _mv.PackedCorpus(key[0], key[1], self.load_audio, key[2], dtype=self.dtype,
                                                          location=self.location)
        return DeviceLoader(corpus, rec["args"], num_additional_real=rec["num_additional_real"], trim_length=rec["trim_length"],
                            repeat_pad=rec["repeat_pad"], batch_size=call["batch_size"], shuffle=bool(call["shuffle"]),
                            num_workers=call["num_workers"], drop_last=call["drop_last"], generator=call["generator"],
                            persistent_workers=call["persistent_workers"])


def _weakrefable(obj) -> bool:
    try:
        weakref.ref(obj)
        return True
    except TypeError:
        return False


def serve_items(loader_module, load_audio, dtype: str = "pcm16", location: str = "device") -> ItemService:
    """Let an unmodified ``main.py`` train on :class:`DeviceLoader`. ``loader_module`` is the imported loader
    (``datautils.asvspoof_2019_augall_3``): its ``Dataset_for.__init__`` is wrapped to record the arguments of every dataset
    built from now on, and ``torch.utils.data.DataLoader`` becomes a factory. It returns a :class:`DeviceLoader` over a
    :class:`multiview.PackedCorpus` (``load_audio``, ``dtype``, ``location`` as there; built once per distinct list of ids,
    base directory and vocoders) when the dataset is such a ``Dataset_for`` with ``augmentation_methods == ['RawBoost12']``
    and ``args.online_aug`` set, and no ``sampler``, ``batch_sampler``, ``worker_init_fn`` or ``collate_fn`` is given;
    ``pin_memory``, ``prefetch_factor``, ``timeout`` and ``multiprocessing_context`` are accepted and ignored. Otherwise it
    returns the real ``DataLoader`` and logs one line saying why. Returns the :class:`ItemService` handle."""
    if dtype not in _mv._PER_CHUNK:
        raise ValueError(f"dtype must be 'pcm16' or 'float32', not {dtype!r}")
    if location not in ("device", "host"):
        raise ValueError(f"location must be 'device' or 'host', not {location!r}")
    return ItemService(loader_module, load_audio, dtype, location)

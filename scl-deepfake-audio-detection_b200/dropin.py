"""Install the B200 RawBoost path under the names the reference's loaders bind to (SURVEY.md 8b).

The loaders do ``from datautils.RawBoost import ISD_additive_noise, LnL_convolutive_noise, SSI_additive_noise,
normWav`` at import (``/root/reference/datautils/asvspoof_2019_augall_3.py:10``) and define their own
``process_Rawboost_feature`` / ``RawBoost12`` that look those four names up in module globals at call time.
Two ways in, both leave the loader sources untouched:

* :func:`install` before the loader is imported: registers this package's ``RawBoost`` module as
  ``sys.modules['datautils.RawBoost']``.
* :func:`patch_loader` after import: rebinds the operator names (and the dispatcher, which then issues one fused
  device call per utterance instead of one per operator) inside an already imported loader module.

CUDA cannot be used in forked DataLoader workers once the parent initialised it (main.py:335 precedes main.py:379).
:func:`serve_workers`, called once in the parent before the loader starts its workers, lets the unmodified loaders run there:
each worker draws on its own numpy stream as before and the parent applies the calls of all workers on the GPU, in batches.
:func:`serve_items` goes further: it replaces the DataLoader the reference builds over ``Dataset_for`` with
:class:`loader.DeviceLoader`, which builds the same epochs on the GPU with no worker processes at all.
The alternatives remain: ``num_workers=0``, ``multiprocessing_context='spawn'``, or the batched path (``plans.draw_batch`` in
the workers, ``engine.Engine.process`` on the collated batch).
"""
from __future__ import annotations

import sys
import types

OPERATORS = ("randRange", "normWav", "genNotchCoeffs", "filterFIR", "LnL_convolutive_noise", "ISD_additive_noise",
             "SSI_additive_noise")
DISPATCH = ("process_Rawboost_feature", "RawBoost12")


def install(module_name: str = "datautils.RawBoost") -> types.ModuleType:
    """Make ``import datautils.RawBoost`` (or ``module_name``) resolve to the B200 implementation."""
    from . import RawBoost as impl
    sys.modules[module_name] = impl
    parent, _, leaf = module_name.rpartition(".")
    if parent and parent in sys.modules:
        setattr(sys.modules[parent], leaf, impl)
    return impl


def patch_loader(loader: types.ModuleType, dispatcher: bool = True) -> types.ModuleType:
    """Rebind the RawBoost names inside an imported loader module (e.g. ``datautils.asvspoof_2019_augall_3``)."""
    from . import RawBoost as impl
    for name in OPERATORS:
        if hasattr(loader, name):
            setattr(loader, name, getattr(impl, name))
    if dispatcher:
        for name in DISPATCH:
            if hasattr(loader, name):
                setattr(loader, name, getattr(impl, name))
    return loader


def serve_workers(device=None, max_batch: int = 64, max_len: int = 211000):
    """Serve the RawBoost calls of this process's DataLoader workers on the GPU; returns the :class:`broker.Broker`.

    Call it in the process that owns the GPU, after :func:`install` / :func:`patch_loader` and before the DataLoader starts its
    workers (forked, spawned or forkserver). Every worker then sends its ``normWav``, ``filterFIR`` and RawBoost applications
    here; the draws stay in the worker, so every numpy stream advances exactly as with the reference. One daemon thread applies
    whatever requests are pending, up to ``max_batch`` utterances per batch, with its own engine and context; the process's own
    drop-in calls are unaffected. ``max_len``: the longest utterance the workers send, for which the device buffers are sized
    once, here (a longer one still works, at the cost of one device-wide synchronise when the buffers grow).
    The handle has ``close()``, ``stats()`` (requests, batches, utterances, errors) and works as a context manager."""
    from .broker import serve
    return serve(device, max_batch, max_len)


def serve_items(loader_module, load_audio, dtype: str = "pcm16", location: str = "device"):
    """Let an unmodified ``main.py`` train on items built on the GPU, with no worker processes; returns the
    :class:`loader.ItemService` handle (``close()``, context manager).

    Call it after :func:`install` and before ``main.py`` runs, with the imported loader module (``datautils.asvspoof_2019_augall_3``)
    and the audio reader. ``Dataset_for.__init__`` then records its arguments, and ``torch.utils.data.DataLoader`` returns a
    :class:`loader.DeviceLoader` over a ``multiview.PackedCorpus`` (``dtype``, ``location``) for a ``Dataset_for`` with
    ``augmentation_methods == ['RawBoost12']`` and ``args.online_aug`` set, and no ``sampler``, ``batch_sampler``,
    ``worker_init_fn`` or ``collate_fn``: the same batches in the same order, every draw from the numpy stream the worker that
    built it would have used. Any other call gets the real ``DataLoader`` and one logged line saying why."""
    from .loader import serve_items as serve
    return serve(loader_module, load_audio, dtype, location)

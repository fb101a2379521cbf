"""The step right after RawBoost for the views of a training item, kept on the device (SURVEY.md 8f-1 / 8f-2).

* :func:`batch_pad_for_multiview` -- drop-in for ``core_scripts/data_io/wav_augmentation.py:209-282`` (same signature,
  same ``np.random.rand()`` draw in the same place, same result): every view is cut / zero-extended / tiled to the length
  of view 0 and one shared crop is taken.
* :func:`crop_plan` -- the host part alone: ``(start, out_len)`` of that crop; the global numpy stream is left exactly
  where the reference leaves it.
* :func:`assemble` -- the device part alone, batched over items: views already on the device (e.g. straight out of
  :meth:`engine.Engine.process`) go to ``[G, length, V]`` (the Dataset's ``batch_data``, asvspoof_2019_augall_3.py:138-142)
  or ``[G, V, length]`` (what the model consumes after main.py:57-60) without visiting the host.
* :func:`item_views` -- one call for whole items in the loader's order (RawBoost12 on the vocoded copies, then on the
  anchor, then the crop: asvspoof_2019_augall_3.py:109-138).
* :class:`ItemBatcher` -- whole ``Dataset_for`` items, every draw on the host from the global numpy stream.
* :class:`DeviceCorpus` + :class:`SeededItemBatcher` -- whole items seeded one by one (``np.random.seed(s)`` before each
  ``__getitem__``), every draw replayed on the device from a corpus that lives there.
* :class:`StreamItemBatcher` -- the same for items that share numpy's running stream, one after another, as
  :class:`ItemBatcher` draws them.
* :class:`PackedCorpus` -- the same corpus for both batchers with rows packed at their own lengths, as 16-bit PCM or float32,
  in device memory or read in place from page-locked host memory.

Integer work (crop start, index map) is bit-exact; the samples are copies of the views' float32 values.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib, plans as _plans
from .engine import Engine, default_engine

LAYOUT_ITEM = 0    # [G, length, V]  (np.concatenate(views, axis=1) of the reference)
LAYOUT_MODEL = 1   # [G, V, length]  (batch_x after the transpose in main.py:57-60)


def crop_plan(first_len: int, length: int, random_trim_nosil: bool = False, repeat_pad: bool = False) -> Tuple[int, int]:
    """``(start, out_len)`` of the shared crop. ``np.random.rand()`` is consumed iff the reference consumes it: only when
    view 0 has at least ``length`` samples and ``random_trim_nosil`` is set (wav_augmentation.py:256, 273)."""
    first_len, length = int(first_len), int(length)
    if first_len < length:
        return 0, (length if repeat_pad else first_len)
    start = int(np.random.rand() * (first_len - length)) if random_trim_nosil else 0
    return start, length


def assemble(eng: Engine, views: torch.Tensor, lengths: torch.Tensor, V: int, starts, length: int, repeat_pad: bool,
             layout: int = LAYOUT_MODEL, out: Optional[torch.Tensor] = None):
    """views: [G*V, ld] float32 on the device (view v of item g in row g*V+v), lengths: int32 [G*V], starts: G crop starts.
    Returns ``(out, out_len)``: out is [G, length, V] or [G, V, length]; out_len int32 [G] = samples written per view.
    Asynchronous on torch's current stream."""
    if views.dtype != torch.float32 or views.dim() != 2 or not views.is_contiguous() or views.device != eng.device:
        raise ValueError("views must be a contiguous [G*V, ld] float32 tensor on the engine's device")
    rows, ld = views.shape
    if V <= 0 or rows % V:
        raise ValueError("rows of `views` must be a multiple of V")
    G = rows // V
    if lengths.dtype != torch.int32 or lengths.numel() != rows or lengths.device != eng.device:
        raise ValueError("lengths must be int32 [G*V] on the engine's device")
    if not torch.is_tensor(starts):
        starts = torch.tensor(np.asarray(starts, dtype=np.int32), device=eng.device)
    if starts.dtype != torch.int32 or starts.numel() != G:
        raise ValueError("one int32 crop start per item")
    shape = (G, length, V) if layout == LAYOUT_ITEM else (G, V, length)
    if out is None:
        out = torch.zeros(shape, dtype=torch.float32, device=eng.device)
    out_len = torch.empty(G, dtype=torch.int32, device=eng.device)
    stream = torch.cuda.current_stream(eng.device).cuda_stream
    with torch.cuda.device(eng.device):
        rc = eng.lib.rb_multiview_assemble(C.c_void_p(views.data_ptr()), C.c_void_p(lengths.data_ptr()), G, V, ld,
                                           C.c_void_p(starts.data_ptr()), int(length), int(bool(repeat_pad)), int(layout),
                                           C.c_void_p(out.data_ptr()), C.c_void_p(out_len.data_ptr()), C.c_void_p(stream))
    _lib.check(rc, "rb_multiview_assemble")
    return out, out_len


def assemble_ex(eng: Engine, a: torch.Tensor, b: Optional[torch.Tensor], view_row: torch.Tensor, lengths: torch.Tensor, V: int,
                starts, length: int, repeat_pad: bool, layout: int = LAYOUT_MODEL, out: Optional[torch.Tensor] = None,
                view_label: Optional[torch.Tensor] = None):
    """:func:`assemble` with the views read where they already are (``rb_multiview_assemble_ex``): view v of item g is row
    ``r = view_row[g*V+v]`` of ``a`` (r >= 0) or row ``-1-r`` of ``b`` (r < 0) -- typically the original waveforms and their
    RawBoost results, two [R, ld] tensors sharing ``lengths`` [R]. No regrouping copy. With ``view_label`` (float32 [V]) the
    item's label vector (asvspoof_2019_augall_3.py:143-146) is produced too. Returns ``(out, out_len, labels or None)``."""
    for t in (a, b):
        if t is not None and (t.dtype != torch.float32 or t.dim() != 2 or not t.is_contiguous() or t.device != eng.device):
            raise ValueError("sources must be contiguous [R, ld] float32 tensors on the engine's device")
    if b is not None and b.shape != a.shape:
        raise ValueError("both sources must have the same shape")
    R, ld = a.shape
    if view_row.dtype != torch.int32 or view_row.device != eng.device or view_row.numel() % V:
        raise ValueError("view_row must be an int32 device tensor with G*V entries")
    G = view_row.numel() // V
    if lengths.dtype != torch.int32 or lengths.numel() != R or lengths.device != eng.device:
        raise ValueError("lengths must be int32 [R] on the engine's device")
    if not torch.is_tensor(starts):
        starts = torch.tensor(np.asarray(starts, dtype=np.int32), device=eng.device)
    if starts.dtype != torch.int32 or starts.numel() != G:
        raise ValueError("one int32 crop start per item")
    shape = (G, length, V) if layout == LAYOUT_ITEM else (G, V, length)
    if out is None:
        out = torch.zeros(shape, dtype=torch.float32, device=eng.device)
    out_len = torch.empty(G, dtype=torch.int32, device=eng.device)
    labels = None
    if view_label is not None:
        view_label = view_label.to(device=eng.device, dtype=torch.float32).contiguous()
        labels = torch.empty((G, V), dtype=torch.float32, device=eng.device)
    stream = torch.cuda.current_stream(eng.device).cuda_stream
    with torch.cuda.device(eng.device):
        rc = eng.lib.rb_multiview_assemble_ex(C.c_void_p(a.data_ptr()), C.c_void_p(b.data_ptr()) if b is not None else None,
                                              C.c_void_p(view_row.data_ptr()), C.c_void_p(lengths.data_ptr()), G, V, ld,
                                              C.c_void_p(starts.data_ptr()), int(length), int(bool(repeat_pad)), int(layout),
                                              C.c_void_p(out.data_ptr()), C.c_void_p(out_len.data_ptr()),
                                              C.c_void_p(view_label.data_ptr()) if view_label is not None else None,
                                              C.c_void_p(labels.data_ptr()) if labels is not None else None, C.c_void_p(stream))
    _lib.check(rc, "rb_multiview_assemble_ex")
    return out, out_len, labels


def batch_pad_for_multiview(input_data_batch_, wav_samp_rate, length, random_trim_nosil=False, repeat_pad=False):
    """Drop-in for the reference function: list of (len_v, 1) arrays in, list of (out_len, 1) float32 arrays out."""
    eng = default_engine()
    waves = [np.asarray(x, dtype=np.float32).reshape(-1) for x in input_data_batch_]
    start, out_len = crop_plan(waves[0].shape[0], length, random_trim_nosil, repeat_pad)
    if out_len == 0:
        return [np.zeros((0, 1), dtype=np.float32) for _ in waves]
    xd, ln = eng.pack_waveforms(waves)
    out, _ = assemble(eng, xd, ln, len(waves), [start], int(length), bool(repeat_pad), LAYOUT_MODEL)
    host = out[0].cpu().numpy()
    return [host[v, :out_len].reshape(out_len, 1) for v in range(len(waves))]


def item_view_rows(G: int, nvoc: int, extra_rows: Optional[np.ndarray] = None) -> np.ndarray:
    """Row table of :func:`assemble_ex` for G items whose waveforms sit in the loader's draw order -- per item ``nvoc`` vocoded
    copies, then the anchor (asvspoof_2019_augall_3.py:109-124) -- in one [G*(nvoc+1), ld] input tensor ``x`` with the RawBoost
    results in ``y``. View order of the Dataset (line 133): anchor, augmented anchor, [additional bona fide rows], vocoded,
    augmented vocoded. ``extra_rows``: int [G, n_add] rows of ``x`` holding each item's additional bona fide utterances."""
    per = nvoc + 1
    base = np.arange(G, dtype=np.int64)[:, None] * per
    voc = base + np.arange(nvoc)[None, :]
    anchor = base + nvoc
    cols = [anchor, -1 - anchor]
    if extra_rows is not None and np.size(extra_rows):
        cols.append(np.asarray(extra_rows, dtype=np.int64).reshape(G, -1))
    cols += [voc, -1 - voc]
    return np.concatenate(cols, axis=1).astype(np.int32)


def item_labels(nvoc: int, n_add: int = 0, n_aug: int = 1) -> np.ndarray:
    """Label vector of one item (asvspoof_2019_augall_3.py:143-146): 1 for the anchor and its positives, 0 for everything vocoded."""
    return np.array([1.0] * (n_aug + n_add + 1) + [0.0] * (2 * nvoc), dtype=np.float32)


def item_views(eng: Engine, items: Sequence[Tuple[np.ndarray, Sequence[np.ndarray]]], args, sr: int, trim_length: int,
               repeat_pad: bool = True, random_trim_nosil: bool = True, layout: int = LAYOUT_MODEL, with_labels: bool = False):
    """Views of whole items, RawBoost and assembly on the device, random draws in the loader's order.

    ``items``: ``(anchor, [vocoded copies])`` float32 waveforms. Per item, as Dataset_for.__getitem__ with
    ``augmentation_methods[0] == 'RawBoost12'`` does (asvspoof_2019_augall_3.py:109-138): RawBoost (algo 5) is drawn for
    each vocoded copy, then for the anchor, then the shared crop. View order: anchor, augmented anchor, vocoded copies,
    augmented vocoded copies. The assembly reads originals and augmented waveforms in place through a row table (no regrouping
    copy). Returns ``(out, out_len)`` as :func:`assemble` (plus the [G, V] label tensor with ``with_labels``)."""
    drawn, starts, all_waves = [], [], []
    nvoc = len(items[0][1])
    for anchor, vocoded in items:
        if len(vocoded) != nvoc:
            raise ValueError("every item needs the same number of vocoded copies")
        order = list(vocoded) + [anchor]
        drawn += [_plans.draw_for_algo(w.shape[0], sr, args, 5) for w in order]
        all_waves += order
        starts.append(crop_plan(anchor.shape[0], trim_length, random_trim_nosil, repeat_pad)[0])
    bp = _plans.pack(drawn)
    x, ln = eng.pack_waveforms(all_waves, ld=bp.ld)
    y = eng.process(5, x, ln, eng.upload_plan(bp))
    G, V = len(items), 2 * (nvoc + 1)
    rows = torch.from_numpy(item_view_rows(G, nvoc).reshape(-1)).to(eng.device)
    label = torch.from_numpy(item_labels(nvoc)) if with_labels else None
    out, out_len, labels = assemble_ex(eng, x, y, rows, ln, V, starts, trim_length, repeat_pad, layout, view_label=label)
    return (out, out_len, labels) if with_labels else (out, out_len)


class ItemBatcher:
    """Loader-level drop-in for ``Dataset_for.__getitem__`` (asvspoof_2019_augall_3.py:103-146) over a BATCH of indices.

    The reference builds one item per call inside a DataLoader worker: RawBoost on every vocoded copy and on the anchor, a
    ``np.random.choice`` of additional bona fide utterances, one shared crop, a column concat. This class does the same for a
    list of indices with ONE device pass: every random draw is made on the host in the reference's order on the process-global
    numpy stream (so the stream ends where the reference leaves it), all RawBoost calls of all items run as one batch, and
    the views are assembled on the device in place. ``augmentation_methods`` is RawBoost12 only -- the other methods of the
    reference (background noise, reverb wrappers) need external corpora and stay with the caller.

    ``load_audio(path) -> float32 waveform`` is the caller's reader (``librosa.load`` in the reference)."""

    def __init__(self, args, list_ids, base_dir, load_audio, vocoders=(), num_additional_real=2, trim_length=64000, wav_samp_rate=16000,
                 repeat_pad=True, engine: Optional[Engine] = None, planner: str = "numpy"):
        import os
        self.args, self.list_ids, self.load_audio = args, list(list_ids), load_audio
        self.bonafide_dir = os.path.join(base_dir, "bonafide")
        self.vocoded_dir = os.path.join(base_dir, "vocoded")
        self.vocoders, self.num_additional_real = list(vocoders), int(num_additional_real)
        self.trim_length, self.sr, self.repeat_pad = int(trim_length), int(wav_samp_rate), bool(repeat_pad)
        self.eng = engine
        self.planner = planner
        self._native = None

    def _draw(self, length):
        if self.planner == "native":
            if self._native is None:
                from .native_planner import NativePlanner
                self._native = NativePlanner(threads=1, pinned=False)
            return self._native.draw([length], self.sr, self.args, 5, use_global_stream=True, copy=True)
        return _plans.draw_for_algo(length, self.sr, self.args, 5)

    def items(self, indices: Sequence[int], layout: int = LAYOUT_ITEM):
        """``[(utt_id, data, label)]``-equivalent for ``indices``: returns ``(ids, data, labels, out_len)`` with ``data`` a device
        tensor [G, trim_length, V] (``layout`` LAYOUT_ITEM, what ``Tensor(batch_data)`` holds per item) or [G, V, trim_length]."""
        import os
        eng = self.eng or default_engine()
        nvoc, n_add = len(self.vocoders), self.num_additional_real
        plans, waves, extra_waves, starts = [], [], [], []
        for idx in indices:
            name = self.list_ids[idx]
            anchor = np.asarray(self.load_audio(os.path.join(self.bonafide_dir, name)), dtype=np.float32)
            for v in self.vocoders:  # vocoded copies first: that is the order in which the loader consumes the stream
                w = np.asarray(self.load_audio(os.path.join(self.vocoded_dir, v + "_" + name)), dtype=np.float32)
                waves.append(w)
                plans.append(self._draw(w.shape[0]))
            waves.append(anchor)
            plans.append(self._draw(anchor.shape[0]))
            others = list(range(len(self.list_ids)))
            others.remove(idx)
            picked = np.random.choice(others, n_add, replace=False)
            extra_waves += [np.asarray(self.load_audio(os.path.join(self.bonafide_dir, self.list_ids[i])), dtype=np.float32) for i in picked]
            starts.append(crop_plan(anchor.shape[0], self.trim_length, True, self.repeat_pad)[0])
        G, per = len(indices), nvoc + 1
        # rows: the RawBoost inputs of all items first, then every item's additional bona fide utterances (not augmented)
        ld = _plans.padded_ld(max([w.shape[0] for w in waves + extra_waves] + [1]))
        if plans and isinstance(plans[0], _plans.BatchPlan):
            bp = _plans.concat(plans, ld)
        else:
            bp = _plans.pack(plans, ld=ld)
        x, ln = eng.pack_waveforms(waves + extra_waves, ld=ld)
        y = torch.zeros_like(x)
        nb = G * per
        eng.process(5, x[:nb], ln[:nb], eng.upload_plan(bp), out=y[:nb])
        extra_rows = nb + np.arange(G * n_add).reshape(G, n_add) if n_add else None
        V = 2 + n_add + 2 * nvoc
        rows = torch.from_numpy(item_view_rows(G, nvoc, extra_rows).reshape(-1)).to(eng.device)
        label = torch.from_numpy(item_labels(nvoc, n_add))
        out, out_len, labels = assemble_ex(eng, x, y, rows, ln, V, starts, self.trim_length, self.repeat_pad, layout, view_label=label)
        return [self.list_ids[i] for i in indices], out, labels, out_len


class DeviceCorpus:
    """Every bona fide utterance of ``list_ids`` and its vocoded copies, loaded once into device memory in the layout the
    per-item device path reads: rows [R, ld] float32 with R = N * (1 + nvoc); row ``idx`` is bona fide utterance ``idx``
    (``<base_dir>/bonafide/<id>``), row ``N + idx*nvoc + v`` is vocoder v's copy (``<base_dir>/vocoded/<vocoder>_<id>``), as
    ``Dataset_for`` names them. ld is the longest waveform rounded up to 4 samples, so the corpus costs R * ld * 4 bytes of
    device memory (2.7 GB for the 2580 bona fide utterances of ASVspoof 2019 LA train with 3 vocoders at 64 600 samples).

    ``load_audio(path) -> float32 waveform`` is the caller's reader (``librosa.load`` in the reference). Every waveform needs at
    least one sample."""

    def __init__(self, list_ids, base_dir, load_audio, vocoders=(), engine: Optional[Engine] = None):
        import os
        self.list_ids, self.vocoders = list(list_ids), list(vocoders)
        self.eng = engine or default_engine()
        self.N, self.nvoc = len(self.list_ids), len(self.vocoders)
        if self.N < 1:
            raise ValueError("the corpus needs at least one utterance")
        paths = [os.path.join(base_dir, "bonafide", name) for name in self.list_ids]
        paths += [os.path.join(base_dir, "vocoded", v + "_" + name) for name in self.list_ids for v in self.vocoders]
        waves = [np.asarray(load_audio(p), dtype=np.float32).reshape(-1) for p in paths]
        lengths = np.array([w.shape[0] for w in waves], dtype=np.int32)
        if lengths.min() < 1:
            raise ValueError(f"empty waveform: {paths[int(np.argmin(lengths))]}")
        self.ld = _plans.padded_ld(int(lengths.max()))
        self.data = torch.zeros((len(waves), self.ld), dtype=torch.float32, device=self.eng.device)
        chunk = max(1, (256 << 20) // (4 * self.ld))  # rows per host staging buffer of at most 256 MB
        for r0 in range(0, len(waves), chunk):
            part = waves[r0:r0 + chunk]
            host = np.zeros((len(part), self.ld), dtype=np.float32)
            for k, w in enumerate(part):
                host[k, :w.shape[0]] = w
            self.data[r0:r0 + len(part)].copy_(torch.from_numpy(host))
        self.lengths = torch.from_numpy(lengths).to(self.eng.device)


#: samples per 16-byte chunk of a packed corpus
_PER_CHUNK = {"pcm16": 8, "float32": 4}


def packed_layout(lengths, dtype: str = "pcm16") -> Tuple[np.ndarray, int]:
    """Where the rows of a packed corpus go: ``(start, chunks)`` with row r at 16-byte chunk ``start[r]`` (int64) taking
    ceil(len * e / 16) chunks (e = 2 bytes per sample for ``"pcm16"``, 4 for ``"float32"``), rows back to back; ``chunks`` is
    the total, so the samples take ``16 * chunks`` bytes."""
    if dtype not in _PER_CHUNK:
        raise ValueError(f"dtype must be 'pcm16' or 'float32', not {dtype!r}")
    per = _PER_CHUNK[dtype]
    n = (np.asarray(lengths, dtype=np.int64).reshape(-1) + per - 1) // per
    start = np.zeros(n.shape[0], dtype=np.int64)
    np.cumsum(n[:-1], out=start[1:])
    return start, int(n.sum())


def pcm16_samples(wave, name: str = "") -> np.ndarray:
    """A waveform as 16-bit PCM: int16 arrays as they are, float arrays whose every sample is k / 32768 with k in
    [-32768, 32767] (what ``librosa.load`` returns for 16-bit audio) as k. ValueError naming ``name`` for anything else."""
    a = np.asarray(wave).reshape(-1)
    if a.dtype == np.int16:
        return a
    if not np.issubdtype(a.dtype, np.floating):
        raise ValueError(f"{name}: a PCM16 corpus takes int16 or float samples, not {a.dtype}")
    k = a.astype(np.float64) * 32768.0
    if a.size and not (np.all(k == np.round(k)) and k.min() >= -32768 and k.max() <= 32767):
        raise ValueError(f"{name}: samples are not 16-bit PCM (k / 32768 with integer k in [-32768, 32767]); "
                         "use dtype='float32' for this corpus")
    return k.astype(np.int16)


def pack_rows(waves, start: np.ndarray, chunks: int, dtype: str = "pcm16") -> np.ndarray:
    """The samples of a packed corpus on the host: one int16 / float32 array of ``16 * chunks`` bytes, row r at chunk
    ``start[r]`` and zeros everywhere else (every row's tail up to its chunk boundary)."""
    per = _PER_CHUNK[dtype]
    buf = np.zeros(chunks * per, dtype=np.int16 if dtype == "pcm16" else np.float32)
    for w, s in zip(waves, start):
        buf[int(s) * per:int(s) * per + w.shape[0]] = w
    return buf


def _unpin(rt, t):
    rt.cudaHostUnregister(t.data_ptr())


class PackedCorpus:
    """The rows of :class:`DeviceCorpus` -- same files, same row order (row ``idx`` bona fide, row ``N + idx*nvoc + v`` vocoder
    v's copy) -- stored back to back at their own lengths, each from a 16-byte chunk boundary, for the ``_packed`` item entries
    (``rb_items_run_packed`` / ``rb_items_stream_run_packed``), which give the same items bit for bit.

    ``dtype="pcm16"`` keeps 2 bytes per sample: every waveform must be int16 or floats k / 32768 (16-bit audio as
    ``librosa.load`` returns it; ValueError naming the file otherwise), read on the device as k / 32768 exactly.
    ``dtype="float32"`` takes any audio. ``location="device"`` puts the samples in device memory; ``location="host"`` keeps them
    in one page-locked host tensor that the gather kernel reads in place over PCIe, so that only the row starts and lengths
    (12 bytes per row) use device memory. For ASVspoof 2019 LA train with three vocoders at the lengths the loaders read, the
    samples take 1.47 GB (pcm16) or 2.94 GB (float32), against 8.71 GB for a padded :class:`DeviceCorpus`.

    Attributes: ``N``, ``nvoc``, ``list_ids``, ``ld`` (longest row rounded up to 4: the batch stride), ``lengths`` (int32
    device), ``start`` (int64 device, in chunks), ``samples`` (the flat int16 / float32 tensor), ``nbytes`` (its bytes),
    ``location`` and ``descriptor`` (the ``rb_corpus`` struct)."""

    def __init__(self, list_ids, base_dir, load_audio, vocoders=(), dtype: str = "pcm16", location: str = "device",
                 engine: Optional[Engine] = None):
        import os
        import weakref
        if dtype not in _PER_CHUNK:
            raise ValueError(f"dtype must be 'pcm16' or 'float32', not {dtype!r}")
        if location not in ("device", "host"):
            raise ValueError(f"location must be 'device' or 'host', not {location!r}")
        self.list_ids, self.vocoders, self.dtype, self.location = list(list_ids), list(vocoders), dtype, location
        self.eng = engine or default_engine()
        self.N, self.nvoc = len(self.list_ids), len(self.vocoders)
        if self.N < 1:
            raise ValueError("the corpus needs at least one utterance")
        paths = [os.path.join(base_dir, "bonafide", name) for name in self.list_ids]
        paths += [os.path.join(base_dir, "vocoded", v + "_" + name) for name in self.list_ids for v in self.vocoders]
        if dtype == "pcm16":
            waves = [pcm16_samples(load_audio(p), p) for p in paths]
        else:
            waves = [np.asarray(load_audio(p), dtype=np.float32).reshape(-1) for p in paths]
        lengths = np.array([w.shape[0] for w in waves], dtype=np.int32)
        if lengths.min() < 1:
            raise ValueError(f"empty waveform: {paths[int(np.argmin(lengths))]}")
        self.ld = _plans.padded_ld(int(lengths.max()))
        start, self.chunks = packed_layout(lengths, dtype)
        host = torch.from_numpy(pack_rows(waves, start, self.chunks, dtype))
        del waves
        self.nbytes = 16 * self.chunks
        if location == "host":
            # cudaHostRegister pins exactly these bytes (a pin_memory copy would round the allocation up to a power of two)
            rt = torch.cuda.cudart()
            rc = rt.cudaHostRegister(host.data_ptr(), self.nbytes, 0)
            if int(rc) != 0:
                raise RuntimeError(f"cudaHostRegister of {self.nbytes} bytes failed: {rc}")
            weakref.finalize(self, _unpin, rt, host)  # holds the tensor: unregistered first, freed after
            self.samples = host
        else:
            self.samples = torch.empty(host.numel(), dtype=host.dtype, device=self.eng.device)
            step = (256 << 20) // host.element_size()  # at most 256 MB per copy
            for i in range(0, host.numel(), step):
                self.samples[i:i + step].copy_(host[i:i + step])
            del host
        self.lengths = torch.from_numpy(lengths).to(self.eng.device)
        self.start = torch.from_numpy(start).to(self.eng.device)
        self.descriptor = _lib.RbCorpus(samples=self.samples.data_ptr(), kind=_lib.RB_CORPUS_PCM16 if dtype == "pcm16" else
                                        _lib.RB_CORPUS_F32, rows=len(lengths), chunks=self.chunks, start=self.start.data_ptr(),
                                        len=self.lengths.data_ptr())


class SeededItemBatcher:
    """``Dataset_for.__getitem__`` (asvspoof_2019_augall_3.py:103-146, ``augmentation_methods == ['RawBoost12']`` with
    ``online_aug``) for a batch of items seeded one by one: item g equals

        np.random.seed(seeds[g]); __getitem__(indices[g])

    -- RawBoost (algo 5) on each vocoded copy and on the anchor, ``np.random.choice`` of ``num_additional_real`` other bona fide
    utterances, one shared crop (``random_trim_nosil``) -- with every draw replayed on the device. Items are independent, so a
    whole batch runs in one pass with no host work beyond the indices and seeds. numpy's global stream is never touched;
    :class:`ItemBatcher` keeps the unseeded semantics, where consecutive items share one stream."""

    def __init__(self, args, corpus: "DeviceCorpus | PackedCorpus", num_additional_real=2, trim_length=64000, repeat_pad=True, wav_samp_rate=16000):
        self.args, self.corpus = args, corpus
        self.num_additional_real, self.trim_length = int(num_additional_real), int(trim_length)
        self.repeat_pad, self.sr = bool(repeat_pad), int(wav_samp_rate)
        if not 0 <= self.num_additional_real <= corpus.N - 1:
            raise ValueError(f"num_additional_real must lie in [0, {corpus.N - 1}] for a corpus of {corpus.N} utterances")

    def _indices(self, indices):
        if torch.is_tensor(indices):
            return indices, indices
        idx = np.asarray(indices, dtype=np.int64).reshape(-1)
        if idx.size and (idx.min() < 0 or idx.max() >= self.corpus.N):
            raise IndexError(f"indices must lie in [0, {self.corpus.N})")
        return idx.astype(np.int32), [self.corpus.list_ids[i] for i in idx]

    def items(self, indices, seeds, layout: int = LAYOUT_ITEM, end_state: Optional[torch.Tensor] = None):
        """``(ids, data, labels, out_len)`` as :meth:`ItemBatcher.items`: ``data`` [G, trim_length, V] (LAYOUT_ITEM) or
        [G, V, trim_length] (LAYOUT_MODEL), ``labels`` [G, V], ``out_len`` int32 [G], all on the device. ``indices`` and ``seeds``
        are host sequences or 32-bit device tensors; with device tensors nothing synchronises with the host and ``ids`` is the
        indices tensor itself (the utterance names stay with the caller). Device indices must lie in [0, N).
        ``end_state``: optional int32 [G, 625] device tensor that receives each item's numpy stream state after its last draw."""
        idx, ids = self._indices(indices)
        c = self.corpus
        if isinstance(c, PackedCorpus):
            data, out_len, labels = c.eng.items_run_packed(self.args, self.sr, c.descriptor, c.ld, c.nvoc, self.num_additional_real,
                                                           self.trim_length, idx, seeds, self.repeat_pad, layout, end_state=end_state)
        else:
            data, out_len, labels = c.eng.items_run(self.args, self.sr, c.data, c.lengths, c.nvoc, self.num_additional_real,
                                                    self.trim_length, idx, seeds, self.repeat_pad, layout, end_state=end_state)
        return ids, data, labels, out_len

    def draw(self, indices, seeds, end_state: bool = False):
        """The draws alone (:meth:`Engine.items_draw`): the RawBoost plan of the G*(nvoc+1) utterances, each batch row's
        corpus row and length, the crop starts and optionally the end states."""
        idx, _ = self._indices(indices)
        c = self.corpus
        return c.eng.items_draw(self.args, self.sr, c.lengths, c.nvoc, self.num_additional_real, c.ld, self.trim_length, idx, seeds,
                                end_state=end_state)


def numpy_state(row) -> tuple:
    """A stream state of the device paths (625 32-bit words: key[624], pos) as the tuple ``np.random.set_state`` takes."""
    w = np.asarray(row.cpu().numpy() if torch.is_tensor(row) else row).astype(np.int64).astype(np.uint32)
    return ("MT19937", w[:624].copy(), int(w[624]), 0, 0.0)


def _state_words(state) -> np.ndarray:
    """numpy's state tuple (``np.random.get_state()``) -> its 625 words key[624], pos; ValueError if it is not one."""
    if not isinstance(state, (tuple, list)) or len(state) < 3 or state[0] != "MT19937":
        raise ValueError("a stream state must be an MT19937 state tuple, as np.random.get_state() returns")
    key = np.asarray(state[1])
    if key.shape != (624,) or not np.issubdtype(key.dtype, np.integer) or key.min() < 0 or key.max() > 0xFFFFFFFF:
        raise ValueError("an MT19937 state needs a key of 624 32-bit words")
    pos = int(state[2])
    if not 0 <= pos <= 624:
        raise ValueError(f"an MT19937 state's pos must lie in 0..624, not {pos}")
    return np.append(key.astype(np.uint32), np.uint32(pos))


class StreamItemBatcher:
    """``Dataset_for.__getitem__`` (asvspoof_2019_augall_3.py:103-146, ``augmentation_methods == ['RawBoost12']`` with
    ``online_aug``) for items that share numpy's running stream, as the reference's loader builds them with no per-item seed:

        for idx in indices: __getitem__(idx)     # every draw from numpy's global stream, item after item

    Every draw is replayed on the device from the stream's state (``rb_items_stream_run``): one warp walks the stream's items in
    order, then the plans, the RawBoost of all items and the assembly run as a batch, as in :class:`SeededItemBatcher`. The walk
    of one stream is serial, so its time grows with the number of items in it; several independent streams (one per loader
    worker, say) walk in parallel.

    The item draws never use numpy's Gaussian cache, so ``has_gauss`` / ``cached_gaussian`` of the global state carry over."""

    def __init__(self, args, corpus: "DeviceCorpus | PackedCorpus", num_additional_real=2, trim_length=64000, repeat_pad=True, wav_samp_rate=16000):
        self.args, self.corpus = args, corpus
        self.num_additional_real, self.trim_length = int(num_additional_real), int(trim_length)
        self.repeat_pad, self.sr = bool(repeat_pad), int(wav_samp_rate)
        if not 0 <= self.num_additional_real <= corpus.N - 1:
            raise ValueError(f"num_additional_real must lie in [0, {corpus.N - 1}] for a corpus of {corpus.N} utterances")

    def _indices(self, indices) -> np.ndarray:
        idx = np.asarray(indices, dtype=np.int64).reshape(-1)
        if idx.size and (idx.min() < 0 or idx.max() >= self.corpus.N):
            raise IndexError(f"indices must lie in [0, {self.corpus.N})")
        return idx

    def _run(self, idx, stream_off, states, layout, end):
        c = self.corpus
        if isinstance(c, PackedCorpus):
            data, out_len, labels = c.eng.items_stream_run_packed(self.args, self.sr, c.descriptor, c.ld, c.nvoc,
                                                                  self.num_additional_real, self.trim_length, idx.astype(np.int32),
                                                                  stream_off, states, self.repeat_pad, layout, end_state=end)
        else:
            data, out_len, labels = c.eng.items_stream_run(self.args, self.sr, c.data, c.lengths, c.nvoc, self.num_additional_real,
                                                           self.trim_length, idx.astype(np.int32), stream_off, states,
                                                           self.repeat_pad, layout, end_state=end)
        return [c.list_ids[i] for i in idx], data, labels, out_len

    def items(self, indices: Sequence[int], layout: int = LAYOUT_ITEM):
        """Drop-in for :meth:`ItemBatcher.items`: ``(ids, data, labels, out_len)`` for ``indices`` drawn from numpy's global
        stream, which afterwards stands exactly where ``for idx in indices: __getitem__(idx)`` leaves it. Synchronises once, to
        read back the stream's end state."""
        idx = self._indices(indices)
        state = np.random.get_state()
        words = _state_words(state)[None]
        if idx.size == 0:  # nothing is drawn
            return self._run(idx, [0, 0], words, layout, None)
        end = torch.empty((1, 625), dtype=torch.int32, device=self.corpus.eng.device)
        out = self._run(idx, [0, idx.size], words, layout, end)
        e = numpy_state(end[0])
        np.random.set_state(e[:3] + tuple(state[3:5]))
        return out

    def items_streams(self, index_lists: Sequence[Sequence[int]], states, layout: int = LAYOUT_ITEM):
        """S independent streams, e.g. one per loader worker: the items of ``index_lists[q]`` are drawn one after another from
        ``states[q]`` -- numpy state tuples, or an int32 [S, 625] device tensor of key[624], pos as the end states below.
        Returns ``(ids, data, labels, out_len, end_states)``: the items in stream order (stream 0's, then stream 1's, ...) as
        :meth:`items` returns them, and int32 [S, 625] device tensor of each stream's state after its last draw
        (:func:`numpy_state` turns a row into a tuple for ``np.random.set_state``). numpy's global stream is not touched, and
        nothing is read back from the device.

        End states are stored with pos 0..623: a used-up block (pos 624, as right after ``np.random.seed``) comes back as the
        next block at pos 0, also for an empty stream. The one exception is a call with no item at all: nothing is launched and
        the end states are the start states exactly as given, so a pos of 624 stays 624. Both forms continue the same stream."""
        lists = [self._indices(ix) for ix in index_lists]
        S = len(lists)
        if torch.is_tensor(states):
            if states.dtype not in (torch.int32, torch.uint32) or tuple(states.shape) != (S, 625):
                raise ValueError(f"states must be an int32 (or uint32) [S, 625] tensor with S = {S}")
        else:
            states = list(states)
            if len(states) != S:
                raise ValueError("one state per index list")
            states = np.stack([_state_words(s) for s in states]) if S else np.zeros((0, 625), np.uint32)
        idx = np.concatenate(lists) if S else np.zeros(0, np.int64)
        stream_off = np.concatenate([[0], np.cumsum([ix.size for ix in lists])]).astype(np.int32)
        dev = self.corpus.eng.device
        if idx.size == 0:  # nothing is drawn: every stream ends where it starts
            end = states.clone() if torch.is_tensor(states) else torch.from_numpy(states.view(np.int32)).to(dev)
            return (*self._run(idx, stream_off, states, layout, None), end)
        end = torch.empty((S, 625), dtype=torch.int32, device=dev)
        return (*self._run(idx, stream_off, states, layout, end), end)


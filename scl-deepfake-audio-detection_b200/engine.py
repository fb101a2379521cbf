"""Batched device execution of RawBoost plans through the C ABI.

PyTorch is plumbing only here (device memory, streams, pinned buffers); all arithmetic happens in
``lib/librawboost_b200.so``. There is no CPU fallback: constructing an :class:`Engine` without CUDA raises.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from .plans import BatchPlan, padded_ld


@dataclass
class DevicePlan:
    """A :class:`BatchPlan` whose arrays live on the device; ``struct`` is the ``rb_plan`` passed to the ABI."""
    B: int
    ld: int
    lengths: torch.Tensor
    tensors: dict
    struct: _lib.RbPlan
    host: Optional[BatchPlan] = None


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


class Engine:
    """One engine per (process, device). Owns a growable device workspace; thread-compatible, not thread-safe."""

    def __init__(self, device: int | str | torch.device = 0):
        if not torch.cuda.is_available():
            raise _lib.RawBoostLibraryError("rawboost_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        self.device = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
        major, _ = torch.cuda.get_device_capability(self.device)
        if major != 10:
            raise _lib.RawBoostLibraryError(f"rawboost_b200 is built for sm_100a only; device capability is {major}.x")
        self._ws: Optional[torch.Tensor] = None
        self._ctx = None

    # -- memory ---------------------------------------------------------------------------------------
    def workspace(self, B: int, ld: int, algo: int = 8) -> torch.Tensor:
        """Growable device workspace, sized for what ``algo`` needs (algo 8 needs the most)."""
        return self._scratch(int(self.lib.rb_workspace_bytes_for(int(algo), B, ld)))

    def _scratch(self, need: int) -> torch.Tensor:
        if self._ws is None or self._ws.numel() < need + 256:
            self._ws = None
            self._ws = torch.empty(need + 256, dtype=torch.uint8, device=self.device)
        return self._ws

    @staticmethod
    def _ws_ptr(ws: torch.Tensor) -> int:
        return (ws.data_ptr() + 255) // 256 * 256

    def upload_plan(self, plan: BatchPlan, non_blocking: bool = True) -> DevicePlan:
        """Copy the CSR arrays of a host plan to the device (pinned staging when available)."""
        t = {}
        for name in ("lnl_taps", "lnl_tap_off", "isd_off", "isd_idx", "isd_fr", "ssi_noise", "ssi_taps", "ssi_tap_off", "ssi_snr_db"):
            arr = getattr(plan, name)
            if arr is not None:
                src = torch.from_numpy(np.ascontiguousarray(arr))
                if src.numel() == 0:
                    # an empty CUDA tensor has a NULL data pointer, which the ABI reads as a missing plan field; a batch
                    # whose utterances draw no impulses at all has empty isd_idx / isd_fr and must still run
                    src = torch.zeros(1, dtype=src.dtype)
                t[name] = src.to(self.device, non_blocking=False)
            else:
                t[name] = None
        lengths = torch.from_numpy(np.ascontiguousarray(plan.lengths)).to(self.device)
        s = _lib.RbPlan()
        s.n_f = int(plan.n_f)
        s.g_sd = float(plan.g_sd)
        for name, v in t.items():
            setattr(s, name, None if v is None else v.data_ptr())
        return DevicePlan(B=plan.B, ld=plan.ld, lengths=lengths, tensors=t, struct=s, host=plan)

    def draw_device_plan(self, lengths: torch.Tensor, seeds, sr, args, algo: int, ld: int) -> DevicePlan:
        """Draw the plans of a seeded batch ON THE DEVICE (``rb_devplan_draw``): ``np.random.seed(seeds[u])`` precedes
        utterance u, exactly as ``plans.draw_batch(..., seeds=...)`` / ``NativePlanner.draw`` do on the host. Asynchronous on
        torch's current stream; the returned plan's arrays live in one device buffer owned by the plan."""
        B = int(lengths.numel())
        if not torch.is_tensor(seeds):
            seeds = torch.from_numpy(np.ascontiguousarray(seeds, dtype=np.uint32).view(np.int32)).to(self.device)
        a = _lib.args_struct(args, sr)
        need = int(self.lib.rb_devplan_bytes(C.byref(a), int(algo), B, int(ld)))
        store = torch.empty(need + 256, dtype=torch.uint8, device=self.device)
        s = _lib.RbPlan()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            rc = self.lib.rb_devplan_draw(C.byref(a), int(algo), B, int(ld), _ptr(lengths), _ptr(seeds), C.c_void_p(self._ws_ptr(store)),
                                          need, C.byref(s), C.c_void_p(stream))
        _lib.check(rc, f"rb_devplan_draw(algo={algo})")
        return DevicePlan(B=B, ld=int(ld), lengths=lengths, tensors={"storage": store, "seeds": seeds}, struct=s, host=None)

    def download_plan(self, dp: DevicePlan) -> BatchPlan:
        """Copy a device-drawn plan back to the host (tests / inspection)."""
        store = dp.tensors["storage"]

        def fetch(ptr, count, dtype):
            if not ptr or count == 0:
                return np.zeros(0, dtype=dtype)
            off = int(ptr) - store.data_ptr()
            return store[off:off + count * np.dtype(dtype).itemsize].cpu().numpy().view(dtype).copy()

        s, B, ld = dp.struct, dp.B, dp.ld
        bp = BatchPlan(B=B, ld=ld, lengths=dp.lengths.cpu().numpy(), g_sd=float(s.g_sd))
        if s.lnl_tap_off:
            bp.n_f = int(s.n_f)
            bp.lnl_tap_off = fetch(s.lnl_tap_off, B * bp.n_f + 1, np.int32)
            bp.lnl_taps = fetch(s.lnl_taps, int(bp.lnl_tap_off[-1]), np.float32)
        if s.isd_off:
            bp.isd_off = fetch(s.isd_off, B + 1, np.int32)
            bp.isd_idx = fetch(s.isd_idx, int(bp.isd_off[-1]), np.int32)
            bp.isd_fr = fetch(s.isd_fr, int(bp.isd_off[-1]), np.float64)
        if s.ssi_tap_off:
            bp.ssi_noise = fetch(s.ssi_noise, B * ld, np.float32).reshape(B, ld)
            bp.ssi_tap_off = fetch(s.ssi_tap_off, B + 1, np.int32)
            bp.ssi_taps = fetch(s.ssi_taps, int(bp.ssi_tap_off[-1]), np.float32)
            bp.ssi_snr_db = fetch(s.ssi_snr_db, B, np.float32)
        return bp

    def _item_arrays(self, indices, seeds):
        """indices / seeds as int32 device tensors (seeds hold the uint32 bit patterns)."""
        if not torch.is_tensor(indices):
            indices = torch.from_numpy(np.ascontiguousarray(indices, dtype=np.int32)).to(self.device)
        if not torch.is_tensor(seeds):
            seeds = torch.from_numpy(np.ascontiguousarray(np.asarray(seeds, dtype=np.int64).astype(np.uint32)).view(np.int32)).to(self.device)
        for name, t in (("indices", indices), ("seeds", seeds)):
            if t.device != self.device or t.element_size() != 4 or t.dim() != 1 or not t.is_contiguous():
                raise ValueError(f"{name} must be a contiguous 1-D 32-bit integer tensor on {self.device}")
        if indices.numel() != seeds.numel():
            raise ValueError("one seed per item")
        return indices, seeds

    def items_draw(self, args, sr, corpus_len: torch.Tensor, nvoc: int, n_add: int, ld: int, trim: int, indices, seeds,
                   end_state: bool = False):
        """Every draw of G independently seeded items (``rb_items_draw``; see ``multiview.SeededItemBatcher``). ``corpus_len``:
        int32 [N*(1+nvoc)] device lengths of the corpus rows. Returns a dict: ``plan`` (a :class:`DevicePlan` of the G*(nvoc+1)
        RawBoost utterances, owning its device buffer), ``src_row`` and ``row_len`` (int32 [G*(nvoc+1+n_add)]), ``start``
        (int32 [G]) and, with ``end_state``, ``end_state`` (int32 [G, 625]: each item's numpy state key[624], pos after its
        last draw, as uint32 bit patterns). Asynchronous on torch's current stream."""
        indices, seeds = self._item_arrays(indices, seeds)
        G, R = int(indices.numel()), int(corpus_len.numel())
        if corpus_len.dtype != torch.int32 or corpus_len.device != self.device or R % (1 + nvoc):
            raise ValueError("corpus_len must be int32 [N*(1+nvoc)] on the engine's device")
        N = R // (1 + nvoc)
        a = _lib.args_struct(args, sr)
        need = int(self.lib.rb_items_workspace_bytes(C.byref(a), G, int(nvoc), int(n_add), N, int(ld)))
        if G and need == 0:
            raise ValueError(f"unsupported item shape: G={G}, nvoc={nvoc}, n_add={n_add}, N={N}, ld={ld}")
        store = torch.empty(need + 256, dtype=torch.uint8, device=self.device)
        rows = G * (nvoc + 1 + n_add)
        src_row = torch.empty(rows, dtype=torch.int32, device=self.device)
        row_len = torch.empty(rows, dtype=torch.int32, device=self.device)
        start = torch.empty(G, dtype=torch.int32, device=self.device)
        end = torch.empty((G, 625), dtype=torch.int32, device=self.device) if end_state else None
        s = _lib.RbPlan()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            rc = self.lib.rb_items_draw(C.byref(a), G, int(nvoc), int(n_add), N, int(ld), int(trim), _ptr(corpus_len), _ptr(indices),
                                        _ptr(seeds), _ptr(src_row), _ptr(row_len), _ptr(start), _ptr(end),
                                        C.c_void_p(self._ws_ptr(store)), need, C.byref(s), C.c_void_p(stream))
        _lib.check(rc, "rb_items_draw")
        B = G * (nvoc + 1)
        plan = DevicePlan(B=B, ld=int(ld), lengths=row_len[:B], tensors={"storage": store}, struct=s, host=None)
        return {"plan": plan, "src_row": src_row, "row_len": row_len, "start": start, "end_state": end}

    def items_run(self, args, sr, corpus: torch.Tensor, corpus_len: torch.Tensor, nvoc: int, n_add: int, trim: int, indices, seeds,
                  repeat_pad: bool = True, layout: int = 0, out: Optional[torch.Tensor] = None, with_labels: bool = True,
                  end_state: Optional[torch.Tensor] = None):
        """Whole items, every step on the device (``rb_items_run``): draw, gather, RawBoost (algo 5), crop and view assembly.
        ``corpus`` [N*(1+nvoc), ld] float32 with lengths ``corpus_len`` (int32). Returns ``(out, out_len, labels)``: out
        [G, trim, V] (layout 0) or [G, V, trim] (layout 1), zero past out_len[g]; labels [G, V] (None without ``with_labels``).
        ``end_state``: optional int32 [G, 625] device tensor for each item's final stream state. Asynchronous on torch's
        current stream; with device ``indices`` / ``seeds`` nothing synchronises with the host."""
        indices, seeds = self._item_arrays(indices, seeds)
        if corpus.dtype != torch.float32 or corpus.dim() != 2 or not corpus.is_contiguous() or corpus.device != self.device:
            raise ValueError("corpus must be a contiguous [R, ld] float32 tensor on the engine's device")
        R, ld = corpus.shape
        if corpus_len.dtype != torch.int32 or corpus_len.device != self.device or corpus_len.numel() != R or R % (1 + nvoc):
            raise ValueError("corpus_len must be int32 [R] on the engine's device, R = N*(1+nvoc)")
        N, G, V = R // (1 + nvoc), int(indices.numel()), 2 + n_add + 2 * nvoc
        shape = (G, trim, V) if layout == 0 else (G, V, trim)
        if out is None:
            out = torch.zeros(shape, dtype=torch.float32, device=self.device)
        elif tuple(out.shape) != shape or out.dtype != torch.float32 or not out.is_contiguous() or out.device != self.device:
            raise ValueError(f"out must be a contiguous float32 tensor {shape} on the engine's device")
        if end_state is not None and (end_state.shape != (G, 625) or end_state.element_size() != 4 or end_state.device != self.device):
            raise ValueError("end_state must be a 32-bit [G, 625] tensor on the engine's device")
        out_len = torch.empty(G, dtype=torch.int32, device=self.device)
        labels = torch.empty((G, V), dtype=torch.float32, device=self.device) if with_labels else None
        a = _lib.args_struct(args, sr)
        need = int(self.lib.rb_items_workspace_bytes(C.byref(a), G, int(nvoc), int(n_add), N, int(ld)))
        if G and need == 0:
            raise ValueError(f"unsupported item shape: G={G}, nvoc={nvoc}, n_add={n_add}, N={N}, ld={ld}")
        ws = self._scratch(need)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            rc = self.lib.rb_items_run(C.byref(a), G, int(nvoc), int(n_add), N, int(ld), int(trim), int(bool(repeat_pad)), int(layout),
                                       _ptr(corpus), _ptr(corpus_len), _ptr(indices), _ptr(seeds), _ptr(out), _ptr(out_len), _ptr(labels),
                                       _ptr(end_state), C.c_void_p(self._ws_ptr(ws)), need, C.c_void_p(stream))
        _lib.check(rc, "rb_items_run")
        return out, out_len, labels

    def _upload(self, host: np.ndarray) -> torch.Tensor:
        """A host array on the device, copied on torch's current stream through page-locked staging: unlike a copy from
        pageable memory, it does not make the host wait for the work already queued on that stream."""
        host = torch.from_numpy(np.ascontiguousarray(host))
        if host.numel() == 0:
            return torch.empty(host.shape, dtype=host.dtype, device=self.device)
        return host.pin_memory().to(self.device, non_blocking=True)

    def _stream_arrays(self, indices, stream_off, start_state):
        """indices, stream_off and start_state as 32-bit device tensors (start_state [S, 625] holds the uint32 bit patterns of
        numpy's key[624], pos)."""
        if not torch.is_tensor(indices):
            indices = self._upload(np.asarray(indices, dtype=np.int32))
        if not torch.is_tensor(stream_off):
            stream_off = self._upload(np.asarray(stream_off, dtype=np.int32))
        if not torch.is_tensor(start_state):
            host = np.asarray(start_state, dtype=np.int64).reshape(-1, 625).astype(np.uint32)
            start_state = self._upload(host.view(np.int32))
        for name, t, dim, dtypes in (("indices", indices, 1, (torch.int32,)), ("stream_off", stream_off, 1, (torch.int32,)),
                                     ("start_state", start_state, 2, (torch.int32, torch.uint32))):
            if t.device != self.device or t.dtype not in dtypes or t.dim() != dim or not t.is_contiguous():
                raise ValueError(f"{name} must be a contiguous {dim}-D {' or '.join(map(str, dtypes))} tensor on {self.device}")
        S = int(stream_off.numel()) - 1
        if S < 0 or start_state.shape != (S, 625):
            raise ValueError("stream_off needs S+1 entries and start_state S rows of 625 words")
        return indices, stream_off, start_state, S

    def _stream_end(self, S: int, end_state):
        if end_state is None or torch.is_tensor(end_state):
            if end_state is not None and (end_state.shape != (S, 625) or end_state.dtype not in (torch.int32, torch.uint32)
                                          or end_state.device != self.device
                                          or not end_state.is_contiguous()):
                raise ValueError("end_state must be a contiguous 32-bit [S, 625] tensor on the engine's device")
            return end_state
        return torch.empty((S, 625), dtype=torch.int32, device=self.device) if end_state else None

    def items_stream_draw(self, args, sr, corpus_len: torch.Tensor, nvoc: int, n_add: int, ld: int, trim: int, indices, stream_off,
                          start_state, end_state=False):
        """:meth:`items_draw` for items that share running numpy streams (``rb_items_stream_draw``; see
        ``multiview.StreamItemBatcher``): stream q walks the items ``[stream_off[q], stream_off[q+1])`` of ``indices`` in order,
        from ``start_state[q]`` (numpy's key[624], pos). ``stream_off`` ([S+1]) and ``start_state`` ([S, 625]) are host arrays or
        32-bit device tensors. ``end_state``: True (a new tensor) or an int32 [S, 625] device tensor that receives each stream's
        state after its last draw. Returns the dict of :meth:`items_draw`; its ``end_state`` is per stream. Asynchronous on torch's
        current stream; with device inputs nothing synchronises with the host."""
        indices, stream_off, start_state, S = self._stream_arrays(indices, stream_off, start_state)
        end = self._stream_end(S, end_state)
        G, R = int(indices.numel()), int(corpus_len.numel())
        if corpus_len.dtype != torch.int32 or corpus_len.device != self.device or R % (1 + nvoc):
            raise ValueError("corpus_len must be int32 [N*(1+nvoc)] on the engine's device")
        N = R // (1 + nvoc)
        a = _lib.args_struct(args, sr)
        need = int(self.lib.rb_items_workspace_bytes(C.byref(a), G, int(nvoc), int(n_add), N, int(ld)))
        if G and need == 0:
            raise ValueError(f"unsupported item shape: G={G}, nvoc={nvoc}, n_add={n_add}, N={N}, ld={ld}")
        store = torch.empty(need + 256, dtype=torch.uint8, device=self.device)
        rows = G * (nvoc + 1 + n_add)
        src_row = torch.empty(rows, dtype=torch.int32, device=self.device)
        row_len = torch.empty(rows, dtype=torch.int32, device=self.device)
        start = torch.empty(G, dtype=torch.int32, device=self.device)
        s = _lib.RbPlan()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            rc = self.lib.rb_items_stream_draw(C.byref(a), S, _ptr(stream_off), G, int(nvoc), int(n_add), N, int(ld), int(trim),
                                               _ptr(corpus_len), _ptr(indices), _ptr(start_state), _ptr(src_row), _ptr(row_len),
                                               _ptr(start), _ptr(end), C.c_void_p(self._ws_ptr(store)), need, C.byref(s),
                                               C.c_void_p(stream))
        _lib.check(rc, "rb_items_stream_draw")
        B = G * (nvoc + 1)
        plan = DevicePlan(B=B, ld=int(ld), lengths=row_len[:B], tensors={"storage": store}, struct=s, host=None)
        return {"plan": plan, "src_row": src_row, "row_len": row_len, "start": start, "end_state": end}

    def items_stream_run(self, args, sr, corpus: torch.Tensor, corpus_len: torch.Tensor, nvoc: int, n_add: int, trim: int, indices,
                         stream_off, start_state, repeat_pad: bool = True, layout: int = 0, out: Optional[torch.Tensor] = None,
                         with_labels: bool = True, end_state=None):
        """:meth:`items_run` for items that share running numpy streams (``rb_items_stream_run``): ``stream_off``,
        ``start_state`` and ``end_state`` as :meth:`items_stream_draw`. Returns ``(out, out_len, labels)`` as :meth:`items_run`.
        Asynchronous on torch's current stream; with device inputs nothing synchronises with the host."""
        indices, stream_off, start_state, S = self._stream_arrays(indices, stream_off, start_state)
        if end_state is not None and not torch.is_tensor(end_state):
            raise ValueError("end_state must be None or an int32 [S, 625] device tensor")
        end = self._stream_end(S, end_state)
        if corpus.dtype != torch.float32 or corpus.dim() != 2 or not corpus.is_contiguous() or corpus.device != self.device:
            raise ValueError("corpus must be a contiguous [R, ld] float32 tensor on the engine's device")
        R, ld = corpus.shape
        if corpus_len.dtype != torch.int32 or corpus_len.device != self.device or corpus_len.numel() != R or R % (1 + nvoc):
            raise ValueError("corpus_len must be int32 [R] on the engine's device, R = N*(1+nvoc)")
        N, G, V = R // (1 + nvoc), int(indices.numel()), 2 + n_add + 2 * nvoc
        shape = (G, trim, V) if layout == 0 else (G, V, trim)
        if out is None:
            out = torch.zeros(shape, dtype=torch.float32, device=self.device)
        elif tuple(out.shape) != shape or out.dtype != torch.float32 or not out.is_contiguous() or out.device != self.device:
            raise ValueError(f"out must be a contiguous float32 tensor {shape} on the engine's device")
        out_len = torch.empty(G, dtype=torch.int32, device=self.device)
        labels = torch.empty((G, V), dtype=torch.float32, device=self.device) if with_labels else None
        a = _lib.args_struct(args, sr)
        need = int(self.lib.rb_items_workspace_bytes(C.byref(a), G, int(nvoc), int(n_add), N, int(ld)))
        if G and need == 0:
            raise ValueError(f"unsupported item shape: G={G}, nvoc={nvoc}, n_add={n_add}, N={N}, ld={ld}")
        ws = self._scratch(need)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            rc = self.lib.rb_items_stream_run(C.byref(a), S, _ptr(stream_off), G, int(nvoc), int(n_add), N, int(ld), int(trim),
                                              int(bool(repeat_pad)), int(layout), _ptr(corpus), _ptr(corpus_len), _ptr(indices),
                                              _ptr(start_state), _ptr(out), _ptr(out_len), _ptr(labels), _ptr(end),
                                              C.c_void_p(self._ws_ptr(ws)), need, C.c_void_p(stream))
        _lib.check(rc, "rb_items_stream_run")
        return out, out_len, labels

    def _packed_items_setup(self, args, sr, corpus: _lib.RbCorpus, ld: int, nvoc: int, n_add: int, trim: int, G: int, layout: int,
                            out: Optional[torch.Tensor], with_labels: bool):
        """Shape, outputs and workspace of the ``_packed`` item entries: ``(N, out, out_len, labels, args struct, ws, need)``."""
        if not isinstance(corpus, _lib.RbCorpus):
            raise TypeError("corpus must be an RbCorpus descriptor (multiview.PackedCorpus.descriptor)")
        R = int(corpus.rows)
        if R <= 0 or R % (1 + nvoc):
            raise ValueError("the corpus needs N*(1+nvoc) rows")
        N, V = R // (1 + nvoc), 2 + n_add + 2 * nvoc
        shape = (G, trim, V) if layout == 0 else (G, V, trim)
        if out is None:
            out = torch.zeros(shape, dtype=torch.float32, device=self.device)
        elif tuple(out.shape) != shape or out.dtype != torch.float32 or not out.is_contiguous() or out.device != self.device:
            raise ValueError(f"out must be a contiguous float32 tensor {shape} on the engine's device")
        out_len = torch.empty(G, dtype=torch.int32, device=self.device)
        labels = torch.empty((G, V), dtype=torch.float32, device=self.device) if with_labels else None
        a = _lib.args_struct(args, sr)
        need = int(self.lib.rb_items_workspace_bytes(C.byref(a), G, int(nvoc), int(n_add), N, int(ld)))
        if G and need == 0:
            raise ValueError(f"unsupported item shape: G={G}, nvoc={nvoc}, n_add={n_add}, N={N}, ld={ld}")
        return N, out, out_len, labels, a, self._scratch(need), need

    def items_run_packed(self, args, sr, corpus: _lib.RbCorpus, ld: int, nvoc: int, n_add: int, trim: int, indices, seeds,
                         repeat_pad: bool = True, layout: int = 0, out: Optional[torch.Tensor] = None, with_labels: bool = True,
                         end_state: Optional[torch.Tensor] = None):
        """:meth:`items_run` from a packed corpus (``rb_items_run_packed``): ``corpus`` is the ``rb_corpus`` descriptor of
        ``multiview.PackedCorpus`` (samples in device or page-locked host memory, row starts and lengths on the device), ``ld``
        the row stride of the gathered batch (a multiple of 4, at least the longest row). Same results as :meth:`items_run` on a
        padded corpus of the same values, bit for bit."""
        indices, seeds = self._item_arrays(indices, seeds)
        G = int(indices.numel())
        if end_state is not None and (end_state.shape != (G, 625) or end_state.element_size() != 4 or end_state.device != self.device):
            raise ValueError("end_state must be a 32-bit [G, 625] tensor on the engine's device")
        N, out, out_len, labels, a, ws, need = self._packed_items_setup(args, sr, corpus, ld, nvoc, n_add, trim, G, layout, out,
                                                                        with_labels)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            rc = self.lib.rb_items_run_packed(C.byref(a), G, int(nvoc), int(n_add), N, int(ld), int(trim), int(bool(repeat_pad)),
                                              int(layout), C.byref(corpus), _ptr(indices), _ptr(seeds), _ptr(out), _ptr(out_len),
                                              _ptr(labels), _ptr(end_state), C.c_void_p(self._ws_ptr(ws)), need, C.c_void_p(stream))
        _lib.check(rc, "rb_items_run_packed")
        return out, out_len, labels

    def items_stream_run_packed(self, args, sr, corpus: _lib.RbCorpus, ld: int, nvoc: int, n_add: int, trim: int, indices,
                                stream_off, start_state, repeat_pad: bool = True, layout: int = 0,
                                out: Optional[torch.Tensor] = None, with_labels: bool = True, end_state=None):
        """:meth:`items_stream_run` from a packed corpus (``rb_items_stream_run_packed``); ``corpus`` and ``ld`` as
        :meth:`items_run_packed`."""
        indices, stream_off, start_state, S = self._stream_arrays(indices, stream_off, start_state)
        if end_state is not None and not torch.is_tensor(end_state):
            raise ValueError("end_state must be None or an int32 [S, 625] device tensor")
        end = self._stream_end(S, end_state)
        G = int(indices.numel())
        N, out, out_len, labels, a, ws, need = self._packed_items_setup(args, sr, corpus, ld, nvoc, n_add, trim, G, layout, out,
                                                                        with_labels)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            rc = self.lib.rb_items_stream_run_packed(C.byref(a), S, _ptr(stream_off), G, int(nvoc), int(n_add), N, int(ld), int(trim),
                                                     int(bool(repeat_pad)), int(layout), C.byref(corpus), _ptr(indices),
                                                     _ptr(start_state), _ptr(out), _ptr(out_len), _ptr(labels), _ptr(end),
                                                     C.c_void_p(self._ws_ptr(ws)), need, C.c_void_p(stream))
        _lib.check(rc, "rb_items_stream_run_packed")
        return out, out_len, labels

    def pack_waveforms(self, waves: Sequence[np.ndarray], ld: Optional[int] = None):
        """Host list of 1-D float arrays -> ([B, ld] float32 device tensor, int32 lengths on device)."""
        lengths = np.array([int(w.shape[0]) for w in waves], dtype=np.int32)
        ld = ld or padded_ld(int(lengths.max()) if len(waves) else 0)
        host = np.zeros((len(waves), ld), dtype=np.float32)
        for u, w in enumerate(waves):
            host[u, :lengths[u]] = np.asarray(w, dtype=np.float32)
        return torch.from_numpy(host).to(self.device), torch.from_numpy(lengths).to(self.device)

    # -- execution ------------------------------------------------------------------------------------
    def process(self, algo: int, x: torch.Tensor, lengths: torch.Tensor, plan: Optional[DevicePlan],
                out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """``process_Rawboost_feature`` for a whole batch on the device: x [B, ld] float32 -> new [B, ld] tensor.

        Asynchronous on torch's current stream. Samples beyond ``lengths[u]`` of the output row are zero when the
        tensor is allocated here, untouched when ``out`` is passed."""
        self._check_batch(x, lengths)
        B, ld = x.shape
        if plan is not None and (plan.B != B or plan.ld != ld):  # CSR offsets and the SSI noise rows are laid out for (B, ld)
            raise ValueError(f"plan was packed for B={plan.B}, ld={plan.ld}; the batch is B={B}, ld={ld}")
        if out is None:
            out = torch.zeros_like(x)
        ws = self.workspace(B, ld, algo)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        ps = C.byref(plan.struct) if plan is not None else None
        with torch.cuda.device(self.device):
            rc = self.lib.rb_process(int(algo), _ptr(x), _ptr(lengths), B, ld, ps, _ptr(out), C.c_void_p(self._ws_ptr(ws)),
                                     ws.numel() - 256, C.c_void_p(stream))
        _lib.check(rc, f"rb_process(algo={algo})")
        return out

    def filter_fir(self, x: torch.Tensor, lengths: torch.Tensor, taps: torch.Tensor, tap_off: torch.Tensor,
                   out: Optional[torch.Tensor] = None) -> torch.Tensor:
        self._check_batch(x, lengths)
        B, ld = x.shape
        if out is None:
            out = torch.zeros_like(x)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            rc = self.lib.rb_filter_fir(_ptr(x), _ptr(lengths), B, ld, _ptr(taps), _ptr(tap_off), _ptr(out), C.c_void_p(stream))
        _lib.check(rc, "rb_filter_fir")
        return out

    def normwav(self, x: torch.Tensor, lengths: torch.Tensor, always: bool, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        self._check_batch(x, lengths)
        B, ld = x.shape
        if out is None:
            out = torch.zeros_like(x)
        ws = self.workspace(B, ld, 0)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            rc = self.lib.rb_normwav(_ptr(x), _ptr(lengths), B, ld, int(bool(always)), _ptr(out), C.c_void_p(self._ws_ptr(ws)),
                                     ws.numel() - 256, C.c_void_p(stream))
        _lib.check(rc, "rb_normwav")
        return out

    def reverb(self, x: torch.Tensor, lengths: torch.Tensor, rir: torch.Tensor, rir_off: torch.Tensor,
               out: Optional[torch.Tensor] = None, ld_out: Optional[int] = None, max_taps: Optional[int] = None):
        """Reverb view of every row (``rb_reverb``): ``normWav(np.convolve(x_u, h_u), 1)`` with h_u = ``rir[rir_off[u]:rir_off[u+1]]``.
        All tensors live on the engine's device: x [B, ld] float32, lengths / rir_off int32, rir float32. Returns
        (y [B, ld_out] float32, out_len int32 [B]) with out_len[u] = lengths[u] + K_u - 1 (0 for an empty row, -1 for a row that
        was not computed: K_u < 1, or an output longer than ld_out); samples of y beyond out_len[u] are untouched.

        The row stride of the result is ``out.shape[1]`` when ``out`` is given, else ``ld_out``. With neither, it is sized from
        the lengths and offsets, which this READS BACK to the host; the call then also waits for the result and raises
        ``ValueError`` if any row was not computed. Otherwise it is asynchronous on torch's current stream, with no host
        synchronisation, and the caller inspects ``out_len``.

        ``max_taps`` (the longest impulse response, when the caller knows it) sizes the workspace and the spectrum grid
        without a read-back: one 64 KB spectrum per row and 8192 taps. Without it the asynchronous form sizes for the longest
        impulse response the output stride allows. A row with more taps than the workspace then holds (``max_taps`` rounded up to
        whole 8192-tap partitions) is not computed (out_len -1)."""
        self._check_batch(x, lengths)
        B, ld = x.shape
        if rir.device != self.device or rir_off.device != self.device:
            raise ValueError(f"tensors must live on {self.device}")
        if rir.dtype != torch.float32 or not rir.is_contiguous() or rir_off.dtype != torch.int32 or rir_off.numel() != B + 1:
            raise ValueError("rir must be a contiguous float32 tensor and rir_off int32 [B + 1]")
        if out is not None:
            if out.device != self.device or out.dtype != torch.float32 or out.dim() != 2 or out.shape[0] != B or not out.is_contiguous():
                raise ValueError("out must be a contiguous [B, ld_out] float32 tensor on the engine's device")
            if ld_out is not None and int(ld_out) != out.shape[1]:
                raise ValueError(f"ld_out={ld_out} but out has {out.shape[1]} columns")
            ld_out = out.shape[1]
        read_back = ld_out is None
        if read_back:
            n = lengths.cpu().numpy().astype(np.int64)
            k = np.diff(rir_off.cpu().numpy().astype(np.int64))
            max_taps = int(k.max()) if B else 1
            ld_out = padded_ld(int(np.max(np.where((n > 0) & (k > 0), n + k - 1, 0))) if B else 0)
        elif max_taps is None:
            # a computed row never has more taps than output samples; rir.numel() bounds every row as well
            max_taps = max(1, min(int(ld_out), rir.numel()))
        if out is None:
            out = torch.zeros((B, int(ld_out)), dtype=torch.float32, device=self.device)
        out_len = torch.empty(B, dtype=torch.int32, device=self.device)
        need = int(self.lib.rb_reverb_workspace_bytes(B, int(max_taps)))
        ws = self._scratch(need)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            rc = self.lib.rb_reverb(_ptr(x), _ptr(lengths), B, ld, _ptr(rir), _ptr(rir_off), _ptr(out), int(ld_out), _ptr(out_len),
                                    C.c_void_p(self._ws_ptr(ws)), need, C.c_void_p(stream))  # exactly `need`: sets the partitions
        _lib.check(rc, "rb_reverb")
        if read_back:
            bad = np.flatnonzero(out_len.cpu().numpy() < 0)
            if bad.size:
                raise ValueError(f"rb_reverb did not compute rows {bad.tolist()[:8]}: every impulse response needs at least one "
                                 f"tap and every length must lie in [0, {ld}]")
        return out, out_len

    def _check_batch(self, x: torch.Tensor, lengths: torch.Tensor) -> None:
        if x.device != self.device or lengths.device != self.device:
            raise ValueError(f"tensors must live on {self.device}")
        if x.dtype != torch.float32 or x.dim() != 2 or not x.is_contiguous():
            raise ValueError("x must be a contiguous [B, ld] float32 tensor")
        if lengths.dtype != torch.int32 or lengths.numel() != x.shape[0]:
            raise ValueError("lengths must be int32 [B]")

    # -- host-buffer path (rb_process_host): what a non-torch caller of the C ABI would use ---------------
    def process_host(self, algo: int, x: np.ndarray, plan: Optional[BatchPlan], out: Optional[np.ndarray] = None) -> np.ndarray:
        """x: [B, ld] float32 host array (pinned for asynchronous DMA); plan: host :class:`BatchPlan`.
        Copies in, computes, copies out; returns when ``out`` is complete."""
        self._host_ctx()
        if x.dtype != np.float32 or x.ndim != 2 or not x.flags.c_contiguous:
            raise ValueError("x must be a C-contiguous [B, ld] float32 array")
        B, ld = x.shape
        if plan is not None and (plan.B != B or plan.ld != ld):
            raise ValueError(f"plan was packed for B={plan.B}, ld={plan.ld}; the batch is B={B}, ld={ld}")
        if out is None:
            out = np.zeros_like(x)
        s = _lib.RbPlan()
        keep = []
        lengths = plan.lengths if plan is not None else np.full(B, ld, dtype=np.int32)
        if plan is not None:
            s.n_f = int(plan.n_f)
            s.g_sd = float(plan.g_sd)
            for name in ("lnl_taps", "lnl_tap_off", "isd_off", "isd_idx", "isd_fr", "ssi_noise", "ssi_taps", "ssi_tap_off", "ssi_snr_db"):
                arr = getattr(plan, name)
                if arr is not None:
                    arr = np.ascontiguousarray(arr)
                    keep.append(arr)
                    setattr(s, name, arr.ctypes.data)
        lengths = np.ascontiguousarray(lengths, dtype=np.int32)
        rc = self.lib.rb_process_host(self._ctx, int(algo), C.c_void_p(x.ctypes.data), C.c_void_p(lengths.ctypes.data), B, ld,
                                      C.byref(s), C.c_void_p(out.ctypes.data))
        _lib.check(rc, f"rb_process_host(algo={algo})")
        return out

    def _host_ctx(self):
        if self._ctx is None:
            ctx = C.c_void_p()
            _lib.check(self.lib.rb_ctx_create(C.byref(ctx), self.device.index or 0), "rb_ctx_create")
            self._ctx = ctx
        return self._ctx

    def set_host_chunk(self, utterances: int) -> None:
        """Utterances per pipeline chunk of the host-buffer entry points (0 = default: four per SM)."""
        _lib.check(self.lib.rb_ctx_set_chunk(self._host_ctx(), int(utterances)), "rb_ctx_set_chunk")

    def process_host_seeded(self, algo: int, x: np.ndarray, lengths: np.ndarray, seeds, sr, args,
                            out: Optional[np.ndarray] = None) -> np.ndarray:
        """Host waveforms in, host results out, plans drawn ON THE DEVICE from per-utterance seeds
        (``np.random.seed(seeds[u])`` before utterance u). x: [B, ld] float32, page-locked for full overlap."""
        if x.dtype != np.float32 or x.ndim != 2 or not x.flags.c_contiguous:
            raise ValueError("x must be a C-contiguous [B, ld] float32 array")
        B, ld = x.shape
        if out is None:
            out = np.zeros_like(x)
        lengths = np.ascontiguousarray(lengths, dtype=np.int32)
        seeds = np.ascontiguousarray(seeds, dtype=np.uint32)
        if lengths.shape[0] != B or seeds.shape[0] != B:
            raise ValueError("one length and one seed per utterance")
        a = _lib.args_struct(args, sr)
        rc = self.lib.rb_process_host_seeded(self._host_ctx(), int(algo), C.byref(a), C.c_void_p(x.ctypes.data),
                                             C.c_void_p(lengths.ctypes.data), C.c_void_p(seeds.ctypes.data), B, ld,
                                             C.c_void_p(out.ctypes.data))
        _lib.check(rc, f"rb_process_host_seeded(algo={algo})")
        return out

    def submit_host_seeded(self, algo: int, x: np.ndarray, lengths: np.ndarray, seeds: np.ndarray, sr, args, out: np.ndarray) -> int:
        """Streaming form of :meth:`process_host_seeded`: queue the call and return a ticket at once. Up to two calls may be in
        flight; ``x``, ``lengths``, ``seeds`` and ``out`` (contiguous, ideally page-locked, of the exact dtypes int32 / uint32 /
        float32) must stay alive and untouched until :meth:`wait_host` has returned for the ticket."""
        if x.dtype != np.float32 or x.ndim != 2 or not x.flags.c_contiguous or out.dtype != np.float32 or out.shape != x.shape:
            raise ValueError("x / out must be C-contiguous [B, ld] float32 arrays of the same shape")
        return self._submit(algo, x, _lib.RB_IO_HOST_F32, lengths, seeds, out.ctypes.data, _lib.RB_IO_HOST_F32, sr, args)

    def submit_host_ex(self, algo: int, x: np.ndarray, dtype: str, lengths: np.ndarray, seeds: np.ndarray, sr, args, out) -> int:
        """General streaming submit (``rb_submit_seeded_ex``) for host input: ``dtype`` "f32" (float32 waveforms) or "pcm16"
        (int16 samples as a wav file holds them; converted on the device as sample / 32768, which is what ``librosa.load``
        returns for 16-bit audio). ``out``: a host float32 array [B, ld] or a device tensor [B, ld] -- then the results stay on
        the device and nothing is copied back. Returns a ticket for :meth:`wait_host`; buffers must stay alive until then."""
        want = np.int16 if dtype == "pcm16" else np.float32
        if x.dtype != want or x.ndim != 2 or not x.flags.c_contiguous:
            raise ValueError(f"x must be a C-contiguous [B, ld] {np.dtype(want).name} array")
        B, ld = x.shape
        if torch.is_tensor(out):
            if out.device != self.device or out.dtype != torch.float32 or tuple(out.shape) != (B, ld) or not out.is_contiguous():
                raise ValueError("a device sink must be a contiguous [B, ld] float32 tensor on the engine's device")
            y_ptr, y_kind = out.data_ptr(), _lib.RB_IO_DEVICE_F32
        else:
            if out.dtype != np.float32 or out.shape != (B, ld) or not out.flags.c_contiguous:
                raise ValueError("out must be a C-contiguous [B, ld] float32 array")
            y_ptr, y_kind = out.ctypes.data, _lib.RB_IO_HOST_F32
        x_kind = _lib.RB_IO_HOST_PCM16 if dtype == "pcm16" else _lib.RB_IO_HOST_F32
        return self._submit(algo, x, x_kind, lengths, seeds, y_ptr, y_kind, sr, args)

    def submit_host_packed(self, algo: int, x: np.ndarray, dtype: str, offsets: np.ndarray, seeds: np.ndarray, sr, args, out) -> int:
        """Streaming submit of a ragged batch packed back to back (``rb_submit_seeded_packed``): utterance u is
        ``x[offsets[u]:offsets[u+1]]``, so the copies carry only real samples. ``x``: 1-D float32 ("f32") or int16 ("pcm16")
        host array of ``offsets[-1]`` samples; ``offsets``: int64 [B+1]; ``seeds``: uint32 [B]. ``out``: a host float32 array
        [offsets[-1]] that receives the results at the same offsets, or a device tensor [B, ld] (ld % 4 == 0, at least the
        longest utterance) whose rows receive them. Returns a ticket for :meth:`wait_host`; every buffer must stay alive and
        untouched until then, and page-locked buffers (:func:`pack_host_utterances`) keep the copies asynchronous."""
        if dtype not in ("f32", "pcm16"):
            raise ValueError('dtype must be "f32" or "pcm16"')
        want = np.int16 if dtype == "pcm16" else np.float32
        if offsets.dtype != np.int64 or offsets.ndim != 1 or offsets.shape[0] < 1 or not offsets.flags.c_contiguous:
            raise ValueError("offsets must be a contiguous int64 array [B + 1]")
        B, total = offsets.shape[0] - 1, int(offsets[-1])
        if x.dtype != want or x.shape != (total,) or not x.flags.c_contiguous:
            raise ValueError(f"x must be a contiguous 1-D {np.dtype(want).name} array of offsets[-1] = {total} samples")
        if seeds.dtype != np.uint32 or seeds.shape != (B,) or not seeds.flags.c_contiguous:
            raise ValueError("seeds must be a contiguous uint32 array, one seed per utterance")
        if torch.is_tensor(out):
            if out.device != self.device or out.dtype != torch.float32 or out.dim() != 2 or out.shape[0] != B or not out.is_contiguous():
                raise ValueError("a device sink must be a contiguous [B, ld] float32 tensor on the engine's device")
            y_ptr, y_kind, ld = out.data_ptr(), _lib.RB_IO_DEVICE_F32, int(out.shape[1])
        else:
            if out.dtype != np.float32 or out.shape != (total,) or not out.flags.c_contiguous:
                raise ValueError(f"out must be a contiguous float32 array of offsets[-1] = {total} samples")
            y_ptr, y_kind, ld = out.ctypes.data, _lib.RB_IO_HOST_F32, 0
        x_kind = _lib.RB_IO_HOST_PCM16 if dtype == "pcm16" else _lib.RB_IO_HOST_F32
        a = _lib.args_struct(args, sr)
        ticket = C.c_uint64(0)
        rc = self.lib.rb_submit_seeded_packed(self._host_ctx(), int(algo), C.byref(a), C.c_void_p(x.ctypes.data), x_kind,
                                              C.c_void_p(offsets.ctypes.data), C.c_void_p(seeds.ctypes.data), B, ld, C.c_void_p(y_ptr),
                                              y_kind, None, 0, C.byref(ticket))
        _lib.check(rc, f"rb_submit_seeded_packed(algo={algo})")
        return int(ticket.value)

    def process_host_packed(self, algo: int, x: np.ndarray, dtype: str, offsets: np.ndarray, seeds: np.ndarray, sr, args,
                            out=None):
        """Blocking form of :meth:`submit_host_packed`; ``out`` None allocates the packed host result. Returns ``out``."""
        if out is None:
            out = np.zeros(int(offsets[-1]), dtype=np.float32)
        self.wait_host(self.submit_host_packed(algo, x, dtype, offsets, seeds, sr, args, out))
        return out

    def process_device_seeded(self, algo: int, x: torch.Tensor, lengths: torch.Tensor, seeds: torch.Tensor, sr, args,
                              out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Seeded batch that already lives on the device: plans drawn on the device chunk by chunk WHILE the previous chunk is
        being filtered (the planner's latency-bound kernels run beside the FIR kernel on their own low-priority streams),
        results left on the device. Ordered after the work queued on torch's current stream, which in turn waits for the
        results: no host synchronisation. ``seeds``: int32 / uint32 device tensor (``np.random.seed(seeds[u])`` per utterance)."""
        self._check_batch(x, lengths)
        B, ld = x.shape
        if out is None:
            out = torch.zeros_like(x)
        if seeds.device != self.device or seeds.numel() != B or seeds.element_size() != 4:
            raise ValueError("seeds must be a 32-bit integer tensor [B] on the engine's device")
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            self._submit(algo, x, _lib.RB_IO_DEVICE_F32, lengths, seeds, out.data_ptr(), _lib.RB_IO_DEVICE_F32, sr, args, stream)
        return out

    def _submit(self, algo: int, x, x_kind: int, lengths, seeds, y_ptr: int, y_kind: int, sr, args, stream=None) -> int:
        """Queue one ``rb_submit_seeded_ex`` call and return its ticket. ``x``, ``lengths`` and ``seeds`` are host arrays, or
        device tensors whose call is ordered against ``stream`` (a ``cudaStream_t``). The call reads them after it returns, so
        host lengths and seeds must already have the exact dtypes: a converted copy would not live long enough."""
        if stream is None:
            if lengths.dtype != np.int32 or seeds.dtype != np.uint32 or not lengths.flags.c_contiguous or not seeds.flags.c_contiguous:
                raise ValueError("lengths must be a contiguous int32 array and seeds a contiguous uint32 array")
            xp, lp, sp = (C.c_void_p(a.ctypes.data) for a in (x, lengths, seeds))
        else:
            xp, lp, sp = (_ptr(t) for t in (x, lengths, seeds))
        B, ld = x.shape
        a = _lib.args_struct(args, sr)
        ticket = C.c_uint64(0)
        rc = self.lib.rb_submit_seeded_ex(self._host_ctx(), int(algo), C.byref(a), xp, x_kind, lp, sp, B, ld, C.c_void_p(y_ptr), y_kind,
                                          C.c_void_p(stream), int(stream is not None), C.byref(ticket))
        _lib.check(rc, f"rb_submit_seeded_ex(algo={algo})")
        return int(ticket.value)

    def wait_host(self, ticket: int = 0) -> None:
        """Block until the submitted call ``ticket`` (0: every submitted call) has delivered its results."""
        _lib.check(self.lib.rb_ctx_wait(self._host_ctx(), int(ticket)), "rb_ctx_wait")

    def trace_host(self, on: bool) -> None:
        """Record a per-chunk timeline of the following host-buffer calls (see :meth:`host_timeline`)."""
        _lib.check(self.lib.rb_ctx_trace(self._host_ctx(), int(bool(on))), "rb_ctx_trace")

    def host_timeline(self):
        """Timeline of the last traced host-buffer call: one dict per pipeline chunk, times in ms from the call's start."""
        n = self.lib.rb_ctx_timeline(self._host_ctx(), None, 0)
        if n <= 0:
            return []
        buf = (C.c_double * n)()
        self.lib.rb_ctx_timeline(self._host_ctx(), buf, n)
        keys = ("first", "count", "copy_in_ms", "plan_ms", "kernels_ms", "copy_out_ms")
        return [dict(zip(keys, buf[i:i + 6])) for i in range(0, n, 6)]

    def last_host_traffic(self):
        h2d, d2h = C.c_uint64(0), C.c_uint64(0)
        if self._ctx is not None:
            _lib.check(self.lib.rb_ctx_last_traffic(self._ctx, C.byref(h2d), C.byref(d2h)))
        return int(h2d.value), int(d2h.value)

    def close(self):
        if self._ctx is not None:
            self.lib.rb_ctx_destroy(self._ctx)
            self._ctx = None
        self._ws = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass


def pack_host_utterances(waves: Sequence[np.ndarray], dtype: str = "f32", pin: bool = True):
    """1-D utterances -> (flat host array, int64 offsets [B+1]) with utterance u at ``flat[offsets[u]:offsets[u+1]]``: the
    input of :meth:`Engine.submit_host_packed`. ``dtype`` "f32" (float32) or "pcm16" (the utterances must be int16 already).
    ``pin``: page-locked memory (needs CUDA), which keeps the pipeline's copies asynchronous."""
    if dtype not in ("f32", "pcm16"):
        raise ValueError('dtype must be "f32" or "pcm16"')
    if dtype == "pcm16" and any(np.asarray(w).dtype != np.int16 for w in waves):
        raise ValueError("pcm16 utterances must be int16 arrays")
    offsets = np.zeros(len(waves) + 1, dtype=np.int64)
    np.cumsum([int(np.asarray(w).shape[0]) for w in waves], out=offsets[1:])
    total = int(offsets[-1])
    if pin:
        flat = torch.empty(total, dtype=torch.int16 if dtype == "pcm16" else torch.float32).pin_memory().numpy()
    else:
        flat = np.empty(total, dtype=np.int16 if dtype == "pcm16" else np.float32)
    for u, w in enumerate(waves):
        flat[offsets[u]:offsets[u + 1]] = w
    return flat, offsets


def split_packed(flat: np.ndarray, offsets: np.ndarray):
    """Per-utterance views ``flat[offsets[u]:offsets[u+1]]`` of a packed result (no copies)."""
    return [flat[int(offsets[u]):int(offsets[u + 1])] for u in range(len(offsets) - 1)]


_default: dict = {}


def default_device() -> int:
    """The device every per-utterance drop-in function uses: ``RAWBOOST_B200_DEVICE`` (default 0), read in ONE place."""
    import os
    return int(os.environ.get("RAWBOOST_B200_DEVICE", "0"))


def default_engine(device: Optional[int] = None) -> Engine:
    """Process-wide engine used by the per-utterance reference-style functions in :mod:`RawBoost`, :mod:`multiview` and
    :mod:`reverb` (``device`` None = :func:`default_device`)."""
    if device is None:
        device = default_device()
    eng = _default.get(device)
    if eng is None:
        eng = _default[device] = Engine(device)
    return eng

"""Apply the drop-in's RawBoost calls of forked DataLoader workers in the process that owns the GPU.

CUDA cannot be used in a process forked after its parent initialised CUDA, and the reference's ``main.py`` initialises CUDA
before its ``DataLoader(num_workers=8)`` forks the workers. With a :class:`Broker` running in the parent (``dropin.
serve_workers``), a worker keeps every random draw -- on its own numpy stream, in the reference's order -- and sends only the
waveform and the drawn plan; the broker applies it on the GPU and sends back the float32 result.

* Transport: a ``multiprocessing.connection.Listener`` on an AF_UNIX socket in a private temporary directory (mode 0700),
  authenticated with ``multiprocessing.current_process().authkey``, which forked, spawned and forkserver children inherit.
  ``RAWBOOST_B200_BROKER`` holds ``<owner pid>:<socket path>``; a process whose pid differs from the owner's routes its calls
  here, connecting on its first call.
* One daemon thread serves every connection. Each round it takes whatever requests are pending, up to ``max_batch``, with no
  waiting for more; groups them by their key (requests of one key can share a batch) and applies each group with one call of
  the executor; then answers every requester with its own row or with the error of its group.
* The executor is a constructor argument, so the transport and the batching can be tested without a GPU.
  :class:`DeviceExecutor` is the one ``serve_workers`` uses: its own :class:`engine.Engine` (its own ``rb_ctx``), never the
  process's ``default_engine()``.
"""
from __future__ import annotations

import multiprocessing as mp
import os
import shutil
import tempfile
import threading
from multiprocessing import connection as mpc
from typing import Callable, Optional

import numpy as np

from . import _lib

ENV = "RAWBOOST_B200_BROKER"

#: strides above this take the global-memory impulse mask of the LnL -> ISD path (csrc/rb_dense.cu: kMaskSmemWords); rows of the
#: two classes are never batched together, so a batched row runs the same kernels as the same row alone
MASK_SMEM_MAX_LD = 393183


def owner() -> Optional[tuple]:
    """``(owner pid, socket path)`` from ``RAWBOOST_B200_BROKER``, or None."""
    value = os.environ.get(ENV)
    if not value:
        return None
    pid, _, address = value.partition(":")
    return int(pid), address


def routed() -> bool:
    """True in a process that must send its RawBoost calls to a broker: one is published and this is not its owner."""
    o = owner()
    return o is not None and o[0] != os.getpid()


class Broker:
    """Serve RawBoost requests of worker processes. ``execute(key, items) -> results`` applies one group: ``items`` is a list of
    ``(x, payload)`` pairs that share ``key``, the result is one array per item. An exception fails every request of the group
    and the broker keeps serving. Publishes itself in ``RAWBOOST_B200_BROKER`` (``publish``) until :meth:`close`, which also
    calls ``execute.close()`` when the executor has one."""

    def __init__(self, execute: Callable, max_batch: int = 64, publish: bool = True):
        if int(max_batch) < 1:
            raise ValueError("max_batch must be at least 1")
        self.execute, self.max_batch = execute, int(max_batch)
        self._dir = tempfile.mkdtemp(prefix="rawboost-b200-")  # mode 0700: only this user can reach the socket
        self.address = os.path.join(self._dir, "broker.sock")
        self._listener = mpc.Listener(self.address, family="AF_UNIX", authkey=bytes(mp.current_process().authkey))
        self._wake_r, self._wake_w = os.pipe()
        self._conns = []
        self._closed = False
        self._counts = {"requests": 0, "batches": 0, "utterances": 0, "errors": 0}
        self._lock = threading.Lock()
        self._published = False
        self._thread = threading.Thread(target=self._serve, name="rawboost-broker", daemon=True)
        self._thread.start()
        if publish:
            os.environ[ENV] = f"{os.getpid()}:{self.address}"
            self._published = True

    # -- public -----------------------------------------------------------------------------------------
    def stats(self) -> dict:
        """Requests received, batches (executor calls) run, utterances applied and requests that failed."""
        with self._lock:
            return dict(self._counts)

    def close(self) -> None:
        """Stop serving: the thread exits, every connection and the socket are closed, the directory is removed and
        ``RAWBOOST_B200_BROKER`` is cleared. A worker's next call then fails at once with ``RawBoostLibraryError``."""
        if self._closed:
            return
        self._closed = True
        if self._published and os.environ.get(ENV) == f"{os.getpid()}:{self.address}":
            del os.environ[ENV]
        os.write(self._wake_w, b"x")
        self._thread.join()
        os.close(self._wake_r)
        os.close(self._wake_w)
        shutil.rmtree(self._dir, ignore_errors=True)
        release = getattr(self.execute, "close", None)
        if release is not None:
            release()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- the serving thread -----------------------------------------------------------------------------
    def _serve(self):
        listen_sock = self._listener._listener._socket  # readable when a worker connects
        try:
            while True:
                ready = mpc.wait([self._wake_r, listen_sock] + self._conns)
                if self._wake_r in ready:
                    return
                if listen_sock in ready:
                    try:
                        self._conns.append(self._listener.accept())
                    except (OSError, EOFError, mp.AuthenticationError):
                        pass  # a client that failed the handshake or vanished during it
                pending = []
                for conn in list(self._conns):
                    if conn not in ready or len(pending) == self.max_batch:
                        continue  # the requests beyond max_batch stay pending for the next round
                    try:
                        msg = conn.recv()
                        if not (isinstance(msg, tuple) and len(msg) == 3):
                            raise ValueError("a request is a (key, x, payload) tuple")
                        hash(msg[0])
                    except (OSError, EOFError):
                        self._drop(conn)  # the worker exited, possibly in the middle of a request
                        continue
                    except Exception as e:
                        self._reply(conn, ("error", f"malformed request: {type(e).__name__}: {e}"))
                        continue
                    pending.append((conn, msg))
                if pending:
                    served = {id(conn) for conn, _ in pending}  # served connections go last: no worker waits behind others twice
                    self._conns = [c for c in self._conns if id(c) not in served] + [c for c in self._conns if id(c) in served]
                    self._run(pending)
        finally:
            for conn in self._conns:
                conn.close()
            self._conns = []
            self._listener.close()

    def _drop(self, conn):
        conn.close()
        self._conns = [c for c in self._conns if c is not conn]

    def _reply(self, conn, msg):
        try:
            conn.send(msg)
        except (OSError, EOFError):
            self._drop(conn)

    def _run(self, pending):
        groups = {}
        for conn, (key, x, payload) in pending:
            groups.setdefault(key, []).append((conn, x, payload))
        with self._lock:
            self._counts["requests"] += len(pending)
        for key, reqs in groups.items():
            try:
                results = self.execute(key, [(x, payload) for _, x, payload in reqs])
                if len(results) != len(reqs):
                    raise RuntimeError(f"the executor returned {len(results)} results for {len(reqs)} requests")
                replies = [("ok", r) for r in results]
                failed = 0
            except Exception as e:
                msg = str(e) if isinstance(e, _lib.RawBoostLibraryError) else f"{type(e).__name__}: {e}"
                replies = [("error", msg)] * len(reqs)
                failed = len(reqs)
            with self._lock:
                self._counts["batches"] += 1
                self._counts["utterances"] += len(reqs) - failed
                self._counts["errors"] += failed
            for (conn, _, _), reply in zip(reqs, replies):
                self._reply(conn, reply)


# -- the worker side ------------------------------------------------------------------------------------
_client = {"pid": None, "conn": None, "lock": threading.Lock()}


def request(key, x, payload):
    """Send one request to the broker and return its result. Raises ``RawBoostLibraryError`` with the broker's message when
    the request failed there, and at once when the broker is closed or cannot be reached."""
    o = owner()
    if o is None:
        raise _lib.RawBoostLibraryError(f"no RawBoost broker is published ({ENV} is not set); call dropin.serve_workers() in the "
                                        "process that owns the GPU before the DataLoader starts its workers")
    with _client["lock"]:
        if _client["pid"] != os.getpid():  # a connection inherited through fork belongs to the parent
            _client["pid"], _client["conn"] = os.getpid(), None
        try:
            if _client["conn"] is None:
                _client["conn"] = mpc.Client(o[1], family="AF_UNIX", authkey=bytes(mp.current_process().authkey))
            _client["conn"].send((key, x, payload))
            status, value = _client["conn"].recv()
        except (OSError, EOFError, mp.AuthenticationError) as e:
            if _client["conn"] is not None:
                _client["conn"].close()
            _client["conn"] = None
            raise _lib.RawBoostLibraryError(f"the RawBoost broker of process {o[0]} at {o[1]} is closed or unreachable "
                                            f"({type(e).__name__}: {e}); dropin.serve_workers() must be running in that process") from e
    if status != "ok":
        raise _lib.RawBoostLibraryError(value)
    return value


# -- the GPU executor -----------------------------------------------------------------------------------
class DeviceExecutor:
    """Apply groups of requests on the GPU with a private :class:`engine.Engine`.

    Keys (built by the routed functions of :mod:`RawBoost`): ``("rb", algo, n_f, g_sd, big)`` with a one-utterance
    :class:`plans.BatchPlan` per item -- one ``rb_process_host`` call over the group's rows, padded to its longest one;
    ``("norm", always)`` -- ``rb_normwav``; ``("fir",)`` with float32 taps per item -- ``rb_filter_fir``. The last two run on a
    private torch stream, so none of them waits for the work queued on the training's streams.

    ``rb_ctx`` grows a buffer through ``cudaDeviceSynchronize`` + ``cudaFree``, which would stall training whenever a batch
    needs more room than any before it. So the context is sized once, here: every algo runs ``max_batch`` rows of ``max_len``
    samples through every pipeline slot, with plans of 5 x 512 LnL taps, 512 SSI taps and an impulse at 10 % of the samples
    per row (the reference's defaults draw at most 5 x 501 taps and impulses at under P = 10 %). Only a batch beyond that
    grows the context again."""

    WARM_TAPS, WARM_FILTERS, WARM_IMPULSE_SHARE = 512, 5, 10

    def __init__(self, device=None, max_batch: int = 64, max_len: int = 211000):
        import torch
        from .engine import Engine, default_device
        from .plans import padded_ld
        self.eng = Engine(default_device() if device is None else device)
        self.max_batch, self.ld_max = int(max_batch), padded_ld(int(max_len))
        with torch.cuda.device(self.eng.device):
            self.stream = torch.cuda.Stream(self.eng.device)
        n = self.max_batch * self.ld_max  # page-locked staging: the host-buffer entry's copies stay asynchronous DMA
        self._pin_x = torch.empty(n, dtype=torch.float32).pin_memory().numpy()
        self._pin_y = torch.empty(n, dtype=torch.float32).pin_memory().numpy()
        self._warm_up()

    def _warm_up(self):
        from .plans import BatchPlan
        B, ld = self.max_batch, self.ld_max
        K, F, n_imp = self.WARM_TAPS, self.WARM_FILTERS, ld * self.WARM_IMPULSE_SHARE // 100
        taps = np.zeros(K, dtype=np.float32)
        taps[K // 2] = 1.0
        bp = BatchPlan(B=B, ld=ld, lengths=np.full(B, ld, dtype=np.int32), n_f=F, g_sd=2.0)
        bp.lnl_taps = np.tile(taps, B * F)
        bp.lnl_tap_off = (np.arange(B * F + 1) * K).astype(np.int32)
        bp.isd_idx = np.tile(np.arange(n_imp, dtype=np.int32) * 10, B)
        bp.isd_fr = np.full(B * n_imp, 0.5)
        bp.isd_off = (np.arange(B + 1) * n_imp).astype(np.int32)
        bp.ssi_noise = np.zeros((B, ld), dtype=np.float32)
        bp.ssi_taps = np.tile(taps, B)
        bp.ssi_tap_off = (np.arange(B + 1) * K).astype(np.int32)
        bp.ssi_snr_db = np.full(B, 20.0, dtype=np.float32)
        x = self._pin_x[:B * ld].reshape(B, ld)
        x[:] = 0.1
        for algo in range(1, 9):
            for _ in range(8):  # rb_api.cu's kSlots: a call of at most one chunk takes the next slot
                self.eng.process_host(algo, x, bp, out=self._pin_y[:B * ld].reshape(B, ld))
        self.__call__(("norm", False), [(x[0], None)])
        self.__call__(("fir",), [(x[0], taps)])

    def __call__(self, key, items):
        import torch
        kind = key[0]
        if kind == "rb":
            return self._rb(key[1], [x for x, _ in items], [p for _, p in items])
        xs = [x for x, _ in items]
        with torch.cuda.device(self.eng.device), torch.cuda.stream(self.stream):
            xd, ln = self.eng.pack_waveforms(xs)
            if kind == "norm":
                y = self.eng.normwav(xd, ln, bool(key[1]))
            elif kind == "fir":
                taps = [np.asarray(b, dtype=np.float32) for _, b in items]
                off = np.concatenate([[0], np.cumsum([t.shape[0] for t in taps])]).astype(np.int32)
                y = self.eng.filter_fir(xd, ln, torch.from_numpy(np.concatenate(taps)).to(self.eng.device),
                                        torch.from_numpy(off).to(self.eng.device))
            else:
                raise ValueError(f"unknown request kind {kind!r}")
            host = y.cpu().numpy()
        return [host[u, :x.shape[0]].copy() for u, x in enumerate(xs)]

    def _rb(self, algo, xs, parts):
        from .plans import concat, padded_ld
        B, ld = len(xs), padded_ld(max(x.shape[0] for x in xs))
        bp = concat(parts, ld)
        if B * ld <= self._pin_x.shape[0]:
            xh, yh = self._pin_x[:B * ld].reshape(B, ld), self._pin_y[:B * ld].reshape(B, ld)
        else:
            xh, yh = np.empty((B, ld), dtype=np.float32), np.empty((B, ld), dtype=np.float32)
        for u, x in enumerate(xs):
            xh[u, :x.shape[0]] = x
            xh[u, x.shape[0]:] = 0
        self.eng.process_host(algo, xh, bp, out=yh)
        return [yh[u, :x.shape[0]].copy() for u, x in enumerate(xs)]

    def close(self):
        self.eng.close()


def serve(device=None, max_batch: int = 64, max_len: int = 211000) -> Broker:
    """:class:`Broker` with a :class:`DeviceExecutor` (see ``dropin.serve_workers``)."""
    o = owner()
    if o is not None and o[0] == os.getpid():
        raise RuntimeError(f"a RawBoost broker of this process is already serving at {o[1]}; close it first")
    return Broker(DeviceExecutor(device, max_batch, max_len), max_batch)

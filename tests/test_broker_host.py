"""The broker that applies forked DataLoader workers' RawBoost calls in the parent (broker.py), without a GPU.

``Broker`` takes the function that applies a batch; these tests give it one built on the oracle's apply-plan functions (or
one that records what arrived), so the transport, the grouping, the routing of the drop-in and the error paths are checked
here, in processes forked the way a DataLoader forks its workers.
"""
import os
import struct
import threading
import time

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from conftest import stream_digest  # noqa: E402
from oracle import rawboost_oracle as orc  # noqa: E402  (checker only)
from scl_deepfake_audio_detection_b200 import _lib, broker as brk, plans  # noqa: E402

ARGS = orc.make_args()
SR = 16000
FORK = torch.multiprocessing.get_context("fork")


# -- a Dataset_for that runs oracle.dataset_item with an injectable RawBoost call -------------------------------------------
class OracleDataset(torch.utils.data.Dataset):
    """``Dataset_for.__getitem__`` as ``oracle.dataset_item`` computes it; ``rawboost(feature, sr, args, algo)`` is the
    RawBoost call the item makes (default: the oracle's own). Items are ``(idx, worker id, utt id, data, label, stream
    digest after the item)``."""

    def __init__(self, n=12, trim_length=12000, rawboost=orc.process, load_audio=orc.corpus_wave, ids=orc.CORPUS_IDS):
        self.n, self.trim_length, self.rawboost, self.load_audio, self.ids = n, trim_length, rawboost, load_audio, ids

    def __len__(self):
        return self.n

    def __getitem__(self, k):
        from unittest import mock
        idx = k % len(self.ids)
        with mock.patch.object(orc, "process", self.rawboost):  # dataset_item looks its RawBoost call up in the oracle module
            uid, data, label = orc.dataset_item(idx, self.ids, self.load_audio, ARGS, orc.CORPUS_VOCODERS, 2, self.trim_length)
        info = torch.utils.data.get_worker_info()
        return k, (info.id if info else -1), uid, data, label, stream_digest()


def worker_seed(wid):
    np.random.seed(4242 + wid)


def run_loader(dataset, workers):
    """Items of a forked DataLoader(batch_size=1, shuffle=True), in the order the loader yields them."""
    loader = torch.utils.data.DataLoader(dataset, batch_size=1, shuffle=True, num_workers=workers, multiprocessing_context=FORK,
                                         worker_init_fn=worker_seed, collate_fn=lambda b: b[0],
                                         generator=torch.Generator().manual_seed(7))
    return list(loader)


def replay(dataset, items):
    """Each worker's index sequence replayed with the oracle from the same worker_init_fn seed: {k: (data, label, digest)}."""
    out = {}
    for wid in sorted({it[1] for it in items}):
        worker_seed(wid)
        for it in items:
            if it[1] == wid:
                _, data, label = orc.dataset_item(it[0] % len(dataset.ids), dataset.ids, dataset.load_audio, ARGS,
                                                  orc.CORPUS_VOCODERS, 2, dataset.trim_length)
                out[it[0]] = (data, label, stream_digest())
    return out


def brokered_oracle_process(feature, sr, args, algo):
    """orc.process(algo 5) with its draws here and its arithmetic sent to the broker."""
    assert algo == 5
    lnl = orc.draw_lnl_plan(args.N_f, args.nBands, args.minF, args.maxF, args.minBW, args.maxBW, args.minCoeff, args.maxCoeff,
                            args.minG, args.maxG, args.minBiasLinNonLin, args.maxBiasLinNonLin, sr)
    isd = orc.draw_isd_plan(feature.shape[0], args.P)
    return brk.request(("oracle", 5), feature, (lnl, isd, args.g_sd))


def oracle_execute(key, items):
    assert key == ("oracle", 5)
    return [orc.apply_isd(orc.apply_lnl(x, lnl), isd, g_sd) for x, (lnl, isd, g_sd) in items]


class Recorder:
    """Executor that records every group and answers ``x + algo`` (float32) per row; ``fail`` algos raise; ``delay`` seconds
    on the first call let requests pile up."""

    def __init__(self, fail=(), delay=0.0):
        self.groups, self.fail, self.delay = [], set(fail), delay

    def __call__(self, key, items):
        if self.delay and not self.groups:
            time.sleep(self.delay)
        self.groups.append((key, [(x.copy(), p) for x, p in items]))
        if key[0] == "rb" and key[1] in self.fail:
            raise ValueError(f"refused algo {key[1]}")
        return [np.asarray(x, dtype=np.float32) + (key[1] if key[0] == "rb" else 0) for x, _ in items]


def forked(fn, *args):
    """Start fn(*args) in a forked child; returns a function that waits (timeout) for ``("ok", value)`` or ``("err", repr)``."""
    r, w = FORK.Pipe(duplex=False)

    def child():
        try:
            w.send(("ok", fn(*args)))
        except BaseException as e:  # noqa: BLE001 -- reported to the parent
            w.send(("err", f"{type(e).__name__}: {e}"))

    p = FORK.Process(target=child)
    p.start()

    def result(timeout=60):
        if not r.poll(timeout):
            p.kill()
            p.join()
            raise AssertionError("the child did not answer in time")
        value = r.recv()
        p.join(timeout)
        return value
    return result


# -- tests -------------------------------------------------------------------------------------------------------------------
def test_forked_loader_items_equal_the_oracle_replay():
    ds = OracleDataset(rawboost=brokered_oracle_process)
    with brk.Broker(oracle_execute, max_batch=8) as b:
        items = run_loader(ds, workers=3)
        stats = b.stats()
    assert sorted(it[0] for it in items) == list(range(ds.n))
    assert {it[1] for it in items} == {0, 1, 2}
    want = replay(ds, items)
    for k, wid, uid, data, label, digest in items:
        w_data, w_label, w_digest = want[k]
        assert data.dtype == np.float32 and np.array_equal(data, w_data), (k, wid)
        assert np.array_equal(label, w_label) and digest == w_digest, (k, wid)
    per_item = len(orc.CORPUS_VOCODERS) + 1
    assert stats["requests"] == stats["utterances"] == ds.n * per_item and stats["errors"] == 0
    assert 1 <= stats["batches"] <= stats["requests"]
    assert FORK.active_children() == []


@pytest.mark.parametrize("algo", [1, 2, 3, 4, 5, 6, 7, 8])
def test_plans_cross_the_wire_bit_for_bit(algo):
    from scl_deepfake_audio_detection_b200 import RawBoost
    from scl_deepfake_audio_detection_b200.native_planner import NativePlanner
    args = orc.make_args(P=0 if algo == 7 else 10)  # algo 7 with P = 0: an ISD plan without impulses
    x64 = np.random.RandomState(algo).standard_normal(3001) * 0.1  # float64 input, rounded to float32 on the way
    rec = Recorder()
    with brk.Broker(rec, max_batch=4):
        def child():
            np.random.seed(99 + algo)
            y = RawBoost.process_Rawboost_feature(x64, SR, args, algo)
            state = np.random.get_state()[1:]
            empty = RawBoost.process_Rawboost_feature(np.zeros(0, np.float32), SR, args, algo)  # answered without a request
            return y, empty, state
        status, value = forked(child)()
    assert status == "ok", value
    y, empty, state = value
    assert len(rec.groups) == 1
    key, [(x_got, plan)] = rec.groups[0]
    np.random.seed(99 + algo)
    want = NativePlanner(threads=1, pinned=False).draw([3001], SR, args, algo, use_global_stream=True, copy=True)
    assert np.array_equal(state[0], np.random.get_state()[1]) and state[1:] == np.random.get_state()[2:]
    assert key == ("rb", algo, want.n_f, want.g_sd, False)
    assert x_got.dtype == np.float32 and np.array_equal(x_got, x64.astype(np.float32))
    for name in ("lengths", "lnl_taps", "lnl_tap_off", "isd_off", "isd_idx", "isd_fr", "ssi_noise", "ssi_taps", "ssi_tap_off",
                 "ssi_snr_db"):
        w, g = getattr(want, name), getattr(plan, name)
        assert (w is None) == (g is None), name
        if w is not None:
            assert w.dtype == g.dtype and np.array_equal(w, g), name
    assert (plan.B, plan.ld, plan.n_f, plan.g_sd) == (want.B, want.ld, want.n_f, want.g_sd)
    if algo == 7:
        assert plan.isd_idx.size == 0
    assert np.array_equal(y, x64.astype(np.float32) + algo)
    assert empty.dtype == np.float32 and empty.shape == (0,)


def test_mixed_requests_are_grouped_and_routed_back():
    from scl_deepfake_audio_detection_b200 import RawBoost
    rec = Recorder(delay=1.0)
    jobs = [(algo, 1000 + 37 * algo + 11 * i) for i, algo in enumerate((1, 3, 5, 5, 2, 5, 8, 3))]

    def child(i, algo, n):
        x = np.random.RandomState(i).uniform(-0.5, 0.5, n).astype(np.float32)
        np.random.seed(i)
        y = RawBoost.process_Rawboost_feature(x, SR, ARGS, algo)
        f = RawBoost.filterFIR(x, np.array([0.5, 0.25]))
        m = RawBoost.normWav(x, 0)
        return bool(np.array_equal(y, x + algo)), bool(np.array_equal(f, x)), m is x

    with brk.Broker(rec, max_batch=64) as b:
        waits = [forked(child, i, algo, n) for i, (algo, n) in enumerate(jobs)]
        results = [w() for w in waits]
        stats = b.stats()
    assert all(r == ("ok", (True, True, True)) for r in results), results
    assert stats["requests"] == 3 * len(jobs) and stats["utterances"] == 3 * len(jobs) and stats["errors"] == 0
    for key, items in rec.groups:
        if key[0] == "rb":
            assert all(p.B == 1 for _, p in items)
            assert {(p.n_f, p.g_sd) for _, p in items} == {key[2:4]}
    assert max(len(items) for _, items in rec.groups) > 1, "no batch held more than one request"
    assert stats["batches"] < stats["requests"]


def test_executor_error_reaches_the_worker_and_the_broker_keeps_serving():
    from scl_deepfake_audio_detection_b200 import RawBoost
    rec = Recorder(fail={3})

    def child():
        x = np.linspace(-0.5, 0.5, 2000, dtype=np.float32)
        try:
            RawBoost.process_Rawboost_feature(x, SR, ARGS, 3)
            first = "no error"
        except _lib.RawBoostLibraryError as e:
            first = str(e)
        return first, bool(np.array_equal(RawBoost.process_Rawboost_feature(x, SR, ARGS, 5), x + 5))

    with brk.Broker(rec) as b:
        status, (msg, ok) = forked(child)()
        stats = b.stats()
    assert status == "ok" and "refused algo 3" in msg and ok
    assert stats["errors"] == 1 and stats["utterances"] == 1


def test_a_client_that_disconnects_mid_request_blocks_no_one():
    import multiprocessing as mp
    from multiprocessing import connection as mpc
    from scl_deepfake_audio_detection_b200 import RawBoost

    def half_request():  # a length header that promises more bytes than ever arrive, then the process is gone
        conn = mpc.Client(brk.owner()[1], family="AF_UNIX", authkey=bytes(mp.current_process().authkey))
        conn._send(struct.pack("!i", 1 << 20) + b"\x80\x05partial")
        os._exit(0)

    def gone_before_reply():  # a whole request, then the process exits before the answer
        conn = mpc.Client(brk.owner()[1], family="AF_UNIX", authkey=bytes(mp.current_process().authkey))
        conn.send((("norm", False), np.ones(10, np.float32), None))
        os._exit(0)

    def good():
        x = np.full(500, 0.25, np.float32)
        return bool(np.array_equal(RawBoost.process_Rawboost_feature(x, SR, ARGS, 2), x + 2))

    with brk.Broker(Recorder(delay=0.5)) as b:
        for fn in (half_request, gone_before_reply):
            p = FORK.Process(target=fn)
            p.start()
            p.join(30)
        t0 = time.monotonic()
        assert forked(good)(timeout=30) == ("ok", True)
        assert time.monotonic() - t0 < 20
        assert b._thread.is_alive()


def test_close_leaves_nothing_behind():
    from scl_deepfake_audio_detection_b200 import RawBoost
    before = {t.ident for t in threading.enumerate()}
    b = brk.Broker(Recorder())
    to_parent, from_child = FORK.Pipe(duplex=False)
    to_child_r, to_child_w = FORK.Pipe(duplex=False)

    def child():
        x = np.full(300, 0.5, np.float32)
        first = RawBoost.normWav(x, 1)
        from_child.send("called")
        to_child_r.poll(60)
        to_child_r.recv()
        t0 = time.monotonic()
        try:
            RawBoost.normWav(x, 1)
            err = "no error"
        except _lib.RawBoostLibraryError as e:
            err = str(e)
        late = "no error"
        try:  # a process that never connected finds no socket
            from scl_deepfake_audio_detection_b200 import broker as b2
            b2._client["pid"] = None
            RawBoost.normWav(x, 1)
        except _lib.RawBoostLibraryError as e:
            late = str(e)
        return bool(np.array_equal(first, x)), err, late, time.monotonic() - t0

    wait = forked(child)
    if not to_parent.poll(60):
        raise AssertionError(f"the child made no first call: {wait(timeout=5)}")
    assert to_parent.recv() == "called"
    address, directory = b.address, os.path.dirname(b.address)
    b.close()
    assert brk.ENV not in os.environ
    assert not b._thread.is_alive() and not os.path.exists(address) and not os.path.exists(directory)
    to_child_w.send("go")
    status, (first_ok, err, late, took) = wait()
    assert status == "ok" and first_ok
    assert "closed or unreachable" in err and "closed or unreachable" in late and took < 10
    assert FORK.active_children() == []
    assert {t.ident for t in threading.enumerate()} <= before
    b.close()  # a second close is harmless


def test_without_a_broker_nothing_is_routed(monkeypatch):
    monkeypatch.delenv(brk.ENV, raising=False)
    assert not brk.routed()
    with pytest.raises(_lib.RawBoostLibraryError, match="serve_workers"):
        brk.request(("norm", False), np.ones(3, np.float32), None)
    monkeypatch.setenv(brk.ENV, f"{os.getpid()}:/nonexistent")
    assert not brk.routed()  # the owner itself applies its calls


def test_concat_carries_every_field_and_relays_the_noise():
    args = orc.make_args()
    np.random.seed(5)
    parts = [plans.pack([plans.draw_for_algo(n, SR, args, 4)]) for n in (40, 1, 77)]
    whole = plans.concat(parts, ld=96)
    np.random.seed(5)
    want = plans.pack([plans.draw_for_algo(n, SR, args, 4) for n in (40, 1, 77)], ld=96)
    for name in ("lengths", "lnl_taps", "lnl_tap_off", "isd_off", "isd_idx", "isd_fr", "ssi_noise", "ssi_taps", "ssi_tap_off",
                 "ssi_snr_db"):
        assert np.array_equal(getattr(whole, name), getattr(want, name)), name
    assert (whole.B, whole.ld, whole.n_f, whole.g_sd) == (3, 96, want.n_f, want.g_sd)
    with pytest.raises(ValueError):
        plans.concat(parts, ld=48)
    with pytest.raises(ValueError):
        plans.concat([parts[0], plans.pack([plans.draw_for_algo(10, SR, orc.make_args(N_f=2), 4)])])

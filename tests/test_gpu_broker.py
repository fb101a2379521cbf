"""The drop-in inside DataLoader workers forked after CUDA was initialised, served by ``dropin.serve_workers`` on the GPU.

Items of an unmodified ``Dataset_for`` (``oracle.dataset_item`` with the drop-in as its RawBoost call) must match the oracle's
replay of each worker's index sequence; every public operator called in a forked worker must equal the same call in the
owner; a batch must equal its rows run one by one; and a brokered call must not wait for the training's queued work.
"""
import os
import threading

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import rawboost_oracle as orc  # noqa: E402  (checker only)
from test_broker_host import FORK, OracleDataset, forked, replay, run_loader  # noqa: E402

pytestmark = pytest.mark.gpu

ARGS = orc.make_args()
SR = 16000
LONG_IDS = [f"long{k}.wav" for k in range(6)]
LONG_LEN = [211000, 30011, 64600, 120001, 47999, 90000]


def long_wave(path):
    """Stand-in for librosa.load with rows up to 211 000 samples: ``<dir>/long<k>.wav`` and ``<dir>/<vocoder>_long<k>.wav``."""
    name = os.path.basename(path)
    for vi, v in enumerate(orc.CORPUS_VOCODERS):
        if name.startswith(v + "_"):
            k = LONG_IDS.index(name[len(v) + 1:])
            return orc.synth_utterance(700 + 10 * k + vi + 1, max(1, LONG_LEN[k] - 977 * (vi + 1)), bool(vi % 2))
    k = LONG_IDS.index(name)
    return orc.synth_utterance(700 + 10 * k, LONG_LEN[k], bool(k % 2))


@pytest.fixture(scope="module")
def served():
    from scl_deepfake_audio_detection_b200 import dropin
    torch.zeros(1, device="cuda")  # CUDA is initialised before the workers are forked, as in main.py
    b = dropin.serve_workers(max_batch=16, max_len=211000)
    yield b
    b.close()


def test_forked_loader_items_match_the_oracle(served):
    from scl_deepfake_audio_detection_b200 import RawBoost
    ds = OracleDataset(n=8, trim_length=64000, rawboost=RawBoost.process_Rawboost_feature, load_audio=long_wave, ids=LONG_IDS)
    before = served.stats()
    items = run_loader(ds, workers=4)
    assert sorted(it[0] for it in items) == list(range(ds.n)) and len({it[1] for it in items}) == 4
    want = replay(ds, items)
    for k, wid, uid, data, label, digest in items:
        w_data, w_label, w_digest = want[k]
        assert data.shape == w_data.shape and data.dtype == np.float32
        assert float(np.max(np.abs(data.astype(np.float64) - w_data))) <= 1e-5, (k, wid)
        assert np.array_equal(label, w_label) and digest == w_digest, (k, wid)
    after = served.stats()
    assert after["utterances"] - before["utterances"] == ds.n * (len(orc.CORPUS_VOCODERS) + 1)
    assert after["errors"] == before["errors"]


def _operators(x, loud):
    from scl_deepfake_audio_detection_b200 import RawBoost as R
    a = ARGS
    ops = [
        ("normWav quiet", lambda: R.normWav(x, 0)),
        ("normWav loud", lambda: R.normWav(loud, 0)),
        ("normWav always", lambda: R.normWav(x, 1)),
        ("filterFIR", lambda: R.filterFIR(x, np.array([0.1, -0.3, 0.5, 0.2, -0.05]))),
        ("LnL", lambda: R.LnL_convolutive_noise(x, a.N_f, a.nBands, a.minF, a.maxF, a.minBW, a.maxBW, a.minCoeff, a.maxCoeff,
                                                  a.minG, a.maxG, a.minBiasLinNonLin, a.maxBiasLinNonLin, SR)),
        ("ISD", lambda: R.ISD_additive_noise(x, a.P, a.g_sd)),
        ("SSI", lambda: R.SSI_additive_noise(x, a.SNRmin, a.SNRmax, a.nBands, a.minF, a.maxF, a.minBW, a.maxBW, a.minCoeff,
                                             a.maxCoeff, a.minG, a.maxG, SR)),
        ("RawBoost12", lambda: R.RawBoost12(x, a)),
    ]
    ops += [(f"algo {k}", (lambda k=k: R.process_Rawboost_feature(x, SR, a, k))) for k in range(9)]
    return ops


def _run_all(x, loud):
    out = []
    for i, (name, op) in enumerate(_operators(x, loud)):
        np.random.seed(31 + i)
        y = op()
        out.append((name, np.array(y), y is x or y is loud, np.random.get_state()[1:]))
    return out


def test_every_operator_in_a_forked_worker_equals_the_owner(served):
    x = orc.synth_utterance(5, 70001, False)
    loud = (2.0 * orc.synth_utterance(6, 70001, True)).astype(np.float32)
    status, got = forked(_run_all, x, loud)(timeout=300)
    assert status == "ok", got
    want = _run_all(x, loud)
    for (name, y, same, state), (_, wy, wsame, wstate) in zip(got, want):
        assert y.dtype == wy.dtype and np.array_equal(y, wy), name
        assert same == wsame, name
        assert np.array_equal(state[0], wstate[0]) and state[1:] == wstate[1:], name
    identity = {name: same for name, _, same, _ in want}
    assert identity["algo 0"] and identity["normWav quiet"] and not identity["normWav loud"]


@pytest.mark.parametrize("g_sd", [2.0, 0.5])
@pytest.mark.parametrize("algo", [1, 2, 3, 4, 5, 6, 7, 8])
def test_a_batch_equals_its_rows_one_by_one(served, algo, g_sd):
    from scl_deepfake_audio_detection_b200 import RawBoost, broker
    from scl_deepfake_audio_detection_b200.native_planner import NativePlanner
    args = orc.make_args(g_sd=g_sd)
    lengths = [1, 3, 4097, 64600, 70001, 211000]
    planner = NativePlanner(threads=1, pinned=False)
    xs = [orc.synth_utterance(40 + u, n, bool(u % 2)) for u, n in enumerate(lengths)]
    parts = [planner.draw([n], SR, args, algo, seeds=[1000 + u], copy=True) for u, n in enumerate(lengths)]
    alone = [RawBoost._run_single(algo, x, p) for x, p in zip(xs, parts)]
    key = ("rb", algo, parts[0].n_f, parts[0].g_sd, False)
    assert all(("rb", algo, p.n_f, p.g_sd, p.ld > broker.MASK_SMEM_MAX_LD) == key for p in parts)
    batched = served.execute(key, list(zip(xs, parts)))
    for u, (a, b) in enumerate(zip(alone, batched)):
        assert a.dtype == b.dtype == np.float32 and np.array_equal(a, b), (algo, g_sd, lengths[u])


def test_a_brokered_call_does_not_wait_for_the_training_stream(served):
    from scl_deepfake_audio_detection_b200 import RawBoost
    to_parent, from_child = FORK.Pipe(duplex=False)
    to_child_r, to_child_w = FORK.Pipe(duplex=False)

    def worker():
        x = orc.synth_utterance(77, 64600, False)
        RawBoost.process_Rawboost_feature(x, SR, ARGS, 5)  # warm: planner, connection
        from_child.send("warm")
        to_child_r.poll(120)
        to_child_r.recv()
        return RawBoost.process_Rawboost_feature(x, SR, ARGS, 5).shape[0]

    wait = forked(worker)
    assert to_parent.poll(120) and to_parent.recv() == "warm"
    torch.cuda.synchronize()
    torch.cuda._sleep(int(8e9))  # several seconds of work queued on torch's current stream
    pending = torch.cuda.Event()
    pending.record()
    to_child_w.send("go")
    status, n = wait(timeout=120)
    still_pending = not pending.query()
    torch.cuda.synchronize()
    assert status == "ok" and n == 64600
    assert still_pending, "the brokered call waited for the work queued on torch's current stream"


def test_nothing_is_left_behind(served):
    from scl_deepfake_audio_detection_b200 import RawBoost, broker
    ds = OracleDataset(n=4, trim_length=16000, rawboost=RawBoost.process_Rawboost_feature)
    assert len(run_loader(ds, workers=2)) == 4
    served.close()
    assert FORK.active_children() == []
    assert not any(t.name == "rawboost-broker" for t in threading.enumerate())
    assert broker.ENV not in os.environ and not os.path.exists(served.address)

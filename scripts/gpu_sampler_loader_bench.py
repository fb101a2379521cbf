"""Items/s of DeviceLoader epochs with a caller's sampler and worker_init_fn, at ASVspoof 2019 LA train's shape.

Workload as in scripts/gpu_device_loader_bench.py: ``Dataset_for`` items with RawBoost12 on three vocoded copies and the
anchor, n_add = 2, a 64 000-sample crop; 2580 bona fide utterances and three vocoded copies each, synthetic 16-bit PCM at
bench.py's ragged length mix, packed as PCM16 in device memory (building it is not timed). Every loader runs
``batch_size=1, num_workers=8`` after ``torch.manual_seed``: one warm-up epoch, then two timed epochs, each from ``iter()`` to
the end of the epoch followed by a device synchronise, with the time to the first batch; the consumer drops every batch.

Rows:
* ``default``: ``shuffle=True``, the same-run reference for profiles/r09_device_loader.json;
* ``distributed R=2`` / ``R=8``: rank 0 of ``DistributedSampler(shuffle=True)``, ``set_epoch(e)`` before each epoch -- one
  rank's epoch on one GPU;
* ``seed_worker``: the default loader with the reproducibility notes' ``worker_init_fn``, non-persistent, so that eight init
  children start at every ``iter()``; ``init_children_ms`` times those eight children alone in this process;
* with more than one GPU visible, ``ranks on N GPUs``: N processes at once, rank r on GPU r, each timing its own epochs
  (no collective).

The card's name and power limit are read in the same run.

    python scripts/gpu_sampler_loader_bench.py --out profiles/r10_sampler_loader.json
"""
import argparse
import json
import os
import random
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import torch  # noqa: E402
from torch.utils.data import DistributedSampler  # noqa: E402

from gpu_device_loader_bench import N_ADD, N_BONAFIDE, TRIM, VOCODERS, card, make_corpus  # noqa: E402
from oracle import rawboost_oracle as orc  # noqa: E402  (RawBoost arguments: main.py's defaults)

WORKERS = 8


def seed_worker(worker_id):
    """The recipe of PyTorch's reproducibility notes."""
    worker_seed = torch.initial_seed() % 2 ** 32
    np.random.seed(worker_seed)
    random.seed(worker_seed)


def build_corpus(device):
    from scl_deepfake_audio_detection_b200 import multiview
    from scl_deepfake_audio_detection_b200.engine import Engine
    ids, waves, lengths = make_corpus()
    corpus = multiview.PackedCorpus(ids, "/data", lambda p: waves[os.path.basename(p)], VOCODERS, dtype="pcm16",
                                    location="device", engine=Engine(device))
    return corpus, lengths


def run(corpus, label, epochs, ranks=None, rank=0, worker_init_fn=None):
    from scl_deepfake_audio_detection_b200 import loader
    torch.manual_seed(1234)
    np.random.seed(0)
    kw = {"shuffle": True}
    sampler = None
    if ranks is not None:
        sampler = DistributedSampler(range(corpus.N), num_replicas=ranks, rank=rank, shuffle=True, seed=1234)
        kw = {"sampler": sampler}
    dl = loader.DeviceLoader(corpus, orc.make_args(), num_additional_real=N_ADD, trim_length=TRIM, batch_size=1,
                             num_workers=WORKERS, worker_init_fn=worker_init_fn, **kw)
    dev = corpus.eng.device
    times, first = [], []
    for e in range(1 + epochs):
        if sampler is not None:
            sampler.set_epoch(e)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        n = 0
        for ids, data, label_ in dl:
            if n == 0:
                torch.cuda.current_stream(dev).synchronize()
                first.append(time.perf_counter() - t0)
            n += 1
        torch.cuda.synchronize(dev)
        if e:
            times.append(time.perf_counter() - t0)
    assert n == len(dl)
    return {"label": label, "num_workers": WORKERS, "ranks": ranks, "rank": rank if ranks else None,
            "worker_init_fn": worker_init_fn.__name__ if worker_init_fn else None, "items_per_epoch": len(dl),
            "chunk_batches": dl.chunk_batches, "epochs_timed": epochs, "epoch_s": times,
            "items_per_s": [round(len(dl) / t, 1) for t in times], "first_batch_s": [round(t, 4) for t in first[1:]]}


def init_children_ms(repeats=5):
    """Wall time of one epoch's init children alone: eight forks from this process, each seeding and running seed_worker."""
    from scl_deepfake_audio_detection_b200 import loader
    out = []
    for k in range(repeats):
        t0 = time.perf_counter()
        loader._init_states(1000 + k, WORKERS, seed_worker, loader.worker_context(WORKERS))
        out.append(round(1e3 * (time.perf_counter() - t0), 2))
    return out


def rank_process(rank, ranks, epochs, queue):
    """One data-parallel rank: its own corpus and loader on GPU ``rank``."""
    try:
        torch.cuda.set_device(rank)
        corpus, _ = build_corpus(rank)
        queue.put(run(corpus, f"rank {rank} of {ranks} processes", epochs, ranks=ranks, rank=rank))
    except Exception as exc:  # reported by the parent
        queue.put({"label": f"rank {rank}", "error": repr(exc)})


def multi_gpu(ranks, epochs):
    ctx = torch.multiprocessing.get_context("spawn")
    queue = ctx.Queue()
    procs = [ctx.Process(target=rank_process, args=(r, ranks, epochs, queue)) for r in range(ranks)]
    for p in procs:
        p.start()
    try:
        rows = [queue.get() for _ in procs]
    finally:
        for p in procs:
            p.join()
    return sorted(rows, key=lambda r: r.get("rank") or 0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_sampler_loader.json"))
    ap.add_argument("--epochs", type=int, default=2)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    corpus, lengths = build_corpus(0)
    res = {"card": card(), "gpus_visible": torch.cuda.device_count(), "host_cores": os.cpu_count(), "torch": torch.__version__,
           "workload": {"items_per_epoch": N_BONAFIDE, "vocoders": len(VOCODERS), "n_add": N_ADD, "trim": TRIM,
                        "corpus": "PackedCorpus pcm16, device", "corpus_bytes": corpus.nbytes,
                        "row_len_mean": float(lengths.mean()), "row_len_max": int(lengths.max()), "batch_size": 1,
                        "num_workers": WORKERS},
           "runs": []}
    for label, kw in (("default", {}), ("distributed R=2", {"ranks": 2}), ("distributed R=8", {"ranks": 8}),
                      ("seed_worker", {"worker_init_fn": seed_worker}), ("default again", {})):
        r = run(corpus, label, a.epochs, **kw)
        res["runs"].append(r)
        print(json.dumps(r), flush=True)
    res["init_children_ms"] = init_children_ms()
    print("init children ms", res["init_children_ms"], flush=True)
    if torch.cuda.device_count() > 1:
        del corpus
        torch.cuda.empty_cache()
        res["multi_gpu"] = multi_gpu(torch.cuda.device_count(), a.epochs)
        print(json.dumps(res["multi_gpu"]), flush=True)
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(f"wrote {a.out}")


if __name__ == "__main__":
    main()

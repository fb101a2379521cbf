"""Items/s of whole DataLoader epochs built on the device (loader.DeviceLoader) at ASVspoof 2019 LA train's shape.

Dataset: ``Dataset_for.__getitem__`` with ``augmentation_methods == ['RawBoost12']`` and ``online_aug``: RawBoost12 on three
vocoded copies and on the anchor, n_add = 2 additional bona fide utterances, one shared 64 000-sample crop, every draw on the
numpy stream of the worker that builds the item. Corpus: 2580 bona fide utterances and three vocoded copies each, synthetic
16-bit PCM at bench.py's ragged length mix (RandomState(2019) gamma(3.2, 16 000) + 20 000, clipped to [24 000, 211 000]),
packed as PCM16 in device memory (multiview.PackedCorpus); building it is not timed.

Loader: ``DeviceLoader(batch_size=1, shuffle=True, num_workers=W)`` after ``torch.manual_seed``, W in {8, 0}, at the default
``chunk_batches`` and, for W = 8, a sweep of it. Per setting: one warm-up epoch, then whole epochs timed with a host clock from
``iter()`` to the end of the epoch followed by a device synchronise; items/s, time per chunk (epoch time / chunks) and the time
to the first batch. The consumer takes each batch and drops it, so the numbers are the loader's alone. The card's name and its
power limit are read in the same run.

    python scripts/gpu_device_loader_bench.py --out profiles/r09_device_loader.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from oracle import rawboost_oracle as orc  # noqa: E402  (RawBoost arguments: main.py's defaults)

N_BONAFIDE, VOCODERS, N_ADD, TRIM = 2580, ["hifigan", "hn-sinc-nsf-hifi", "waveglow"], 2, 64000


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["unknown, unknown"])[0].split(", ")
    return {"name": name, "power_limit": power}


def make_corpus():
    ids = [f"LA_T_{k:07d}.flac" for k in range(N_BONAFIDE)]
    rows = N_BONAFIDE * (1 + len(VOCODERS))
    lengths = np.clip(np.random.RandomState(2019).gamma(3.2, 16000.0, rows) + 20000, 24000, 211000).astype(np.int64)
    rng = np.random.default_rng(11)
    waves = {}
    for r, n in enumerate(lengths):
        k, v = r % N_BONAFIDE, r // N_BONAFIDE
        name = ids[k] if v == 0 else f"{VOCODERS[v - 1]}_{ids[k]}"
        waves[name] = np.clip(3000.0 * rng.standard_normal(int(n), dtype=np.float32), -32768, 32767).astype(np.int16)
    return ids, waves, lengths


def run(corpus, workers, chunk_batches, epochs):
    from scl_deepfake_audio_detection_b200 import loader
    torch.manual_seed(1234)
    np.random.seed(0)
    kw = {} if chunk_batches is None else {"chunk_batches": chunk_batches}
    dl = loader.DeviceLoader(corpus, orc.make_args(), num_additional_real=N_ADD, trim_length=TRIM, batch_size=1, shuffle=True,
                             num_workers=workers, **kw)
    times, first = [], []
    for e in range(1 + epochs):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        n = 0
        for ids, data, label in dl:
            if n == 0:
                torch.cuda.current_stream().synchronize()
                first.append(time.perf_counter() - t0)
            n += 1
        torch.cuda.synchronize()
        if e:
            times.append(time.perf_counter() - t0)
    assert n == len(dl) == N_BONAFIDE
    chunks = -(-len(dl) // dl.chunk_batches)
    return {"num_workers": workers, "chunk_batches": dl.chunk_batches, "chunks_per_epoch": chunks, "epochs_timed": epochs,
            "epoch_s": times, "items_per_s": [round(len(dl) / t, 1) for t in times],
            "ms_per_chunk": [round(1e3 * t / chunks, 2) for t in times], "first_batch_s": [round(t, 4) for t in first[1:]]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_device_loader.json"))
    ap.add_argument("--epochs", type=int, default=2)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    from scl_deepfake_audio_detection_b200 import multiview
    ids, waves, lengths = make_corpus()
    corpus = multiview.PackedCorpus(ids, "/data", lambda p: waves[os.path.basename(p)], VOCODERS, dtype="pcm16",
                                    location="device")
    del waves
    res = {"card": card(), "host_cores": os.cpu_count(), "torch": torch.__version__,
           "workload": {"items_per_epoch": N_BONAFIDE, "vocoders": len(VOCODERS), "n_add": N_ADD, "trim": TRIM,
                        "corpus": "PackedCorpus pcm16, device", "corpus_bytes": corpus.nbytes,
                        "row_len_mean": float(lengths.mean()), "row_len_max": int(lengths.max()), "batch_size": 1, "shuffle": True},
           "runs": []}
    for workers, chunk in ((8, None), (0, None), (8, 64), (8, 1024)):
        r = run(corpus, workers, chunk, a.epochs)
        res["runs"].append(r)
        print(json.dumps(r), flush=True)
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(f"wrote {a.out}")


if __name__ == "__main__":
    main()

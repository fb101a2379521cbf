"""Items/s of a forked DataLoader over Dataset_for items: the reference's CPU RawBoost in the workers vs the brokered drop-in.

Dataset: ``Dataset_for.__getitem__`` with ``augmentation_methods == ['RawBoost12']`` (oracle.dataset_item): RawBoost12 on three
vocoded copies and on the anchor, n_add = 2 additional bona fide utterances, one shared 64 000-sample crop. Corpus: synthetic
ragged rows held in memory (no decoding: the times exclude reading audio), 96 bona fide utterances and three vocoded copies
each, at bench.py's length mix (RandomState(2019) gamma(3.2, 16 000) + 20 000, clipped to [24 000, 211 000]).

Loader: ``DataLoader(batch_size=1, shuffle=True, num_workers=W)`` forked after CUDA was initialised, W in {1, 2, 4, 8, host
cores}. Arms:
* ``reference``: the RawBoost call the workers make is the reference's own code (oracle/_ref) where it is present, else the
  numpy port (oracle.rawboost_oracle.process); which one ran is recorded. Each worker runs with one BLAS / OpenMP thread.
* ``brokered``: ``dropin.serve_workers()`` in the parent, the drop-in's ``process_Rawboost_feature`` in the workers.

Per arm and W: items/s over the timed items (at least 256, after 2 W items of warm-up), the RawBoost call latency measured in
the workers (mean, median, p90 over the timed items), and for the brokered arm the broker's mean batch size over the timed
window. A parity sample of the brokered items (each worker's first items) is checked against the oracle replay of the same
worker seeds in the same run. The card's name, its power limit and the host core count are read in the same run.

    python scripts/gpu_forked_loader_bench.py --out profiles/r08_forked_loader.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

for _k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
    os.environ.setdefault(_k, "1")

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from oracle import build_ref, rawboost_oracle as orc  # noqa: E402  (the CPU arm and the parity check)

N_BONAFIDE, VOCODERS, N_ADD, TRIM, SR = 96, ["hifigan", "hn-sinc-nsf-hifi", "waveglow"], 2, 64000, 16000
ARGS = orc.make_args()


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["unknown, unknown"])[0].split(", ")
    return {"name": name, "power_limit": power}


IDS = [f"u{k}.wav" for k in range(N_BONAFIDE)]
_lengths = np.clip(np.random.RandomState(2019).gamma(3.2, 16000.0, N_BONAFIDE * (1 + len(VOCODERS))) + 20000, 24000,
                   211000).astype(np.int64)
_rng = np.random.default_rng(11)
CORPUS = {}
for _r, _n in enumerate(_lengths):
    _k, _v = _r % N_BONAFIDE, _r // N_BONAFIDE
    _name = IDS[_k] if _v == 0 else f"{VOCODERS[_v - 1]}_{IDS[_k]}"
    CORPUS[_name] = np.clip(0.1 * _rng.standard_normal(int(_n), dtype=np.float32), -1, 1)


def load_audio(path):
    return CORPUS[os.path.basename(path)]


class Items(torch.utils.data.Dataset):
    """Dataset_for items with ``rawboost`` as the RawBoost call; each item also returns its RawBoost call times (s)."""

    def __init__(self, n, rawboost):
        self.n, self.rawboost = n, rawboost

    def __len__(self):
        return self.n

    def __getitem__(self, k):
        times = []

        def timed(feature, sr, args, algo):
            t0 = time.perf_counter()
            y = self.rawboost(feature, sr, args, algo)
            times.append(time.perf_counter() - t0)
            return y

        saved, orc.process = orc.process, timed  # dataset_item looks its RawBoost call up in the oracle module
        try:
            _, data, label = orc.dataset_item(k % N_BONAFIDE, IDS, load_audio, ARGS, VOCODERS, N_ADD, TRIM)
        finally:
            orc.process = saved
        return k, torch.utils.data.get_worker_info().id, data, times


def seed_worker(wid):
    np.random.seed(5150 + wid)


def run(arm_fn, W, broker=None):
    warm, timed = 2 * W, max(256, 4 * W)
    loader = torch.utils.data.DataLoader(Items(warm + timed, arm_fn), batch_size=1, shuffle=True, num_workers=W,
                                         multiprocessing_context="fork", worker_init_fn=seed_worker, collate_fn=lambda b: b[0],
                                         generator=torch.Generator().manual_seed(W))
    items, t0, s0 = [], None, None
    for it in loader:
        items.append(it)
        if len(items) == warm:
            t0, s0 = time.perf_counter(), (broker.stats() if broker else None)
    dt = time.perf_counter() - t0
    lat = np.array([t for it in items[warm:] for t in it[3]]) * 1e3
    rec = {"workers": W, "timed_items": timed, "items_per_s": round(timed / dt, 2), "seconds": round(dt, 3),
           "rawboost_call_ms": {"mean": round(float(lat.mean()), 3), "median": round(float(np.median(lat)), 3),
                                "p90": round(float(np.percentile(lat, 90)), 3), "calls": int(lat.size)}}
    if broker:
        s1 = broker.stats()
        rec["broker_mean_batch"] = round((s1["utterances"] - s0["utterances"]) / max(1, s1["batches"] - s0["batches"]), 3)
        rec["broker_errors"] = s1["errors"]
    return rec, items


def parity(items, per_worker=2):
    """Max |item - oracle replay| over each worker's first items (replayed from the worker seed, in the worker's order)."""
    worst, checked = 0.0, 0
    for wid in sorted({it[1] for it in items}):
        mine = [it for it in items if it[1] == wid]
        seed_worker(wid)
        for it in mine[:per_worker]:
            _, want, _ = orc.dataset_item(it[0] % N_BONAFIDE, IDS, load_audio, ARGS, VOCODERS, N_ADD, TRIM)
            worst = max(worst, float(np.max(np.abs(it[2].astype(np.float64) - want))))
            checked += 1
    return {"items": checked, "max_abs": worst, "ok": bool(worst <= 1e-5)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--workers", default=None, help="comma-separated W list (default 1,2,4,8,<host cores>)")
    opt = ap.parse_args()
    cores = os.cpu_count()
    ws = [int(w) for w in opt.workers.split(",")] if opt.workers else sorted({1, 2, 4, 8, cores})
    torch.zeros(1, device="cuda")  # CUDA first, then the loader forks (main.py:335 before main.py:379)
    from scl_deepfake_audio_detection_b200 import RawBoost, dropin
    ref = build_ref.load()
    ref_fn, ref_kind = (ref[1], "reference (oracle/_ref)") if ref is not None else (orc.process, "port (oracle.rawboost_oracle)")
    out = {"card": card(), "host_cores": cores, "torch": torch.__version__, "cpu_arm": ref_kind,
           "workload": {"bonafide": N_BONAFIDE, "vocoders": len(VOCODERS), "n_add": N_ADD, "trim": TRIM,
                        "mean_len": float(_lengths.mean()), "decoding": "excluded (rows held in memory)"},
           "reference": [], "brokered": []}
    for W in ws:
        rec, _ = run(ref_fn, W)
        out["reference"].append(rec)
        print(json.dumps({"arm": "reference", **rec}), flush=True)
    with dropin.serve_workers(max_batch=64, max_len=211000) as broker:
        for W in ws:
            rec, items = run(RawBoost.process_Rawboost_feature, W, broker)
            rec["parity"] = parity(items)
            out["brokered"].append(rec)
            print(json.dumps({"arm": "brokered", **rec}), flush=True)
        out["broker_totals"] = broker.stats()
    for r, b in zip(out["reference"], out["brokered"]):
        b["speedup_vs_reference"] = round(b["items_per_s"] / r["items_per_s"], 2)
    if opt.out:
        with open(opt.out, "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("card", "host_cores", "cpu_arm")}))


if __name__ == "__main__":
    main()

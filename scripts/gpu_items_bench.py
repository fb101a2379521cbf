"""Per-item-seeded Dataset_for items on the device (rb_items_run) at BASELINE config 4's shape, against the config-4 path.

Workload: 8192 items per step, 3 vocoders, 64 600-sample rows, a corpus of N = 2580 bona fide utterances (the ASVspoof 2019 LA
train bona fide count) and their vocoded copies, crop 64 000, model layout [G, V, 64000]. Two runs: n_add = 0 (the 8 views of
config 4) and n_add = 2 (10 views). Each reports items/s and ms/step of the whole call, and a per-phase split timed with CUDA
events on the same shapes: rb_items_draw (walk + per-utterance plans + choice + row tables), rb_process(5) on the gathered
batch and rb_multiview_assemble_ex. The gather is not a separate entry point; its share is the whole call minus those three.

In the same run: the config-4-style step (per-utterance seeds, process_device_seeded + assemble_ex: bench.bench_config4),
ItemBatcher(planner="native") at a small G as the host baseline, a parity sample against the numpy reference, and the card's
name and power limit.

    python scripts/gpu_items_bench.py --out profiles/r04_items.json
"""
import argparse
import json
import os
import subprocess
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from scl_deepfake_audio_detection_b200 import multiview, workload  # noqa: E402
from scl_deepfake_audio_detection_b200.engine import Engine  # noqa: E402

N_BONAFIDE, NVOC, LENGTH, TRIM = 2580, 3, 64600, 64000


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["unknown, unknown"])[0].split(", ")
    return {"name": name, "power_limit": power}


def timed(fn, steps, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    ev[0].record()
    for i in range(steps):
        fn()
        ev[i + 1].record()
    torch.cuda.synchronize()
    ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]
    return {"ms_mean": ev[0].elapsed_time(ev[-1]) / steps, "ms_min": min(ms), "ms_max": max(ms)}


def synthetic_corpus(dev):
    """[N*(1+nvoc), ld] rows: speech-level gaussian for even rows, loud uniform for odd ones (normWav fires), as config 4."""
    R, ld = N_BONAFIDE * (1 + NVOC), (LENGTH + 3) // 4 * 4
    gen = torch.Generator(device=dev).manual_seed(4)
    x = torch.zeros((R, ld), dtype=torch.float32, device=dev)
    x[:, :LENGTH].normal_(0, 0.1, generator=gen).clamp_(-1, 1)
    x[1::2, :LENGTH].uniform_(-0.9, 0.9, generator=gen)
    return x, torch.full((R,), LENGTH, dtype=torch.int32, device=dev)


def bench_items(eng, args, corpus, corpus_len, G, n_add, steps, orc=None):
    dev = eng.device
    rs = np.random.RandomState(40 + n_add)
    indices = torch.from_numpy(rs.randint(0, N_BONAFIDE, G).astype(np.int32)).to(dev)
    seeds = torch.from_numpy(rs.randint(0, 2 ** 32, G, dtype=np.int64).astype(np.uint32).view(np.int32)).to(dev)
    V = 2 + n_add + 2 * NVOC
    out = torch.empty((G, V, TRIM), dtype=torch.float32, device=dev)
    res = {}

    def run():
        res["r"] = eng.items_run(args, workload.SAMPLE_RATE, corpus, corpus_len, NVOC, n_add, TRIM, indices, seeds, True,
                                 multiview.LAYOUT_MODEL, out=out)

    total = timed(run, steps)
    torch.cuda.synchronize()
    rec = {"n_add": n_add, "views": V, "items_per_step": G, "rawboost_utterances_per_step": G * (NVOC + 1),
           "step_ms": total, "items_per_s": G / total["ms_mean"] * 1e3}
    if orc is not None:
        rec["parity"] = parity(eng, args, corpus, corpus_len, indices, seeds, out, n_add, orc)
    # per-phase split on the same shapes
    ld = corpus.shape[1]
    d = {}

    def draw():
        d["d"] = eng.items_draw(args, workload.SAMPLE_RATE, corpus_len, NVOC, n_add, ld, TRIM, indices, seeds)

    t_draw = timed(draw, steps)
    dd = d["d"]
    nb = G * (NVOC + 1)
    x = corpus.index_select(0, dd["src_row"].long())
    y = torch.empty((nb, ld), dtype=torch.float32, device=dev)
    t_proc = timed(lambda: eng.process(5, x[:nb], dd["row_len"][:nb], dd["plan"], out=y), steps)
    extra = nb + np.arange(G * n_add).reshape(G, n_add) if n_add else None
    rows = torch.from_numpy(multiview.item_view_rows(G, NVOC, extra).reshape(-1)).to(dev)
    label = torch.from_numpy(multiview.item_labels(NVOC, n_add)).to(dev)
    row_len = dd["row_len"]
    xy = torch.empty_like(x)
    xy[:nb] = y
    t_asm = timed(lambda: multiview.assemble_ex(eng, x, xy, rows, row_len, V, dd["start"], TRIM, True, multiview.LAYOUT_MODEL,
                                                out=out, view_label=label), steps)
    rec["phases_ms"] = {"walk_and_plan": t_draw["ms_mean"], "rawboost": t_proc["ms_mean"], "assembly": t_asm["ms_mean"],
                        "gather_derived": total["ms_mean"] - t_draw["ms_mean"] - t_proc["ms_mean"] - t_asm["ms_mean"]}
    del x, y, xy, d, dd, out, res
    torch.cuda.empty_cache()
    return rec


def parity(eng, args, corpus, corpus_len, indices, seeds, out, n_add, orc):
    """Two items (the first and the last) against np.random.seed(s); dataset_item(...) on the same corpus rows."""
    worst = 0.0
    G = indices.numel()
    ids = [f"u{k}" for k in range(N_BONAFIDE)]
    vocs = [f"v{k}" for k in range(NVOC)]
    cache = {}

    def load(path):
        name = os.path.basename(path)
        if name not in cache:
            if "_" in name:
                v, u = name.split("_")
                row = N_BONAFIDE + int(u[1:]) * NVOC + int(v[1:])
            else:
                row = int(name[1:])
            cache[name] = corpus[row, :int(corpus_len[row])].cpu().numpy()
        return cache[name]

    state = np.random.get_state()
    idx_h, seed_h = indices.cpu().numpy(), seeds.cpu().numpy().view(np.uint32)
    for g in (0, G - 1):
        np.random.seed(int(seed_h[g]))
        _, ref, _ = orc.dataset_item(int(idx_h[g]), ids, load, orc.make_args(), vocs, n_add, TRIM)
        worst = max(worst, float(np.max(np.abs(out[g].cpu().numpy().T.astype(np.float64) - ref))))
    np.random.set_state(state)
    return {"max_abs_vs_reference": worst, "items": 2, "tolerance": 1e-5, "ok": bool(worst <= 1e-5)}


def bench_host_batcher(args, G=16):
    """ItemBatcher(planner="native"): every draw on the host, in order, on the global stream (waveforms generated on load)."""
    ids = [f"u{k}" for k in range(N_BONAFIDE)]

    def load(path):
        name = os.path.basename(path)
        return workload.synth_utterance(zlib.crc32(name.encode()) % 100000, LENGTH, False)

    bat = multiview.ItemBatcher(args, ids, "/data", load, vocoders=[f"v{k}" for k in range(NVOC)], num_additional_real=2,
                                trim_length=TRIM, planner="native")
    rs = np.random.RandomState(7)
    state = np.random.get_state()
    np.random.seed(7)
    bat.items(list(rs.randint(0, N_BONAFIDE, 2)))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    bat.items(list(rs.randint(0, N_BONAFIDE, G)))
    torch.cuda.synchronize()
    s = time.perf_counter() - t0
    np.random.set_state(state)
    return {"items": G, "n_add": 2, "s": s, "items_per_s": G / s,
            "includes": "waveform synthesis on load, host plans (native planner), upload, RawBoost, assembly"}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--items", type=int, default=8192)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_items.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    import bench
    from oracle import rawboost_oracle as orc  # checker only
    eng = Engine(0)
    args = workload.default_args()
    rec = {"card": card(), "workload": {"items": a.items, "vocoders": NVOC, "row_samples": LENGTH, "corpus_bona_fide": N_BONAFIDE,
                                        "trim": TRIM, "layout": "[G, V, 64000]"}}
    corpus, corpus_len = synthetic_corpus(eng.device)
    rec["corpus_gb"] = corpus.numel() * 4 / 1e9
    rec["items"] = [bench_items(eng, args, corpus, corpus_len, a.items, n_add, a.steps, orc) for n_add in (0, 2)]
    del corpus, corpus_len
    torch.cuda.empty_cache()
    c4 = bench.bench_config4(eng, args, items=a.items, steps=a.steps, orc=orc)
    rec["config4_style"] = {k: c4[k] for k in ("ms_per_step", "step_ms_min_median_max", "items_per_s", "parity") if k in c4}
    rec["ratio_items_n_add0_over_config4"] = rec["items"][0]["step_ms"]["ms_mean"] / c4["ms_per_step"]
    rec["host_item_batcher"] = bench_host_batcher(args)
    rec["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec))


if __name__ == "__main__":
    main()

"""Dataset_for items on numpy's running stream (rb_items_stream_run, multiview.StreamItemBatcher) against the other item paths.

Workload: gpu_items_bench.py's shape -- 3 vocoders, 64 600-sample rows, a corpus of N = 2580 bona fide utterances and their
vocoded copies, crop 64 000, 2 additional bona fide utterances (10 views), model layout [G, V, 64000] -- with G items per step.
One warp walks each stream's items in series, so the step of a single stream is bound by that walk; G is therefore smaller than
gpu_items_bench.py's 8192. Runs, on the same items:
  * StreamItemBatcher, S = 1 (the num_workers=0 loader: one stream) and S = 8 (eight streams of G/8 items)
  * SeededItemBatcher (one seed per item)
  * ItemBatcher(planner="native") against StreamItemBatcher.items (S = 1) on the first --host-items of them, alternating,
    from the same numpy state: ItemBatcher makes every draw on the host, with the waveforms pre-loaded from the corpus so that
    loading does not count against it
Per run: items/s and ms/step (CUDA events, warm-ups, several timed steps); for the device runs the walk kernel's own time (a
torch.profiler pass of its own) against the rest of the step; a parity sample against oracle.dataset_item.

--parent-lib: also time rb_items_run (seeded) of this build against another build of the library at gpu_items_bench.py's
shape (8192 items, n_add = 2), alternating in the same process, and check that both give the same bits.

    python scripts/gpu_stream_items_bench.py --out profiles/r05_stream_items.json
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import torch  # noqa: E402

from gpu_items_bench import N_BONAFIDE, NVOC, TRIM, card, synthetic_corpus, timed  # noqa: E402
from scl_deepfake_audio_detection_b200 import multiview, workload  # noqa: E402
from scl_deepfake_audio_detection_b200.engine import Engine  # noqa: E402

N_ADD = 2


class Corpus:
    """The synthetic device corpus, with the host view the reference and ItemBatcher read through load_audio."""

    def __init__(self, eng):
        self.data, self.lengths = synthetic_corpus(eng.device)
        self.ids = [f"u{k}" for k in range(N_BONAFIDE)]
        self.vocoders = [f"v{k}" for k in range(NVOC)]
        self.dc = multiview.DeviceCorpus.__new__(multiview.DeviceCorpus)
        self.dc.list_ids, self.dc.vocoders, self.dc.eng = self.ids, self.vocoders, eng
        self.dc.N, self.dc.nvoc, self.dc.ld = N_BONAFIDE, NVOC, self.data.shape[1]
        self.dc.data, self.dc.lengths = self.data, self.lengths
        self.cache = {}

    def row(self, name):
        if "_" in name:
            v, u = name.split("_")
            return N_BONAFIDE + int(u[1:]) * NVOC + int(v[1:])
        return int(name[1:])

    def preload(self, rows):
        rows = sorted(set(int(r) for r in rows) - set(self.cache))
        if rows:
            host = self.data[torch.tensor(rows, device=self.data.device)].cpu().numpy()
            lens = self.lengths.cpu().numpy()
            for k, r in enumerate(rows):
                self.cache[r] = host[k, :lens[r]].copy()

    def load(self, path):
        r = self.row(os.path.basename(path))
        if r not in self.cache:
            self.preload([r])
        return self.cache[r]


def state_after_seed(seed, skip=0):
    rs = np.random.RandomState(seed)
    rs.random_sample(skip)
    return rs.get_state()


def walk_ms(fn):
    """Device time of the walk kernels in one call of fn, from a torch.profiler pass of its own."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    us = sum(getattr(e, "device_time_total", 0) for e in prof.key_averages() if "walk_kernel" in e.key)
    return us / 1e3


def parity(c, out, args, refs):
    """refs: [(row of out, start state, indices to run from it, which of them is that row)] -> worst max-abs vs the oracle."""
    from oracle import rawboost_oracle as orc  # checker only
    worst = 0.0
    saved = np.random.get_state()
    for row, st, run, k in refs:
        np.random.set_state(st)
        for j, idx in enumerate(run):
            _, ref, _ = orc.dataset_item(int(idx), c.ids, c.load, orc.make_args(), c.vocoders, N_ADD, TRIM)
            if j == k:
                worst = max(worst, float(np.max(np.abs(out[row].cpu().numpy().T.astype(np.float64) - ref))))
    np.random.set_state(saved)
    return {"max_abs_vs_reference": worst, "items": len(refs), "tolerance": 1e-5, "ok": bool(worst <= 1e-5)}


def bench_stream(c, eng, args, indices, S, steps):
    G = len(indices)
    bat = multiview.StreamItemBatcher(args, c.dc, num_additional_real=N_ADD, trim_length=TRIM)
    per = G // S
    lists = [indices[q * per:(q + 1) * per] for q in range(S - 1)] + [indices[(S - 1) * per:]]
    states = [state_after_seed(500 + q, 3 * q) for q in range(S)]
    words = np.stack([multiview._state_words(s) for s in states])
    dev = eng.device
    di = torch.from_numpy(np.concatenate(lists).astype(np.int32)).to(dev)
    doff = torch.from_numpy(np.concatenate([[0], np.cumsum([len(x) for x in lists])]).astype(np.int32)).to(dev)
    dst = torch.from_numpy(words.view(np.int32)).to(dev)
    end = torch.empty((S, 625), dtype=torch.int32, device=dev)
    V = 2 + N_ADD + 2 * NVOC
    out = torch.empty((G, V, TRIM), dtype=torch.float32, device=dev)

    def run():
        eng.items_stream_run(args, workload.SAMPLE_RATE, c.data, c.lengths, NVOC, N_ADD, TRIM, di, doff, dst, True,
                             multiview.LAYOUT_MODEL, out=out, end_state=end)

    total = timed(run, steps, warmup=1)
    ld = c.data.shape[1]
    t_draw = timed(lambda: eng.items_stream_draw(args, workload.SAMPLE_RATE, c.lengths, NVOC, N_ADD, ld, TRIM, di, doff, dst),
                   steps, warmup=1)
    walk = walk_ms(run)
    run()
    torch.cuda.synchronize()
    refs = [(0, states[0], lists[0][:2], 0), (1, states[0], lists[0][:2], 1)]
    if S > 1:
        refs.append((per, states[1], lists[1][:1], 0))
    # the same call through StreamItemBatcher.items on numpy's global stream gives the same bits (S = 1 only)
    same = None
    if S == 1:
        saved = np.random.get_state()
        np.random.set_state(states[0])
        _, d2, _, _ = bat.items(indices, layout=multiview.LAYOUT_MODEL)
        same = bool(torch.equal(d2, out))
        del d2
        np.random.set_state(saved)
    return {"run": f"StreamItemBatcher S={S}", "streams": S, "items_per_step": G, "step_ms": total,
            "items_per_s": G / total["ms_mean"] * 1e3, "walk_ms": walk, "rest_of_step_ms": total["ms_mean"] - walk,
            "walk_share_of_step": walk / total["ms_mean"], "draw_ms_walk_and_plan": t_draw["ms_mean"],
            "batcher_items_equals_engine_call": same, "parity": parity(c, out, args, refs)}


def bench_seeded(c, eng, args, indices, steps):
    G = len(indices)
    dev = eng.device
    seeds_h = (np.arange(G, dtype=np.int64) * 2654435761 + 17) % 2 ** 32
    di = torch.from_numpy(np.asarray(indices, np.int32)).to(dev)
    ds = torch.from_numpy(seeds_h.astype(np.uint32).view(np.int32)).to(dev)
    V = 2 + N_ADD + 2 * NVOC
    out = torch.empty((G, V, TRIM), dtype=torch.float32, device=dev)

    def run():
        eng.items_run(args, workload.SAMPLE_RATE, c.data, c.lengths, NVOC, N_ADD, TRIM, di, ds, True, multiview.LAYOUT_MODEL, out=out)

    total = timed(run, steps, warmup=1)
    walk = walk_ms(run)
    run()
    torch.cuda.synchronize()
    refs = [(g, np.random.RandomState(int(seeds_h[g])).get_state(), [indices[g]], 0) for g in (0, G - 1)]
    return {"run": "SeededItemBatcher", "items_per_step": G, "step_ms": total, "items_per_s": G / total["ms_mean"] * 1e3,
            "walk_ms": walk, "rest_of_step_ms": total["ms_mean"] - walk, "walk_share_of_step": walk / total["ms_mean"],
            "parity": parity(c, out, args, refs)}


def bench_host_vs_stream(c, eng, args, indices, steps):
    """ItemBatcher(planner="native") and StreamItemBatcher.items (one stream, numpy's global stream) on the same items from the
    same numpy state, alternating, `steps` timed calls each after one warm-up call each; host clock around a device synchronise
    for both. Returns the two run records and the largest difference between their outputs."""
    host = multiview.ItemBatcher(args, c.ids, "/data", c.load, vocoders=c.vocoders, num_additional_real=N_ADD, trim_length=TRIM,
                                 engine=eng, planner="native")
    stream = multiview.StreamItemBatcher(args, c.dc, num_additional_real=N_ADD, trim_length=TRIM)
    c.preload(range(N_BONAFIDE))  # every bona fide row (the additional utterances can be any of them) ...
    c.preload([N_BONAFIDE + i * NVOC + v for i in indices for v in range(NVOC)])  # ... and the items' vocoded copies
    saved = np.random.get_state()
    st = state_after_seed(500)
    times, outs = {"host": [], "stream": []}, {}
    for rep in range(steps + 1):  # rep 0 is the warm-up
        for k, bat in (("host", host), ("stream", stream)):
            np.random.set_state(st)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            _, outs[k], _, _ = bat.items(indices, layout=multiview.LAYOUT_MODEL)
            torch.cuda.synchronize()
            if rep:
                times[k].append(time.perf_counter() - t0)
    np.random.set_state(saved)
    G = len(indices)
    recs = []
    for k, name in (("host", 'ItemBatcher(planner="native")'), ("stream", "StreamItemBatcher.items, S=1")):
        t = times[k]
        recs.append({"run": name, "items": G, "s_per_call": t, "s_mean": float(np.mean(t)), "s_min": min(t), "s_max": max(t),
                     "items_per_s": G / float(np.mean(t)),
                     "parity": parity(c, outs[k], args, [(0, st, indices[:2], 0), (1, st, indices[:2], 1)])})
    recs[0]["includes"] = "host plans (native planner) and draws, upload, RawBoost, assembly; waveforms pre-loaded"
    recs[1]["includes"] = "numpy state read, device walk + plans + gather + RawBoost + assembly, end state read back and set"
    return recs, float((outs["host"] - outs["stream"]).abs().max())


def bench_parent(args, parent_lib, steps, reps=3):
    """rb_items_run of this build and of `parent_lib`, alternating, at gpu_items_bench.py's shape."""
    import ctypes as C
    from scl_deepfake_audio_detection_b200 import _lib
    new_lib, old_lib = _lib.load(), C.CDLL(parent_lib)
    for name in ("rb_items_workspace_bytes", "rb_items_run"):  # all that Engine.items_run calls
        f, g = getattr(old_lib, name), getattr(new_lib, name)
        f.restype, f.argtypes = g.restype, g.argtypes
    eng_new, eng_old = Engine(0), Engine(0)
    eng_old.lib = old_lib
    data, lengths = synthetic_corpus(eng_new.device)
    G = 8192
    rs = np.random.RandomState(42)
    di = torch.from_numpy(rs.randint(0, N_BONAFIDE, G).astype(np.int32)).cuda()
    ds = torch.from_numpy(rs.randint(0, 2 ** 32, G, dtype=np.int64).astype(np.uint32).view(np.int32)).cuda()
    V = 2 + N_ADD + 2 * NVOC
    outs = {k: torch.empty((G, V, TRIM), dtype=torch.float32, device="cuda") for k in ("new", "old")}
    res = {"new": [], "old": []}
    for _ in range(reps):
        for k, e in (("new", eng_new), ("old", eng_old)):
            t = timed(lambda: e.items_run(args, workload.SAMPLE_RATE, data, lengths, NVOC, N_ADD, TRIM, di, ds, True,
                                          multiview.LAYOUT_MODEL, out=outs[k]), steps)
            res[k].append(t["ms_mean"])
    same = bool(torch.equal(outs["new"], outs["old"]))
    del data, lengths, outs
    torch.cuda.empty_cache()
    return {"items_per_step": G, "n_add": N_ADD, "ms_per_step_this_build": res["new"], "ms_per_step_parent_build": res["old"],
            "outputs_bit_identical": same, "order": "alternating, this build first in each pair"}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--items", type=int, default=1024)
    ap.add_argument("--host-items", type=int, default=128)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_stream_items.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    eng = Engine(0)
    args = workload.default_args()
    rec = {"card": card(), "workload": {"items": a.items, "vocoders": NVOC, "row_samples": 64600, "corpus_bona_fide": N_BONAFIDE,
                                        "n_add": N_ADD, "views": 2 + N_ADD + 2 * NVOC, "trim": TRIM, "layout": "[G, V, 64000]"}}
    if a.parent_lib:
        rec["rb_items_run_vs_parent"] = bench_parent(args, a.parent_lib, 5)
        torch.cuda.empty_cache()
    c = Corpus(eng)
    indices = [int(i) for i in np.random.RandomState(44).randint(0, N_BONAFIDE, a.items)]
    rec["runs"] = [bench_stream(c, eng, args, indices, 1, a.steps), bench_stream(c, eng, args, indices, 8, a.steps),
                   bench_seeded(c, eng, args, indices, a.steps)]
    same_items, diff = bench_host_vs_stream(c, eng, args, indices[:a.host_items], a.steps)
    rec["same_items_alternating"] = same_items
    rec["same_items_max_abs_item_batcher_vs_stream"] = diff
    rec["s1_over_item_batcher_items_per_s"] = same_items[1]["items_per_s"] / same_items[0]["items_per_s"]
    rec["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec))


if __name__ == "__main__":
    main()

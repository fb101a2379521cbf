"""Per-item-seeded items (rb_items_run / rb_items_run_packed) from the five corpus storage forms, in one run.

Workload: a corpus of N = 2580 bona fide utterances (ASVspoof 2019 LA train) with 3 vocoded copies each, R = 10 320 rows whose
lengths follow bench.py's ragged mix of un-cropped utterances (RandomState(2019) gamma(3.2, 16 000) + 20 000, clipped to
[24 000, 211 000]); 16-bit PCM synthetic samples read as k / 32768, so that every form holds the same float values. Steps of
G = 1024 seeded items, n_add = 2, crop 64 000, model layout [G, 10, 64000].

Variants: padded float32 on the device (DeviceCorpus, rows padded to the longest) and PackedCorpus as float32 / PCM16, on the
device / in page-locked host memory. Per variant: corpus bytes on the device (torch.cuda.memory_allocated delta) and in
page-locked host memory; step time (CUDA events, warm-up, then the median over rounds in which the variants alternate) and
items/s; the gather kernel's device time from a torch.profiler pass of its own, and its rate over the bytes it must read (the
chunks of the rows a step uses) and write; for the host variants, a copy ceiling measured in the same run: one cudaMemcpyAsync of
the same byte count from page-locked memory. Every variant's step outputs (out, out_len, labels, end states) are compared with
the padded variant's, bit for bit. The card's name and power limit are read in the same run.

    python scripts/gpu_corpus_bench.py --out profiles/r07_packed_corpus.json
"""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from scl_deepfake_audio_detection_b200 import multiview, workload  # noqa: E402
from scl_deepfake_audio_detection_b200.engine import Engine  # noqa: E402

N_BONAFIDE, NVOC, N_ADD, TRIM, G = 2580, 3, 2, 64000, 1024
VARIANTS = [("padded_f32_device", None, None), ("packed_f32_device", "float32", "device"), ("packed_pcm16_device", "pcm16", "device"),
            ("packed_f32_host", "float32", "host"), ("packed_pcm16_host", "pcm16", "host")]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["unknown, unknown"])[0].split(", ")
    return {"name": name, "power_limit": power}


def ragged_lengths(R):
    rs = np.random.RandomState(2019)  # bench.bench_ragged's mix
    return np.clip(rs.gamma(shape=3.2, scale=16000.0, size=R) + 20000, 24000, 211000).astype(np.int32)


class SyntheticPcm:
    """Row r of the corpus (DeviceCorpus order) as float32 k / 32768, k int16 from a fixed generator."""

    def __init__(self, lengths):
        rng = np.random.default_rng(7)
        self.rows = [np.clip(np.round(rng.standard_normal(int(L), dtype=np.float32) * 3000), -32768, 32767).astype(np.int16)
                     for L in lengths]
        self.ids = [f"u{k}" for k in range(N_BONAFIDE)]
        self.vocoders = [f"v{k}" for k in range(NVOC)]

    def load(self, path):
        name = os.path.basename(path)
        if "_" in name:
            v, u = name.split("_")
            row = N_BONAFIDE + int(u[1:]) * NVOC + int(v[1:])
        else:
            row = int(name[1:])
        return self.rows[row].astype(np.float32) * np.float32(1.0 / 32768.0)


def build(eng, src, dtype, location):
    torch.cuda.synchronize()
    m0 = torch.cuda.memory_allocated(eng.device)
    if dtype is None:
        c = multiview.DeviceCorpus(src.ids, "/data", src.load, src.vocoders, engine=eng)
        host = 0
    else:
        c = multiview.PackedCorpus(src.ids, "/data", src.load, src.vocoders, dtype=dtype, location=location, engine=eng)
        host = c.nbytes if location == "host" else 0
    torch.cuda.synchronize()
    return c, {"device_bytes": torch.cuda.memory_allocated(eng.device) - m0, "pinned_host_bytes": host}


def step_fn(eng, args, c, indices, seeds, out, end):
    if isinstance(c, multiview.PackedCorpus):
        return lambda: eng.items_run_packed(args, workload.SAMPLE_RATE, c.descriptor, c.ld, NVOC, N_ADD, TRIM, indices, seeds, True,
                                            multiview.LAYOUT_MODEL, out=out, end_state=end)
    return lambda: eng.items_run(args, workload.SAMPLE_RATE, c.data, c.lengths, NVOC, N_ADD, TRIM, indices, seeds, True,
                                 multiview.LAYOUT_MODEL, out=out, end_state=end)


def timed_ms(fn, steps):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(steps):
        fn()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / steps


def gather_profile(fn, steps=3):
    """Device time per launch of the gather kernel (items_gather_kernel / items_gather_packed_kernel<...>)."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
    us, n, names = 0.0, 0, set()
    for e in prof.events():
        if "items_gather" in e.name:
            us += e.time_range.elapsed_us()
            n += 1
            names.add(re.search(r"items_gather\w*(<\w+>)?", e.name).group(0))
    return {"kernel": sorted(names), "launches": n, "ms_per_step": us / 1e3 / max(n, 1)}  # one launch per step


def copy_ceiling_ms(eng, pinned, nbytes, reps=5):
    """One cudaMemcpyAsync of nbytes from page-locked memory to the device: median ms."""
    src = pinned.view(torch.uint8)[:nbytes]
    dst = torch.empty(nbytes, dtype=torch.uint8, device=eng.device)
    dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        ms.append(timed_ms(lambda: dst.copy_(src, non_blocking=True), 1))
    del dst
    return statistics.median(ms)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--steps", type=int, default=5, help="steps per variant and round")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_packed_corpus.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    eng = Engine(0)
    args = workload.default_args()
    rec = {"card": card(), "workload": {"bona_fide": N_BONAFIDE, "vocoders": NVOC, "n_add": N_ADD, "trim": TRIM, "items_per_step": G,
                                        "layout": "[G, V, 64000]", "rows": N_BONAFIDE * (1 + NVOC),
                                        "row_lengths": "bench.py ragged mix, RandomState(2019)"}}
    lengths = ragged_lengths(N_BONAFIDE * (1 + NVOC))
    rec["workload"]["row_len_mean"] = float(lengths.mean())
    src = SyntheticPcm(lengths)
    corpora, variants = {}, {}
    for name, dtype, location in VARIANTS:
        corpora[name], variants[name] = build(eng, src, dtype, location)
    del src

    rs = np.random.RandomState(41)
    indices = torch.from_numpy(rs.randint(0, N_BONAFIDE, G).astype(np.int32)).to(eng.device)
    seeds = torch.from_numpy(rs.randint(0, 2 ** 32, G, dtype=np.int64).astype(np.uint32).view(np.int32)).to(eng.device)
    V = 2 + N_ADD + 2 * NVOC
    out = torch.empty((G, V, TRIM), dtype=torch.float32, device=eng.device)
    end = torch.empty((G, 625), dtype=torch.int32, device=eng.device)
    fns = {name: step_fn(eng, args, c, indices, seeds, out, end) for name, c in corpora.items()}

    # the rows a step gathers (the same draws for every variant) and the bytes the gather must move
    pad = corpora["padded_f32_device"]
    drawn = eng.items_draw(args, workload.SAMPLE_RATE, pad.lengths, NVOC, N_ADD, pad.ld, TRIM, indices, seeds)
    used = lengths[drawn["src_row"].cpu().numpy()].astype(np.int64)
    write_bytes = int(16 * ((used + 3) // 4).sum())
    read_bytes = {"float32": write_bytes, "pcm16": int(16 * ((used + 7) // 8).sum()), None: write_bytes}
    rec["gathered_rows_per_step"] = int(used.size)

    # outputs of one step per variant against the padded variant's
    ref = None
    for name in corpora:
        res = fns[name]()
        torch.cuda.synchronize()
        got = [t.clone() for t in res] + [end.clone()]
        if ref is None:
            ref = got
        variants[name]["bit_identical_to_padded"] = all(torch.equal(x, y) for x, y in zip(got, ref))
    del ref, got, res

    # warm-up, then rounds in which the variants alternate
    for fn in fns.values():
        for _ in range(2):
            fn()
    torch.cuda.synchronize()
    per_round = {name: [] for name in fns}
    for _ in range(a.rounds):
        for name, fn in fns.items():
            per_round[name].append(timed_ms(fn, a.steps))
    for name, (_, dtype, location) in zip(fns, VARIANTS):
        v = variants[name]
        ms = per_round[name]
        v["step_ms_median"] = statistics.median(ms)
        v["step_ms_rounds"] = ms
        v["items_per_s"] = G / v["step_ms_median"] * 1e3
        g = gather_profile(fns[name])
        rb = read_bytes[dtype]
        g["read_bytes"] = rb
        g["write_bytes"] = write_bytes
        g["read_gb_per_s"] = rb / g["ms_per_step"] / 1e6
        g["read_plus_write_gb_per_s"] = (rb + write_bytes) / g["ms_per_step"] / 1e6
        if location == "host":
            cm = copy_ceiling_ms(eng, corpora[name].samples, rb)
            g["copy_ceiling"] = {"bytes": rb, "ms": cm, "gb_per_s": rb / cm / 1e6}
            g["share_of_copy_ceiling"] = cm / g["ms_per_step"]
        v["gather"] = g
    base = variants["padded_f32_device"]["step_ms_median"]
    for v in variants.values():
        v["step_vs_padded"] = v["step_ms_median"] / base
    rec["variants"] = variants
    rec["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec))


if __name__ == "__main__":
    main()

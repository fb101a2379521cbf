"""End to end on an un-cropped ragged batch: padded host rows against utterances packed back to back (rb_submit_seeded_packed).

Workload: bench.py's ragged length mix (gamma(3.2, 16 000) + 20 000 samples, clipped to [24 000, 211 000]) at B = 4096, algo 5,
plans drawn on the device from per-utterance seeds, two calls in flight, page-locked host buffers. The samples are 16-bit PCM
values, so the float32 variants carry exactly pcm / 32768 and every variant must give the same bits. Variants:

  padded_f32            [B, ld] float32 in and out (rb_submit_seeded_ex: today's path)
  packed_f32            packed float32 in, packed float32 out
  packed_pcm16_host     packed int16 in, packed float32 out
  packed_pcm16_device   packed int16 in, device rows [B, ld] out
  uniform_padded_f32    reference point: 4096 rows of 64 600 samples, padded float32 in and out (bench.py's end-to-end line)

The variants are timed in alternation, round after round. Each reports utt/s, the bytes it moves each way and their GB/s, and
the fraction of a copy ceiling measured in the same run for the same byte counts (one whole-buffer cudaMemcpyAsync per direction
on two streams, nothing computed). Parity: every variant against the padded float32 rows, bit for bit, and four rows of the
ragged batch against the float64 oracle. The card's name and power limit are read in the same run.

    python scripts/gpu_packed_e2e_bench.py --out profiles/r06_packed_e2e.json
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

from scl_deepfake_audio_detection_b200 import workload  # noqa: E402
from scl_deepfake_audio_detection_b200.engine import Engine, pack_host_utterances, split_packed  # noqa: E402

ALGO, SR = 5, workload.SAMPLE_RATE


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["unknown, unknown"])[0].split(", ")
    return {"name": name, "power_limit": power}


def ragged_lengths(B):
    rs = np.random.RandomState(2019)  # bench.bench_ragged's mix
    return np.clip(rs.gamma(shape=3.2, scale=16000.0, size=B) + 20000, 24000, 211000).astype(np.int32)


def pinned(shape, dtype):
    return torch.empty(shape, dtype=dtype).pin_memory()


def in_flight(eng, submit, n):
    """n steps, two calls in flight, as bench.py's streaming end-to-end loop."""
    prev = None
    for k in range(n):
        t = submit(k)
        if prev is not None:
            eng.wait_host(prev)
        prev = t
    eng.wait_host(prev)


def copy_ceiling(dev, h_src, h_dst, in_bytes, out_bytes, steps):
    """Seconds per step of the same byte counts moved by two whole-buffer copies on two streams, nothing computed."""
    d_in = torch.empty(max(in_bytes, 1), dtype=torch.uint8, device=dev)
    d_out = torch.empty(max(out_bytes, 1), dtype=torch.uint8, device=dev)
    src, dst = h_src.view(-1).view(torch.uint8)[:in_bytes], h_dst.view(-1).view(torch.uint8)[:out_bytes]
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def once():
        with torch.cuda.stream(s1):
            d_in[:in_bytes].copy_(src, non_blocking=True)
        if out_bytes:
            with torch.cuda.stream(s2):
                dst.copy_(d_out[:out_bytes], non_blocking=True)

    for _ in range(2):
        once()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        once()
    s1.synchronize()
    s2.synchronize()
    return (time.perf_counter() - t0) / steps


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=5, help="timed steps per variant and round (>= 5)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_packed_e2e.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    from oracle import rawboost_oracle as orc  # checker only
    eng = Engine(0)
    dev = eng.device
    args = workload.default_args()
    B = a.batch
    lengths = ragged_lengths(B)
    ld = (int(lengths.max()) + 3) // 4 * 4
    seeds = np.array([workload.seed_for(u) for u in range(B)], dtype=np.uint32)
    rec = {"card": card(), "workload": {"batch": B, "algo": ALGO, "ld": ld, "mean_len": float(lengths.mean()),
                                        "min_len": int(lengths.min()), "max_len": int(lengths.max()),
                                        "padded_over_real_samples": B * ld / float(lengths.sum()),
                                        "in_flight": 2, "warmup_steps": a.warmup, "timed_steps_per_round": a.steps,
                                        "rounds": a.rounds}}

    # the utterances: speech-level 16-bit PCM, the float32 variants carry pcm / 32768
    rs = np.random.RandomState(64600)
    pcm_waves = [np.clip(np.round(rs.standard_normal(n) * 3000.0), -32768, 32767).astype(np.int16) for n in lengths]
    pcm, off = pack_host_utterances(pcm_waves, "pcm16")
    total = int(off[-1])
    x_pk = pinned(total, torch.float32)
    x_pk.copy_(torch.from_numpy(pcm).float() / 32768.0)
    x_pad = pinned((B, ld), torch.float32)
    x_pad.zero_()
    xp = x_pad.numpy()
    for u in range(B):
        xp[u, :lengths[u]] = x_pk.numpy()[off[u]:off[u + 1]]
    y_pad = [pinned((B, ld), torch.float32) for _ in range(2)]
    y_pk = [y.view(-1)[:total] for y in y_pad]  # the variants run one after another, so they share the output buffers
    y_dev = torch.empty((B, ld), dtype=torch.float32, device=dev)
    # uniform reference: bench.py's 64 600-sample rows
    L = workload.UTT_LEN
    x_uni = pinned((B, L), torch.float32)
    x_uni.copy_(torch.from_numpy(np.clip(np.random.RandomState(7).standard_normal((B, L)) * 0.1, -1, 1).astype(np.float32)))
    y_uni = [y.view(-1)[:B * L].view(B, L) for y in y_pad]
    len_uni = np.full(B, L, dtype=np.int32)

    variants = {
        "padded_f32": (lambda k: eng.submit_host_ex(ALGO, xp, "f32", lengths, seeds, SR, args, out=y_pad[k % 2].numpy()),
                       4 * B * ld, 4 * B * ld),
        "packed_f32": (lambda k: eng.submit_host_packed(ALGO, x_pk.numpy(), "f32", off, seeds, SR, args, out=y_pk[k % 2].numpy()),
                       4 * total, 4 * total),
        "packed_pcm16_host": (lambda k: eng.submit_host_packed(ALGO, pcm, "pcm16", off, seeds, SR, args, out=y_pk[k % 2].numpy()),
                              2 * total, 4 * total),
        "packed_pcm16_device": (lambda k: eng.submit_host_packed(ALGO, pcm, "pcm16", off, seeds, SR, args, out=y_dev),
                                2 * total, 0),
        "uniform_padded_f32": (lambda k: eng.submit_host_ex(ALGO, x_uni.numpy(), "f32", len_uni, seeds, SR, args,
                                                            out=y_uni[k % 2].numpy()), 4 * B * L, 4 * B * L),
    }
    res = {name: {"round_s_per_step": []} for name in variants}
    for name, (submit, _, _) in variants.items():  # warm-up, and the traffic the library reports
        in_flight(eng, submit, a.warmup)
        res[name]["h2d_bytes_per_step"], res[name]["d2h_bytes_per_step"] = eng.last_host_traffic()
        # parity of the warm-up results, against the padded rows (bit for bit)
        if name == "padded_f32":
            ref = [y_pad[(a.warmup - 1) % 2].numpy()[u, :lengths[u]].copy() for u in range(B)]
        elif name == "uniform_padded_f32":
            pass
        else:
            got = (split_packed(y_pk[(a.warmup - 1) % 2].numpy(), off) if name != "packed_pcm16_device" else
                   [r[:n] for r, n in zip(y_dev.cpu().numpy(), lengths)])
            res[name]["equals_padded_f32_rows"] = bool(all(np.array_equal(g, w) for g, w in zip(got, ref)))
    # four rows against the float64 oracle (the shortest, the longest and two between)
    order = np.argsort(lengths)
    worst = 0.0
    state = np.random.get_state()
    for u in (int(order[0]), int(order[B // 3]), int(order[2 * B // 3]), int(order[-1])):
        np.random.seed(int(seeds[u]))
        want = orc.process(x_pk.numpy()[off[u]:off[u + 1]].copy(), SR, orc.make_args(), ALGO)
        worst = max(worst, float(np.max(np.abs(ref[u].astype(np.float64) - want))))
    np.random.set_state(state)
    rec["parity_vs_oracle"] = {"rows": 4, "max_abs": worst, "tolerance": 1e-5, "ok": bool(worst <= 1e-5),
                               "applies_to": "every ragged variant (each equals the padded rows bit for bit where equals_padded_f32_rows)"}
    ceil = {name: [] for name in variants}
    for _ in range(a.rounds):  # the variants in alternation
        for name, (submit, in_b, out_b) in variants.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            in_flight(eng, submit, a.steps)
            res[name]["round_s_per_step"].append((time.perf_counter() - t0) / a.steps)
            ceil[name].append(copy_ceiling(dev, x_pad, y_pad[1], in_b, out_b, a.steps))
    for name, (_, in_b, out_b) in variants.items():
        r = res[name]
        s = float(np.median(r["round_s_per_step"]))
        c = float(np.median(ceil[name]))
        r.update({"ms_per_step_median": s * 1e3, "ms_per_step_rounds": [v * 1e3 for v in r.pop("round_s_per_step")],
                  "utt_per_s": B / s, "payload_bytes_in": in_b, "payload_bytes_out": out_b,
                  "gb_s_in": r["h2d_bytes_per_step"] / s / 1e9, "gb_s_out": r["d2h_bytes_per_step"] / s / 1e9,
                  "copy_ceiling": {"ms_per_step_median": c * 1e3, "utt_per_s": B / c,
                                   "gb_s_in": in_b / c / 1e9, "gb_s_out": out_b / c / 1e9},
                  "frac_of_copy_ceiling": c / s})
    rec["variants"] = res
    rec["packed_f32_over_padded_f32"] = res["packed_f32"]["utt_per_s"] / res["padded_f32"]["utt_per_s"]
    rec["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec))


if __name__ == "__main__":
    main()

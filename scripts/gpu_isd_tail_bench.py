#!/usr/bin/env python
"""Where the LnL -> ISD kernel's extra time goes: algo 1, algo 5, and algo 5 without impulses, alternated in one process.

At B = 4096 and 65536 (default arguments, 64600-sample utterances, resident in HBM) one device-drawn algo-5 plan serves three
modes, so every mode runs the same LnL taps and FLOPs:
  * algo1  -- the plan run as algo 1 (LnL only: no impulse mask, no impulses);
  * p0     -- algo 5 with every utterance's impulse list emptied (the mask launch and the mask reads stay);
  * p10    -- algo 5 as drawn (P = 10: on average P/2 % of the samples are impulses).
`rounds` rounds of `steps` timed steps per mode, the modes alternating within each round. Per mode it records the median
ms/step and its spread over the rounds and the FIR-bank kernel time (rb_profile_*); then
  mask_epilogue_ms = fir(p0) - fir(algo1)    the impulse mask and its reads in the FIR epilogue,
  impulse_tail_ms  = fir(p10) - fir(p0)      the impulse work in the fused tail (gather, peak, scatter).
The card's name, power limit and SM clocks are read by the same process.

    python scripts/gpu_isd_tail_bench.py [--rounds 3] [--steps 10] [--out profiles/r12_isd_tail.json] [--label NAME]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from scl_deepfake_audio_detection_b200 import workload  # noqa: E402
from scl_deepfake_audio_detection_b200.engine import Engine  # noqa: E402

UNIQUE = 1024  # distinct waveforms per batch (repeated beyond that; every utterance has its own seed and plan)
MODES = (("algo1", 1), ("p0", 5), ("p10", 5))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def run_mode(eng, algo, x, ln, dp, y, steps):
    eng.process(algo, x, ln, dp, out=y)  # warm-up
    torch.cuda.synchronize()
    eng.lib.rb_profile_read(None, None, 1)
    eng.lib.rb_profile_enable(1)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    ev[0].record()
    for i in range(steps):
        eng.process(algo, x, ln, dp, out=y)
        ev[i + 1].record()
    torch.cuda.synchronize()
    eng.lib.rb_profile_enable(0)
    fir_ms, fir_n = C.c_double(0.0), C.c_uint64(0)
    eng.lib.rb_profile_read(C.byref(fir_ms), C.byref(fir_n), 1)
    return ev[0].elapsed_time(ev[-1]) / steps, fir_ms.value / steps


def config(eng, B, rounds, steps):
    L = workload.UTT_LEN
    uniq = min(B, UNIQUE)
    x = torch.from_numpy(workload.synth_batch(0, uniq, L)).to(eng.device)
    if B > uniq:
        x = x.repeat((B + uniq - 1) // uniq, 1)[:B].contiguous()
    ld = int(x.shape[1])
    ln = torch.full((B,), L, dtype=torch.int32, device=eng.device)
    seeds = np.array([workload.seed_for(u) for u in range(B)], np.uint32)
    dp10 = eng.draw_device_plan(ln, seeds, workload.SAMPLE_RATE, workload.default_args(), 5, ld)
    bp = eng.download_plan(dp10)
    n_imp = np.diff(bp.isd_off)
    bp.isd_off = np.zeros_like(bp.isd_off)
    bp.isd_idx = np.zeros(0, np.int32)
    bp.isd_fr = np.zeros(0, np.float64)
    dp0 = eng.upload_plan(bp)
    plans = {"algo1": dp10, "p0": dp0, "p10": dp10}
    y = torch.empty_like(x)
    res = {name: [] for name, _ in MODES}
    for _ in range(rounds):
        for name, algo in MODES:
            res[name].append(run_mode(eng, algo, x, ln, plans[name], y, steps))
    rec = {"batch": B, "length": L, "rounds": rounds, "steps_per_round": steps,
           "impulses_per_utt_mean": float(n_imp.mean()), "impulses_per_utt_max": int(n_imp.max())}
    for name, _ in MODES:
        step = [r[0] for r in res[name]]
        fir = [r[1] for r in res[name]]
        rec[name] = {"ms_per_step_median": statistics.median(step), "ms_per_step_min_max": [min(step), max(step)],
                     "fir_ms_per_step_median": statistics.median(fir), "fir_ms_per_step_min_max": [min(fir), max(fir)],
                     "utt_per_s": B / (statistics.median(step) * 1e-3)}
    fir = {name: rec[name]["fir_ms_per_step_median"] for name, _ in MODES}
    rec["mask_epilogue_ms"] = fir["p0"] - fir["algo1"]
    rec["impulse_tail_ms"] = fir["p10"] - fir["p0"]
    rec["algo5_minus_algo1_fir_ms"] = fir["p10"] - fir["algo1"]
    print(json.dumps(rec), flush=True)
    del x, y, dp0, dp10, plans
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r12_isd_tail.json"))
    ap.add_argument("--label", default="this build", help="what the loaded library is (RAWBOOST_B200_LIB picks another one)")
    a = ap.parse_args()
    eng = Engine(0)
    out = {"gpu": card(), "torch_device": torch.cuda.get_device_name(0), "build": a.label,
           "configs": []}
    for B in (4096, 65536):
        out["configs"].append(config(eng, B, a.rounds, a.steps if B <= 4096 else max(2, a.steps // 4)))
    out["gpu_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()

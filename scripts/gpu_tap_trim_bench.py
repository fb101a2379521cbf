#!/usr/bin/env python
"""Tap trimming on against off (rb_set_tap_trim), alternated in one process on the bench workload.

For algo 5 / 1 / 3 at B = 4096 and 1024, and algo 5 at B = 65536 (default arguments, 64600-sample utterances, device plans,
resident in HBM): `rounds` rounds of `steps` timed steps with trimming on, then off. Per configuration and mode it records the
median ms/step and the spread over the rounds, the FIR-bank kernel time (rb_profile_*), and the FIR rate counted two ways --
the drawn taps (what bench.py's roofline counts) and the taps that run (rb_tap_support) -- against the FP32-pipe rate measured
here (rb_probe_fp32). The card's name and power limit are read by the same process.

    python scripts/gpu_tap_trim_bench.py [--rounds 3] [--steps 10] [--out profiles/r11_tap_trim.json]
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


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def fp32_peak(eng):
    sink = torch.zeros(4, device=eng.device)
    stream = torch.cuda.current_stream(eng.device).cuda_stream
    best, flops = 0.0, C.c_double(0.0)
    for i in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        assert eng.lib.rb_probe_fp32(1, 2000, sink.data_ptr(), C.byref(flops), C.c_void_p(stream)) == 0
        e1.record()
        e1.synchronize()
        if i:
            best = max(best, flops.value / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    return best


def fir_flops(eng, bp, L):
    """(drawn, executed) FIR FLOPs of one step: 2 * L * taps, over every LnL / SSI filter."""
    drawn = executed = 0
    for taps, off in ((bp.lnl_taps, bp.lnl_tap_off), (bp.ssi_taps, bp.ssi_tap_off)):
        if off is None:
            continue
        sup = eng.tap_support(torch.from_numpy(np.ascontiguousarray(taps)).to(eng.device),
                              torch.from_numpy(np.ascontiguousarray(off)).to(eng.device)).cpu().numpy()
        drawn += int(off[-1] - off[0])
        executed += int((sup[:, 1] - sup[:, 0]).sum())
    return 2.0 * L * drawn, 2.0 * L * executed


def run_mode(eng, algo, x, ln, dp, y, steps, trim):
    eng.set_tap_trim(trim)
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


def config(eng, algo, B, rounds, steps, peak):
    L = workload.UTT_LEN
    uniq = min(B, UNIQUE)
    host = workload.synth_batch(0, uniq, L)
    x = torch.from_numpy(host).to(eng.device)
    if B > uniq:
        x = x.repeat((B + uniq - 1) // uniq, 1)[:B].contiguous()
    ld = int(x.shape[1])
    ln = torch.full((B,), L, dtype=torch.int32, device=eng.device)
    seeds = np.array([workload.seed_for(u) for u in range(B)], np.uint32)
    dp = eng.draw_device_plan(ln, seeds, workload.SAMPLE_RATE, workload.default_args(), algo, ld)
    drawn, executed = fir_flops(eng, eng.download_plan(dp), L)
    y_on, y_off = torch.empty_like(x), torch.empty_like(x)
    res = {True: [], False: []}
    for _ in range(rounds):
        for trim in (True, False):
            res[trim].append(run_mode(eng, algo, x, ln, dp, y_on if trim else y_off, steps, trim))
    eng.set_tap_trim(True)
    torch.cuda.synchronize()
    diff = (y_on - y_off).abs()
    rec = {"algo": algo, "batch": B, "rounds": rounds, "steps_per_round": steps,
           "drawn_fir_flops_per_step": drawn, "executed_fir_flops_per_step": executed,
           "max_abs_trim_minus_full": float(diff.max()), "bit_identical_share": float((diff == 0).float().mean())}
    for trim, name in ((True, "trim_on"), (False, "trim_off")):
        step = [r[0] for r in res[trim]]
        fir = [r[1] for r in res[trim]]
        fir_med = statistics.median(fir)
        rec[name] = {"ms_per_step_median": statistics.median(step), "ms_per_step_min_max": [min(step), max(step)],
                     "fir_ms_per_step_median": fir_med, "utt_per_s": B / (statistics.median(step) * 1e-3),
                     "drawn_tap_tflops": drawn / (fir_med * 1e-3) / 1e12,
                     "executed_tap_tflops": (executed if trim else drawn) / (fir_med * 1e-3) / 1e12}
        rec[name]["executed_tap_frac_of_fp32"] = rec[name]["executed_tap_tflops"] / peak
    rec["speedup_median"] = rec["trim_off"]["ms_per_step_median"] / rec["trim_on"]["ms_per_step_median"]
    print(json.dumps(rec), flush=True)
    del x, y_on, y_off, dp
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11_tap_trim.json"))
    a = ap.parse_args()
    eng = Engine(0)
    gpu = card()
    peak = fp32_peak(eng)
    out = {"gpu": gpu, "torch_device": torch.cuda.get_device_name(0), "fp32_ffma2_tflops_measured": peak, "configs": []}
    for algo, B in ((5, 4096), (1, 4096), (3, 4096), (5, 1024), (1, 1024), (3, 1024), (5, 65536)):
        out["configs"].append(config(eng, algo, B, a.rounds, a.steps if B <= 4096 else max(2, a.steps // 4), peak))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()

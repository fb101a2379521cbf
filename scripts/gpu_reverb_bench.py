"""Reverb view: direct-form FIR path against the FFT overlap-save entry (rb_reverb), one JSON line on stdout.

For every impulse-response length K it times, with CUDA events (warm-ups, then the median of timed runs):
  direct  the device work reverb.reverb_batch launches -- rb_filter_fir over the rows delayed by (K+1)//2 and zero-extended,
          then rb_normwav(always=1) in place -- without the host packing;
  fft     Engine.reverb (rb_reverb) on the undelayed rows, output stride and longest impulse response given (asynchronous,
          no read-back).
B rows of L samples (B = 1024, L = 64600 by default: 264 MB of input, more than the 126 MB L2), one distinct impulse response
per row. Reported per K: views/s of both paths and their ratio, the direct path's TFLOP/s (2 (L + 1.5 K) K per view, what the
FIR kernel computes over the delayed row), the FFT path's algorithmic bytes (read x and the taps, write y) per second against
the data-sheet HBM bandwidth, and a parity sample (two rows) against the float64 oracle.

    python scripts/gpu_reverb_bench.py [--B 1024] [--L 64600] [--K 513,2049,8000,16000,32000] [--warmup 3] [--runs 10] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from scl_deepfake_audio_detection_b200.engine import Engine  # noqa: E402
from scl_deepfake_audio_detection_b200.plans import padded_ld  # noqa: E402
from oracle import rawboost_oracle as orc  # noqa: E402  (parity sample only)

HBM_PEAK = 7.7e12  # B/s, HGX B200 data sheet, one GPU


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
    except (OSError, subprocess.TimeoutExpired):
        info["nvidia_smi"] = None
    return info


def timed(fn, warmup, runs):
    for _ in range(warmup):
        fn()
    ms = []
    for _ in range(runs):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return float(np.median(ms)), ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=1024)
    ap.add_argument("--L", type=int, default=64600)
    ap.add_argument("--K", default="513,2049,8000,16000,32000")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--runs", type=int, default=10)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: this script measures the B200")
    eng = Engine(0)
    dev = eng.device
    B, L = a.B, a.L
    gen = torch.Generator(device=dev).manual_seed(2024)
    x = torch.zeros((B, padded_ld(L)), dtype=torch.float32, device=dev)
    x[:, :L] = 0.05 * torch.randn((B, L), generator=gen, device=dev)
    ln = torch.full((B,), L, dtype=torch.int32, device=dev)
    rows = []
    for K in [int(k) for k in a.K.split(",")]:
        decay = torch.exp(-torch.arange(K, device=dev, dtype=torch.float32) / max(1.0, K / 6.0))
        taps = (torch.randn((B, K), generator=gen, device=dev) * decay).reshape(-1).contiguous()
        off = (torch.arange(B + 1, device=dev, dtype=torch.int32) * K).contiguous()
        n_out = L + K - 1
        # direct: the rows delayed by (K+1)//2 and zero-extended, as reverb_batch stages them
        s = (K + 1) // 2
        ld_in = padded_ld(n_out + s)
        xs = torch.zeros((B, ld_in), dtype=torch.float32, device=dev)
        xs[:, s:s + L] = x[:, :L]
        ln_in = torch.full((B,), n_out + s, dtype=torch.int32, device=dev)
        yd = torch.zeros_like(xs)

        def direct():
            eng.filter_fir(xs, ln_in, taps, off, out=yd)
            eng.normwav(yd, ln_in, True, out=yd)

        yf = torch.zeros((B, padded_ld(n_out)), dtype=torch.float32, device=dev)
        out_len = None

        def fft():
            nonlocal out_len
            _, out_len = eng.reverb(x, ln, taps, off, out=yf, max_taps=K)

        d_ms, d_all = timed(direct, a.warmup, a.runs)
        f_ms, f_all = timed(fft, a.warmup, a.runs)
        torch.cuda.synchronize()
        assert int(out_len.min()) == int(out_len.max()) == n_out
        parity, cross = [], []
        h_all = taps.reshape(B, K)
        for u in (0, B - 1):
            xu = x[u, :L].cpu().numpy()
            ref = orc.reverb_convolve(xu, h_all[u].cpu().numpy())
            fu = yf[u, :n_out].cpu().numpy().astype(np.float64)
            du = yd[u, :n_out].cpu().numpy().astype(np.float64)
            parity.append(float(np.max(np.abs(fu - ref))))
            cross.append(float(np.max(np.abs(fu - du))))
        flops = 2.0 * (L + 1.5 * K) * K * B
        fft_bytes = 4.0 * (L + K + n_out) * B
        rows.append({
            "K": K, "direct_ms": round(d_ms, 4), "fft_ms": round(f_ms, 4),
            "direct_views_per_s": round(B / (d_ms * 1e-3), 1), "fft_views_per_s": round(B / (f_ms * 1e-3), 1),
            "fft_speedup": round(d_ms / f_ms, 2),
            "direct_tflops": round(flops / (d_ms * 1e-3) / 1e12, 2),
            "fft_algorithmic_gbps": round(fft_bytes / (f_ms * 1e-3) / 1e9, 1),
            "fft_share_of_hbm_peak": round(fft_bytes / (f_ms * 1e-3) / HBM_PEAK, 4),
            "fft_max_abs_err_vs_oracle": max(parity), "fft_vs_direct_max_abs": max(cross),
            "direct_ms_runs": [round(v, 4) for v in d_all], "fft_ms_runs": [round(v, 4) for v in f_all],
        })
        del xs, yd, yf, taps, off
        torch.cuda.empty_cache()
    slower = [r["K"] for r in rows if r["fft_speedup"] < 1.0]
    result = {
        "metric": "reverb_view_direct_vs_fft", "B": B, "L": L, "warmup": a.warmup, "runs": a.runs, "card": card(),
        "rows": rows,
        "direct_faster_at_K": slower,
        "hbm_peak_datasheet_Bps": HBM_PEAK,
        "note": "x is 4*B*L bytes (> L2); timing: CUDA events, median of the timed runs after the warm-ups",
    }
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

#!/usr/bin/env python3
"""RawBoost throughput benchmark: augmented utterances/sec on 64600-sample 16 kHz synthetic waveforms.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--algo 5] [--batch 4096] [--impl b200|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path (process_Rawboost_feature, fused on the device) over one batch of synthetic
utterances. Rank 0 prints ONE JSON line. ``--dump-outputs DIR`` also writes rank 0's result of the last timed step of the
headline configuration (inputs are seeded, so two builds can be compared output for output): ``DIR/y.npy`` (float32
[rows, length], every utterance of the batch or a fixed seeded sample of them, under 64 MB) and ``DIR/rows.npy`` (their batch
rows, float64).

* N = 1 (the default): BASELINE config 3 -- algo 5, 4096 utterances resident on the GPU. The same line carries, under
  ``configs``, the other configurations the metric names (algo 1 / 3 at 4096, config 2 = algo 2 and 3 at 1024, config 4 =
  the 4-view item path, config 5's one-GPU point at 65536 utterances), each with its own value, roofline fraction and an
  oracle parity sample.
* N > 1 (launched by torchrun, one rank per GPU): BASELINE config 5 -- algo 5, a GLOBAL batch of 65536 utterances sharded by
  index (strong scaling, no data-path collective); torch.distributed (NCCL) carries only the barrier and the MAX of the step time.

* ``value``   : whole-job utterances/s with inputs and the pre-drawn plan bank resident in HBM (CUDA events).
* ``e2e``     : the same metric through the host-buffer C ABI: every step copies its waveforms + seeds host->device from pinned
                memory, draws the plans on the device, runs the kernels and copies the result back; also reported as a
                fraction of what the two concurrent pinned copies alone allow on this box with N ranks (``copy_ceiling``).
* ``roofline``: the dominant kernel -- algorithmic FLOPs (bytes for the HBM-bound algo 2) of the actual drawn plans over its
                device time, against the FP32-pipe rate measured in this run / the measured HBM peak.
* ``parity``  : max-abs difference between the timed batch's results and the CPU oracle on a random sample of utterances.
* ``cpu_baseline`` (N=1) and ``--impl reference``: the reference's own CPU implementation (oracle/_ref: the reference's
                bytecode, compiled by oracle/build_ref.py; falls back to the numpy restatement), one process per host core.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import multiprocessing as mp
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "augmented utterances/sec (64600-sample, 16 kHz)"
UNIT = "utt/s"
CONFIG5_GLOBAL_BATCH = 65536
UNIQUE_WAVES = 4096      # distinct synthetic waveforms generated per rank; larger batches cycle through them (own seeds / plans)


def host_cores() -> int:
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:  # pragma: no cover
        return max(1, os.cpu_count() or 1)


# ---------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own code (oracle/_ref) or its numpy restatement, one process per core
# ---------------------------------------------------------------------------------------------------------
_CPU_CACHE = {}


def _reference_dispatch():
    """(process_Rawboost_feature, kind): the reference's own bytecode when oracle/_ref travelled here, else the oracle port."""
    from oracle import build_ref, rawboost_oracle as orc  # CPU legs: the only place bench.py executes oracle/
    ref = build_ref.load()
    if ref is not None:
        return ref[1], "reference"
    return orc.process, "port"


def _cpu_task(job):
    """Run the reference path on a fixed set of utterances; returns seconds spent inside it."""
    import warnings
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = "1"
    from oracle import rawboost_oracle as orc
    warnings.simplefilter("ignore")
    fn, _ = _reference_dispatch()
    algo, length, indices = job
    args = orc.make_args()
    key = (length, tuple(indices))
    if key not in _CPU_CACHE:
        _CPU_CACHE.clear()
        _CPU_CACHE[key] = [orc.synth_utterance(u, length, bool(u % 2)) for u in indices]
    waves = _CPU_CACHE[key]
    t0 = time.perf_counter()
    for u, x in zip(indices, waves):
        np.random.seed(orc.seed_for(u))
        fn(x, 16000, args, algo)
    return time.perf_counter() - t0


class CpuArm:
    def __init__(self, algo: int, length: int, per_core: int, cores: int):
        self.algo, self.length, self.per_core, self.cores = algo, length, per_core, cores
        for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
            os.environ.setdefault(k, "1")
        self.pool = mp.get_context("fork").Pool(cores)
        self.jobs = [(algo, length, list(range(w * per_core, (w + 1) * per_core))) for w in range(cores)]

    def step(self) -> float:
        t0 = time.perf_counter()
        self.pool.map(_cpu_task, self.jobs, chunksize=1)
        return time.perf_counter() - t0

    @property
    def utterances_per_step(self) -> int:
        return self.per_core * self.cores

    def close(self):
        self.pool.close()
        self.pool.join()


def run_cpu_arm(algo, length, per_core, cores, steps, warmup):
    arm = CpuArm(algo, length, per_core, cores)
    try:
        for _ in range(warmup):
            arm.step()
        times = [arm.step() for _ in range(steps)]
    finally:
        arm.close()
    total = sum(times)
    return arm.utterances_per_step * steps / total, 1e3 * total / steps, arm.utterances_per_step


def cpu_kind() -> str:
    return _reference_dispatch()[1]


def cpu_description(kind, n, per_core, cores, extra=""):
    from oracle import build_ref
    what = ("the reference's own datautils/RawBoost.py + process_Rawboost_feature (bytecode compiled from /root/reference by "
            "oracle/build_ref.py)" if kind == "reference" else
            f"numpy/scipy restatement of datautils/RawBoost.py (oracle port; oracle/_ref unusable here: {build_ref.last_error})")
    return (f"{n} utterances per step ({per_core} per core x {cores} cores) of the same seeded workload{extra}; {what}, "
            f"draw + apply, BLAS threads pinned to 1")


def workload_name(algo, batch, length, world=1):
    if world > 1:
        return (f"RawBoost algo={algo} (main.py:258-298 default args), global batch {batch * world} synthetic {length}-sample 16 kHz "
                f"utterances sharded over {world} GPUs (BASELINE config 5)")
    return f"RawBoost algo={algo} (main.py:258-298 default args), {batch} synthetic {length}-sample 16 kHz utterances per GPU"


def reference_arm(a):
    """--impl reference: the reference's CPU implementation of the path, all host cores, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores = host_cores()
    per_core = a.cpu_per_core
    kind = cpu_kind()
    value, ms, n = run_cpu_arm(a.algo, a.length, per_core, cores, a.steps, a.warmup)
    batch = a.batch if world == 1 else CONFIG5_GLOBAL_BATCH // world
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak" if world == 1 else "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": workload_name(a.algo, batch, a.length, world), "algo": a.algo, "utt_len": a.length, "sample_per_step": n},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": cpu_description(kind, n, per_core, cores)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ---------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi sampling of SM clocks and throttle reasons during the timed region."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.proc = None
        self.gpu_index = gpu_index
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
        self.first = None
        if self.proc is not None:  # nvidia-smi needs a few hundred ms to start: do not let a short timed region slip past it
            import select
            if select.select([self.proc.stdout], [], [], 3.0)[0]:
                self.first = self.proc.stdout.readline()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        lines = out.strip().splitlines()  # (the sample taken before the load started is not part of the record)
        for line in lines:
            f = [c.strip() for c in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "power_w_max": max(power), "samples": len(sm),
                "reasons": sorted(reasons)}


def build_id() -> str:
    """Digest of the kernel sources this library was built from (what profiles/traffic.json entries are keyed by)."""
    h = hashlib.sha1()
    base = os.path.join(ROOT, "scl-deepfake-audio-detection_b200", "csrc")
    for name in sorted(os.listdir(base)):
        if name.endswith((".cu", ".cuh", ".cpp", ".sh", ".py")):  # build.sh carries the compile flags, sass_reuse_patch.py the post-link step
            with open(os.path.join(base, name), "rb") as f:
                h.update(name.encode() + b"\0" + f.read())
    with open(os.path.join(ROOT, "include", "rawboost_b200.h"), "rb") as f:
        h.update(f.read())
    return h.hexdigest()[:12]


def traffic_for(kernel, algo, batch):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the dominant kernel from the committed
    ``ncu --set full`` capture of the same configuration AND the same build (profiles/traffic.json is keyed by the digest of
    the kernel sources), or None when this build has not been captured."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(path):
        return None
    with open(path) as f:
        table = json.load(f)
    return table.get(build_id(), {}).get(f"{kernel}:algo{algo}:b{batch}")


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def _synth_rows(job):
    from scl_deepfake_audio_detection_b200 import workload
    first, count, length, ld = job
    return workload.synth_batch(first, count, length, ld)


class Bench:
    """Everything one rank needs: engine, pools, synthetic inputs, timing helpers."""

    def __init__(self, a):
        from scl_deepfake_audio_detection_b200 import sharding, workload
        self.a = a
        self.sharding, self.workload = sharding, workload
        self.rank, self.local_rank, self.world = sharding.env_rank_world()
        self.cores = host_cores()
        self.workers = max(1, self.cores // max(1, self.world))
        # forked BEFORE CUDA is initialised; the workers only run numpy (waveform synthesis, numpy planner cross-check)
        self.pool = mp.get_context("fork").Pool(self.workers)
        import torch
        from scl_deepfake_audio_detection_b200.engine import Engine
        self.torch = torch
        torch.cuda.set_device(self.local_rank)
        if self.world > 1:
            sharding.init_process_group("nccl")
        self.dev = torch.device("cuda", self.local_rank)
        self.eng = Engine(self.local_rank)
        self.lib = self.eng.lib
        self.args = workload.default_args()
        self.hbm_peak, self.hbm_src = measured_peaks()
        self._unique = {}
        self._fp32 = None
        from oracle import rawboost_oracle as orc  # the checker of the in-run parity samples
        self.orc = orc

    # ---- inputs -------------------------------------------------------------------------------------------------------
    def unique_host(self, first, count, length, ld):
        """[count, ld] float32 host rows of utterances first .. first+count-1, synthesised in parallel (SURVEY.md 8d)."""
        key = (first, count, length, ld)
        if key not in self._unique:
            step = max(1, (count + 4 * self.workers - 1) // (4 * self.workers))
            jobs = [(first + i, min(step, count - i), length, ld) for i in range(0, count, step)]
            self._unique = {key: np.concatenate(self.pool.map(_synth_rows, jobs), axis=0)}
        return self._unique[key]

    def device_batch(self, lo, B, length, ld):
        """Utterance u of the batch carries waveform (lo + (u mod UNIQUE_WAVES)); its seed / plan is its own."""
        uniq = min(B, UNIQUE_WAVES)
        host = self.unique_host(lo, uniq, length, ld)
        x = self.torch.from_numpy(host).to(self.dev)
        if B > uniq:
            x = x.repeat((B + uniq - 1) // uniq, 1)[:B].contiguous()
        return x

    def wave_of(self, lo, u, length):
        return self.workload.synth_utterance(lo + (u % UNIQUE_WAVES), length, bool((lo + (u % UNIQUE_WAVES)) % 2))

    # ---- roofline denominators -------------------------------------------------------------------------------------------
    def fp32_peak(self):
        """FP32-pipe rate of this GPU measured here by a register-resident FFMA2 / FFMA chain."""
        if self._fp32 is None:
            import ctypes as C
            torch = self.torch
            sink = torch.zeros(4, device=self.dev)
            stream = torch.cuda.current_stream(self.dev).cuda_stream

            def probe(packed):
                best, flops = 0.0, C.c_double(0.0)
                for i in range(4):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    rc = self.lib.rb_probe_fp32(packed, 2000, sink.data_ptr(), C.byref(flops), C.c_void_p(stream))
                    e1.record()
                    e1.synchronize()
                    assert rc == 0, rc
                    if i:
                        best = max(best, flops.value / (e0.elapsed_time(e1) * 1e-3) / 1e12)
                return best

            self._fp32 = (probe(1), probe(0))
        return self._fp32

    # ---- one device-resident configuration --------------------------------------------------------------------------------
    def resident(self, algo, B, length, steps, warmup, lo=0, planner="device", parity_n=8, clocks=False, keep=False):
        """Time `steps` passes of `algo` over B resident utterances (global indices lo ..). Returns a record; with keep=True also
        the tensors (x, lengths, device plan, y, host plan) for the legs that follow."""
        import ctypes as C
        torch, eng, lib, workload = self.torch, self.eng, self.lib, self.workload
        ld = (length + 3) // 4 * 4
        seeds = np.array([workload.seed_for(u) for u in range(lo, lo + B)], dtype=np.uint32)
        x = self.device_batch(lo, B, length, ld)
        ln = torch.full((B,), length, dtype=torch.int32, device=self.dev)
        t0 = time.perf_counter()
        bp = None
        if planner == "native":
            from scl_deepfake_audio_detection_b200.native_planner import NativePlanner
            self._native = getattr(self, "_native", None) or NativePlanner(threads=self.workers, pinned=False)
            bp = self._native.draw([length] * B, workload.SAMPLE_RATE, self.args, algo, seeds=seeds, ld=ld, copy=True)
            dp = eng.upload_plan(bp)
        else:
            dp = eng.draw_device_plan(ln, seeds, workload.SAMPLE_RATE, self.args, algo, ld)
            torch.cuda.synchronize()
        t_plan = time.perf_counter() - t0
        flops, nbytes = self.plan_work(dp, bp, algo, B, length)
        y = torch.zeros_like(x)
        # the sampler covers warm-up and timed steps alike (the GPU is under the same load in both); when the timed region is
        # shorter than nvidia-smi's 100 ms period, extra untimed steps run first so that several samples fall under load
        sampler = ClockSampler(self.local_rank) if (clocks and self.rank == 0) else None
        t_w = time.perf_counter()
        for _ in range(warmup):
            eng.process(algo, x, ln, dp, out=y)
        torch.cuda.synchronize()
        while clocks and time.perf_counter() - t_w < 0.6:
            eng.process(algo, x, ln, dp, out=y)
            torch.cuda.synchronize()
        lib.rb_profile_read(None, None, 1)
        lib.rb_profile_enable(1)
        self.sharding.barrier()
        torch.cuda.synchronize()
        launches0 = lib.rb_launch_count()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        ev[0].record()
        for i in range(steps):
            eng.process(algo, x, ln, dp, out=y)
            ev[i + 1].record()
        torch.cuda.synchronize()
        self.sharding.barrier()
        total_ms = ev[0].elapsed_time(ev[-1])
        step_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]
        launches = int(lib.rb_launch_count() - launches0)
        clk = sampler.stop() if sampler else None
        lib.rb_profile_enable(0)
        fir_ms, fir_n = C.c_double(0.0), C.c_uint64(0)
        lib.rb_profile_read(C.byref(fir_ms), C.byref(fir_n), 1)
        ms = self.sharding.max_over_ranks(total_ms / steps, self.dev)
        rec = {"algo": algo, "batch_per_gpu": B, "value": self.world * B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps,
               "step_ms_min_median_max": [min(step_ms), statistics.median(step_ms), max(step_ms)], "gpu_launches": launches,
               "plan_bank": f"{planner} planner, resident before timing ({t_plan:.2f} s)"}
        step_s = ms * 1e-3
        step_hbm = {"bound": "hbm", "achieved": nbytes / step_s / 1e9, "peak": self.hbm_peak, "unit": "GB/s",
                    "frac": nbytes / step_s / 1e9 / self.hbm_peak, "peak_source": self.hbm_src, "algorithmic_bytes_per_step": nbytes}
        if fir_n.value:  # FP32-pipe bound: the FIR-bank kernel (with its fused per-utterance tail) is the step
            ffma2, ffma = self.fp32_peak()
            peak = max(ffma2, ffma)
            fir_avg_ms = fir_ms.value / fir_n.value
            per_step = fir_n.value / steps
            tf = flops / (fir_avg_ms * per_step * 1e-3) / 1e12
            rec["roofline"] = {
                "bound": "fp32", "kernel": "fir_bank_kernel", "achieved": tf, "peak": peak, "unit": "TFLOP/s", "frac": tf / peak,
                "traffic": traffic_for("fir_bank_kernel", algo, B),
                "peak_source": "FFMA2 register-resident chain measured in this run (rb_probe_fp32; multiplier in a uniform register, "
                               "two register-file operands per FFMA2: 99 %% of SMs x 128 lanes x 2 x clock -- the round-1 probe with "
                               "three register operands measured 2 %% less); scalar FFMA chain gave %.1f; "
                               "MEASURED_PEAKS.json carries HBM and bf16-tensor peaks only and north_star puts this path on the "
                               "non-tensor FP32 pipe" % ffma,
                "kernel_ms_per_launch": fir_avg_ms, "kernel_launches_per_step": per_step,
                "kernel_share_of_step": (fir_avg_ms * per_step) / (total_ms / steps),
                "algorithmic_flops_per_step": flops, "step_hbm": step_hbm}
        else:            # HBM bound (algo 2): one streaming kernel per step, algorithmic bytes over the step time
            rec["roofline"] = dict(step_hbm, kernel="norm_stream_kernel", traffic=traffic_for("norm_stream_kernel", algo, B),
                                   kernel_ms_per_launch=total_ms / steps, kernel_launches_per_step=1.0)
        if parity_n:
            rec["parity"] = self.parity_sample(algo, y, lo, B, length, parity_n, seeds)
        if clk is not None:
            rec["clocks"] = clk
        if keep:
            return rec, (x, ln, dp, y, bp, seeds, ld)
        del x, y, dp
        torch.cuda.empty_cache()
        return rec

    def plan_work(self, dp, bp, algo, B, length):
        """Algorithmic FLOPs (sum of 2*L*K over the actual drawn taps) and HBM bytes (8L [+4L noise] + 12 n) of one step."""
        import ctypes as C
        torch = self.torch
        if bp is not None:
            return bp.fir_flops(), bp.io_bytes()
        s = dp.struct
        store = dp.tensors["storage"]

        def last(ptr, index):  # one int32 of a CSR offset array that lives in the plan storage
            off = int(ptr) - store.data_ptr() + 4 * index
            return int(store[off:off + 4].view(torch.int32).item())

        ktot = 0
        if s.lnl_tap_off:
            ktot += last(s.lnl_tap_off, B * int(s.n_f))
        if s.ssi_tap_off:
            ktot += last(s.ssi_tap_off, B)
        nimp = last(s.isd_off, B) if s.isd_off else 0
        nbytes = 8.0 * B * length + (4.0 * B * length if s.ssi_tap_off else 0.0) + 12.0 * nimp
        return 2.0 * length * ktot, nbytes

    def parity_sample(self, algo, y, lo, B, length, n, seeds):
        """Oracle on n random utterances of the batch that was just timed (the checker, on the CPU)."""
        rs = np.random.RandomState(99 + algo)
        pick = sorted(set(int(v) for v in rs.randint(0, B, size=n)))
        got = y[pick, :length].cpu().numpy()
        worst = 0.0
        state = np.random.get_state()
        for row, u in zip(got, pick):
            np.random.seed(int(seeds[u]))
            ref = np.asarray(self.orc.process(self.wave_of(lo, u, length), 16000, self.orc.make_args(), algo), dtype=np.float64)
            worst = max(worst, float(np.max(np.abs(row.astype(np.float64) - ref))))
        np.random.set_state(state)
        return {"max_abs_vs_oracle": worst, "utterances": len(pick), "tolerance": 0.0 if algo == 2 else 1e-5,
                "ok": bool(worst <= (0.0 if algo == 2 else 1e-5))}


DUMP_BYTES = 60 * 2 ** 20  # --dump-outputs stays under 64 MB: larger batches are sampled by row


def dump_outputs(path, y, B, length):
    """Write rows of the [B, ld] result ``y`` (their first ``length`` samples, float32) to ``path/y.npy`` and their batch
    indices to ``path/rows.npy``; every row when they fit DUMP_BYTES, otherwise a sample fixed by its own seed (at least one
    row, cut to its first DUMP_BYTES / 4 samples when a single row is larger than that)."""
    import torch
    cols = min(length, DUMP_BYTES // 4)
    n = min(B, DUMP_BYTES // (4 * cols))
    rows = np.arange(B) if n == B else np.sort(np.random.RandomState(0).choice(B, n, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "y.npy"), y[torch.from_numpy(rows).to(y.device), :cols].cpu().numpy())
    np.save(os.path.join(path, "rows.npy"), rows.astype(np.float64))


def gpu_arm(a):
    b = Bench(a)
    torch, eng, sharding, workload = b.torch, b.eng, b.sharding, b.workload
    world, rank = b.world, b.rank
    L, algo = a.length, a.algo
    if world > 1 and not a.weak:
        B = CONFIG5_GLOBAL_BATCH // world   # BASELINE config 5: one global batch, sharded by index
        lo = rank * B
        scaling = "strong"
    else:
        B = a.batch
        lo = rank * B
        scaling = "weak"

    # ---- device-resident timing of the headline configuration -----------------------------------------------------------------
    rec, (x, ln, dp, y, bp, seeds, ld) = b.resident(algo, B, L, a.steps, a.warmup, lo=lo, planner=a.bank_planner, parity_n=16,
                                                      clocks=True, keep=True)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, y, B, L)
    if bp is not None and rank == 0:  # guard: the native planner must reproduce numpy's own draws on a sample
        from scl_deepfake_audio_detection_b200 import plans as _pl
        ref = _pl.draw_batch([L] * 4, workload.SAMPLE_RATE, b.args, algo, seeds=seeds[:4], ld=ld)
        for name in ("lnl_tap_off", "lnl_taps", "isd_off", "isd_idx", "isd_fr"):
            r = getattr(ref, name)
            if r is not None:
                assert np.array_equal(r, getattr(bp, name)[:r.shape[0]]), f"native planner diverges from numpy on {name}"

    # ---- end to end through the host-buffer C ABI --------------------------------------------------------------------------------
    e2e = {"value": None, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "skipped": "--no-e2e"}
    if not a.no_e2e:
        e2e = e2e_leg(b, algo, B, L, ld, lo, seeds, y, a)

    # ---- the other configurations of the metric (N = 1 only: they are single-GPU configurations) ---------------------------------
    configs = {}
    if world == 1 and not a.no_configs:
        del x, y, dp
        torch.cuda.empty_cache()
        configs = config_records(b, a)

    # ---- CPU baseline on this box's host cores (N=1 only) ------------------------------------------------------------------------
    cpu = None
    b.pool.close()
    if world == 1 and not a.no_cpu:
        kind = cpu_kind()
        v, ms, n = run_cpu_arm(algo, L, a.cpu_per_core, b.cores, 2, 1)
        cpu = {"value": v, "unit": UNIT, "cores": b.cores, "kind": kind,
               "sample": cpu_description(kind, n, a.cpu_per_core, b.cores, ", 2 timed steps")}
        if configs:  # BASELINE config 1: algo 1 on 32 utterances through the reference's CPU path (one batch, all host cores)
            per_core = max(1, 32 // b.cores)
            v1, ms1, n1 = run_cpu_arm(1, L, per_core, min(b.cores, 32), 2, 1)
            configs["config1_algo1_cpu_b32"] = {"algo": 1, "value": v1, "unit": UNIT, "ms_per_step": ms1, "utterances_per_step": n1,
                                                "kind": kind, "cores": min(b.cores, 32),
                                                "what": "the reference CPU path itself (no GPU): the configuration BASELINE.json lists first"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": rec["value"], "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": rec["ms_per_step"], "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": workload_name(algo, B, L, world if scaling == "strong" else 1), "algo": algo, "batch_per_gpu": B,
                       "global_batch": world * B, "utt_len": L,
                       "sharding": f"utterances by index over {world} GPU(s), no collective",
                       "l2": "inputs (%.2f GB per GPU) larger than L2; no explicit flush" % (B * ld * 4 / 1e9),
                       "plan_bank": rec["plan_bank"],
                       "waveforms": f"{min(B, UNIQUE_WAVES)} distinct synthetic waveforms per GPU (SURVEY.md 8d recipe); larger batches cycle "
                                    f"through them, every utterance with its own seed and plan",
                       "step_ms_min_median_max": rec["step_ms_min_median_max"], "host_plan_workers": b.workers, "build_id": build_id(),
                       "single_gpu_point_of_config5": "configs.config5_b65536 of the --gpus 1 line" if scaling == "strong" else None},
            "roofline": rec["roofline"],
            "parity": rec.get("parity"),
            "e2e": e2e,
            "gpu_launches": rec["gpu_launches"],
            "clocks": rec.get("clocks"),
        }
        if configs:
            line["configs"] = configs
        if cpu:
            line["cpu_baseline"] = cpu
        emit(line)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def e2e_leg(b, algo, B, L, ld, lo, seeds, y_dev, a):
    """Host buffers in, host buffers out, every step: H2D + device plan draw + kernels + D2H through rb_submit_host_seeded."""
    torch, eng, sharding, workload = b.torch, b.eng, b.sharding, b.workload
    Be = min(B, a.e2e_batch)  # utterances per end-to-end step (bounded so that the pinned buffers stay a few GB per rank)
    uniq = min(Be, UNIQUE_WAVES)
    host = b.unique_host(lo, min(B, UNIQUE_WAVES), L, ld)[:uniq]
    x_host = torch.empty((Be, ld), dtype=torch.float32).pin_memory()
    for i in range(0, Be, uniq):
        x_host[i:i + uniq] = torch.from_numpy(host[:min(uniq, Be - i)])
    y_host = [torch.empty((Be, ld), dtype=torch.float32).pin_memory() for _ in range(2)]
    seeds_e = np.ascontiguousarray(seeds[:Be], dtype=np.uint32)
    lengths = np.full(Be, L, dtype=np.int32)
    if a.host_chunk:
        eng.set_host_chunk(a.host_chunk)
    steps = max(1, min(a.steps, a.e2e_steps))

    def blocking(n):
        for _ in range(n):
            eng.process_host_seeded(algo, x_host.numpy(), lengths, seeds_e, workload.SAMPLE_RATE, b.args, out=y_host[0].numpy())

    def streaming(n):
        prev = None
        for k in range(n):
            t = eng.submit_host_seeded(algo, x_host.numpy(), lengths, seeds_e, workload.SAMPLE_RATE, b.args, out=y_host[k % 2].numpy())
            if prev is not None:
                eng.wait_host(prev)
            prev = t
        eng.wait_host(prev)

    def timed(fn):
        fn(2)
        sharding.barrier()
        t0 = time.perf_counter()
        fn(steps)
        dt = time.perf_counter() - t0
        sharding.barrier()
        return sharding.max_over_ranks(dt / steps, b.dev)

    sync_s = timed(blocking)
    h2d, d2h = eng.last_host_traffic()
    check = y_host[0].numpy()[:, :L].copy()
    e2e_s = timed(streaming)
    assert np.array_equal(y_host[0].numpy()[:, :L], check) and np.array_equal(y_host[1].numpy()[:, :L], check), \
        "streamed results differ from the blocking call's"
    # the end-to-end result must be the resident path's result, bit for bit (same seeds -> same plans, drawn on the device)
    same = bool(np.array_equal(check, y_dev[:Be, :L].cpu().numpy())) if a.bank_planner == "device" or algo in (2,) else None
    parity = b.parity_sample(algo, torch.from_numpy(check), lo, Be, L, 16, seeds_e)

    # what the copies alone allow on this box with every rank copying at once: H2D of x and D2H into y, concurrently
    xd = torch.empty((Be, ld), dtype=torch.float32, device=b.dev)
    yd = torch.empty((Be, ld), dtype=torch.float32, device=b.dev)
    s1, s2 = torch.cuda.Stream(b.dev), torch.cuda.Stream(b.dev)

    def copies(n):
        for _ in range(n):
            with torch.cuda.stream(s1):
                xd.copy_(x_host, non_blocking=True)
            with torch.cuda.stream(s2):
                y_host[1].copy_(yd, non_blocking=True)
        s1.synchronize()
        s2.synchronize()

    copy_s = timed(copies)

    def identity(n):  # the library's own chunked pipeline with nothing to compute (algo 0 = copy): H2D | D2D | D2H
        prev = None
        for k in range(n):
            t = eng.submit_host_seeded(0, x_host.numpy(), lengths, seeds_e, workload.SAMPLE_RATE, b.args, out=y_host[k % 2].numpy())
            if prev is not None:
                eng.wait_host(prev)
            prev = t
        eng.wait_host(prev)

    ident_s = timed(identity)
    world = b.world
    copy_best = min(copy_s, ident_s)
    ceiling = world * Be / copy_best
    out = {"value": world * Be / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "batch_per_gpu": Be, "ms_per_step": e2e_s * 1e3, "steps": steps,
           "includes": "every step: H2D of its waveforms + seeds from pinned host memory, plan draw ON THE DEVICE (bit-exact replay of "
                       "numpy's MT19937 stream), kernels, D2H of its results into pinned host memory; streaming API "
                       "rb_submit_host_seeded / rb_ctx_wait with two calls in flight; blocking_call_* = one rb_process_host_seeded per step",
           "blocking_call_ms_per_step": sync_s * 1e3, "blocking_call_value": world * Be / sync_s,
           "copy_ceiling": {"value": ceiling, "unit": UNIT, "ms_per_step": copy_best * 1e3,
                            "aggregate_gb_s_each_way": world * Be * ld * 4 / copy_best / 1e9,
                            "whole_buffer_copies_ms": copy_s * 1e3, "chunked_identity_pipeline_ms": ident_s * 1e3,
                            "what": f"{world} rank(s) each moving one step's waveforms H2D and one step's results D2H concurrently from / "
                                    f"to pinned memory with nothing to compute -- the faster of two whole-buffer cudaMemcpyAsync calls on "
                                    f"two streams and the library's own chunked pipeline running algo 0 (copy); the box's PCIe / "
                                    f"host-memory ceiling for this interface"},
           "frac_of_copy_ceiling": (world * Be / e2e_s) / ceiling,
           "equals_resident_result": same, "parity": parity}
    out.update(e2e_variants(b, algo, Be, L, ld, x_host, y_host, lengths, seeds_e, check, steps, timed))
    return out


def e2e_variants(b, algo, Be, L, ld, x_host, y_host, lengths, seeds_e, check, steps, timed):
    """Reduced-traffic forms of the same step, where the caller's data allows them: 16-bit PCM in (what a wav file holds;
    librosa.load of 16-bit audio is exactly int16 / 32768), results left on the device for the consumer that lives there
    (main.py:57-60)."""
    eng = b.eng
    if not hasattr(eng, "submit_host_ex"):
        return {}
    torch, workload, world = b.torch, b.workload, b.world
    out = {}
    pcm = torch.empty((Be, ld), dtype=torch.int16).pin_memory()
    pcm.copy_(torch.clamp(torch.round(x_host * 32768.0), -32768, 32767).to(torch.int16))
    y_dev = torch.empty((Be, ld), dtype=torch.float32, device=b.dev)
    for name, xin, dtype, sink in (("pcm16_in_host_out", pcm, "pcm16", None), ("pcm16_in_device_out", pcm, "pcm16", y_dev),
                                   ("f32_in_device_out", x_host, "f32", y_dev)):
        def run(n, xin=xin, dtype=dtype, sink=sink):
            prev = None
            for k in range(n):
                dst = sink if sink is not None else y_host[k % 2].numpy()
                t = eng.submit_host_ex(algo, xin.numpy(), dtype, lengths, seeds_e, workload.SAMPLE_RATE, b.args, out=dst)
                if prev is not None:
                    eng.wait_host(prev)
                prev = t
            eng.wait_host(prev)

        s = timed(run)
        h2d, d2h = eng.last_host_traffic()
        out[name] = {"value": world * Be / s, "unit": UNIT, "ms_per_step": s * 1e3, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h}
        if dtype == "f32" and sink is not None:
            out[name]["equals_host_out_result"] = bool(np.array_equal(y_dev[:, :L].cpu().numpy(), check))
    return {"variants": out}


def config_records(b, a):
    """The other configurations BASELINE.json's metric names, each timed resident in HBM with its own roofline and parity."""
    L = a.length
    out = {}
    quick = dict(steps=max(10, a.steps), warmup=a.warmup)
    out["algo1_b4096"] = b.resident(1, 4096, L, parity_n=4, **quick)
    out["algo3_b4096"] = b.resident(3, 4096, L, parity_n=4, **quick)
    out["config2_algo2_b1024"] = b.resident(2, 1024, L, steps=50, warmup=5, parity_n=8)
    out["config2_algo3_b1024"] = b.resident(3, 1024, L, parity_n=4, **quick)
    out["algo2_b4096"] = b.resident(2, 4096, L, steps=50, warmup=5, parity_n=8)
    if not a.no_config5:
        out["config5_b65536"] = b.resident(5, CONFIG5_GLOBAL_BATCH, L, steps=3, warmup=1, parity_n=4)
    try:
        out["ragged_uncropped_b1024"] = bench_ragged(b, a)
    except Exception as e:  # a sub-record must never take the headline down
        out["ragged_uncropped_b1024"] = {"error": repr(e)}
    if not a.no_config4:
        try:
            out["config4_multiview_8192x4"] = bench_config4(b.eng, b.args, items=8192, steps=3, length=L, orc=b.orc)
        except Exception as e:  # a sub-record must never take the headline down
            out["config4_multiview_8192x4"] = {"error": repr(e)}
    return out


def bench_ragged(b, a, B=1024, steps=5):
    """What the loaders really feed RawBoost (asvspoof_2019_augall_3.py:105-117): the un-cropped utterance. A ragged batch with an
    ASVspoof-2019-LA-like length mix (1.5 - 13 s at 16 kHz), algo 5, plans drawn on the device (rows beyond 65536 samples take
    the planner's global-memory permutation), device-resident. Reported in utterances/s and in 64600-sample equivalents/s."""
    import ctypes as C
    torch, eng, workload = b.torch, b.eng, b.workload
    rs = np.random.RandomState(2019)
    lengths = np.clip(rs.gamma(shape=3.2, scale=16000.0, size=B) + 20000, 24000, 211000).astype(np.int32)
    ld = (int(lengths.max()) + 3) // 4 * 4
    gen = torch.Generator(device=b.dev).manual_seed(7)
    x = torch.zeros((B, ld), dtype=torch.float32, device=b.dev)
    x.normal_(0, 0.1, generator=gen).clamp_(-1, 1)
    ln = torch.from_numpy(lengths).to(b.dev)
    seeds = np.array([workload.seed_for(u) for u in range(B)], dtype=np.uint32)
    t0 = time.perf_counter()
    dp = eng.draw_device_plan(ln, seeds, workload.SAMPLE_RATE, b.args, 5, ld)
    torch.cuda.synchronize()
    t_plan = time.perf_counter() - t0
    bp = eng.download_plan(dp)
    flops = bp.fir_flops()
    y = torch.zeros_like(x)
    for _ in range(2):
        eng.process(5, x, ln, dp, out=y)
    torch.cuda.synchronize()
    b.lib.rb_profile_read(None, None, 1)
    b.lib.rb_profile_enable(1)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(steps):
        eng.process(5, x, ln, dp, out=y)
    ev[1].record()
    torch.cuda.synchronize()
    b.lib.rb_profile_enable(0)
    fir_ms, fir_n = C.c_double(0.0), C.c_uint64(0)
    b.lib.rb_profile_read(C.byref(fir_ms), C.byref(fir_n), 1)
    ms = ev[0].elapsed_time(ev[1]) / steps
    ffma2, ffma = b.fp32_peak()
    tf = flops / (fir_ms.value / steps * 1e-3) / 1e12
    # parity: four rows (the longest among them) against the oracle on the very samples that were filtered
    worst, state = 0.0, np.random.get_state()
    pick = sorted({int(np.argmax(lengths)), int(np.argmin(lengths)), 3, B - 1})
    for u in pick:
        n = int(lengths[u])
        np.random.seed(int(seeds[u]))
        ref = np.asarray(b.orc.process(x[u, :n].cpu().numpy(), 16000, b.orc.make_args(), 5), dtype=np.float64)
        worst = max(worst, float(np.max(np.abs(y[u, :n].cpu().numpy().astype(np.float64) - ref))))
    np.random.set_state(state)
    total = float(lengths.astype(np.int64).sum())
    rec = {"algo": 5, "batch_per_gpu": B, "value": B / ms * 1e3, "unit": UNIT, "ms_per_step": ms,
           "lengths": {"min": int(lengths.min()), "mean": total / B, "max": int(lengths.max()), "rows_beyond_65536": int((lengths > 65536).sum())},
           "equivalent_64600_sample_utt_per_s": total / 64600.0 / ms * 1e3,
           "device_plan_draw_ms": t_plan * 1e3,
           "roofline": {"bound": "fp32", "kernel": "fir_bank_kernel", "achieved": tf, "peak": max(ffma2, ffma), "unit": "TFLOP/s",
                        "frac": tf / max(ffma2, ffma), "algorithmic_flops_per_step": flops},
           "parity": {"max_abs_vs_oracle": worst, "utterances": len(pick), "tolerance": 1e-5, "ok": bool(worst <= 1e-5)},
           "waveforms": "speech-level gaussian generated on the device (a sub-record: not the 64600-sample recipe of SURVEY.md 8d)"}
    del x, y, dp
    torch.cuda.empty_cache()
    return rec


def bench_config4(eng, args, items=8192, steps=3, length=64600, trim=64000, orc=None):
    """BASELINE config 4, device-resident: per bona fide sample 4 RawBoost (algo 5) utterances -- its 3 vocoded copies and the
    anchor, seeded in the loader's order -- then the shared crop and the assembly of the item's 8 views in the model's layout
    [V, 64000] with the label vector. Plans are drawn on the device from the seeds, overlapped with the filtering; the
    assembly reads x / y in place. ``orc``: the oracle module for an in-run parity sample (checker only)."""
    import torch
    from scl_deepfake_audio_detection_b200 import plans as _plans, workload
    from scl_deepfake_audio_detection_b200.multiview import LAYOUT_MODEL, assemble_ex, item_labels, item_view_rows
    G, nvoc = int(items), 3
    B, V = 4 * G, 8
    dev = eng.device
    ld = _plans.padded_ld(length)
    gen = torch.Generator(device=dev).manual_seed(1)
    x = torch.zeros((B, ld), dtype=torch.float32, device=dev)
    x[:, :length].normal_(0, 0.1, generator=gen).clamp_(-1, 1)
    x[1::2, :length].uniform_(-0.9, 0.9, generator=gen)
    ln = torch.full((B,), length, dtype=torch.int32, device=dev)
    seeds_np = np.array([workload.seed_for(u) for u in range(B)], dtype=np.uint32)
    seeds = torch.from_numpy(seeds_np.view(np.int32)).to(dev)
    rs = np.random.RandomState(4)
    starts_np = np.array([int(rs.rand() * (length - trim)) for _ in range(G)], dtype=np.int32)
    starts = torch.from_numpy(starts_np).to(dev)
    rows = torch.from_numpy(item_view_rows(G, nvoc).reshape(-1)).to(dev)
    label = torch.from_numpy(item_labels(nvoc)).to(dev)
    y = torch.empty_like(x)
    out = torch.empty((G, V, trim), dtype=torch.float32, device=dev)
    res = {}

    def step():
        eng.process_device_seeded(5, x, ln, seeds, workload.SAMPLE_RATE, args, out=y)
        res["out"] = assemble_ex(eng, x, y, rows, ln, V, starts, trim, True, LAYOUT_MODEL, out=out, view_label=label)

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    ev[0].record()
    for i in range(steps):
        step()
        ev[i + 1].record()
    torch.cuda.synchronize()
    ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]
    mean = ev[0].elapsed_time(ev[-1]) / steps
    rec = {"config": "BASELINE config 4: 4 RawBoost views per bona fide sample + shared crop + view assembly [V=8, 64000] + labels",
           "items_per_step": G, "rawboost_utterances_per_step": B, "value": B / mean * 1e3, "unit": "utt/s", "ms_per_step": mean,
           "step_ms_min_median_max": [min(ms), statistics.median(ms), max(ms)], "items_per_s": G / mean * 1e3,
           "includes": "device plan draw from seeds (overlapped with the filtering, rb_submit_seeded_ex device -> device) + algo-5 kernels "
                       "+ rb_multiview_assemble_ex reading originals and results in place (no regrouping copy) + label vector",
           "output_gb_per_step": out.numel() * 4 / 1e9}
    if orc is not None:  # parity sample: the last item and one in the middle, all 8 views, against the oracle
        worst, state = 0.0, np.random.get_state()
        _, _, labels = res["out"]
        for g in (G // 2, G - 1):
            xs = x[4 * g:4 * g + 4, :length].cpu().numpy()
            views = [xs[3], None, xs[0], xs[1], xs[2], None, None, None]
            for k, r in ((1, 3), (5, 0), (6, 1), (7, 2)):
                np.random.seed(int(seeds_np[4 * g + r]))
                views[k] = np.asarray(orc.process(xs[r], workload.SAMPLE_RATE, orc.make_args(), 5))
            s0 = int(starts_np[g])
            got = out[g].cpu().numpy().astype(np.float64)
            for v in range(V):
                worst = max(worst, float(np.max(np.abs(got[v] - np.asarray(views[v], dtype=np.float64)[s0:s0 + trim]))))
            assert labels[g].cpu().numpy().tolist() == item_labels(nvoc).tolist()
        np.random.set_state(state)
        rec["parity"] = {"max_abs_vs_oracle": worst, "items": 2, "views": V, "tolerance": 1e-5, "ok": bool(worst <= 1e-5)}
    del x, y, out
    torch.cuda.empty_cache()
    return rec


_REAL_STDOUT = None


def quiet_stdout():
    """Route everything libraries print to fd 1 (e.g. NCCL's version banner) to stderr; rank 0's JSON line goes to the real
    stdout through :func:`emit`, so stdout carries exactly one line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps of the headline configuration (its 'value', and what "
                    "--dump-outputs writes); the sub-records under 'configs' and 'e2e' time their own step counts and report them")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--algo", type=int, default=5, help="RawBoost algo (BASELINE config 3: algo 5 = LnL -> ISD)")
    ap.add_argument("--batch", type=int, default=4096, help="utterances per GPU per step at N=1 (BASELINE config 3: 4096)")
    ap.add_argument("--length", type=int, default=64600)
    ap.add_argument("--weak", action="store_true", help="N>1: --batch utterances per GPU instead of config 5's global 65536")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--e2e-batch", type=int, default=4096, help="utterances per GPU per end-to-end step (upper bound; keeps the pinned buffers at ~4 GB per rank)")
    ap.add_argument("--bank-planner", choices=["native", "device"], default="native",
                    help="who draws the resident plan bank of the headline configuration: the native host planner (checked against "
                         "numpy on a sample) or the device planner")
    ap.add_argument("--host-chunk", type=int, default=0, help="utterances per pipeline chunk of the host-buffer entry (0 = 4 per SM)")
    ap.add_argument("--no-e2e", action="store_true", help="skip the end-to-end leg (profiling runs)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg (profiling runs)")
    ap.add_argument("--no-configs", action="store_true", help="skip the sub-records of the other configurations")
    ap.add_argument("--no-config4", action="store_true")
    ap.add_argument("--no-config5", action="store_true")
    ap.add_argument("--cpu-per-core", type=int, default=32, help="utterances per host core per CPU-baseline step (SURVEY.md 8d: >= 32)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the headline configuration's last timed result to DIR/*.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs needs --impl b200")
    a.warmup = max(a.warmup, 3) if a.impl == "b200" else a.warmup
    quiet_stdout()
    if a.impl == "reference":
        reference_arm(a)
    else:
        gpu_arm(a)


if __name__ == "__main__":
    main()

"""CPU-side tests: plan drawing vs the oracle and the reference's stream digests, CSR packing, the C-ABI library's
exported symbols, loud failure without a GPU, and the sharding helpers under a 2-process gloo group."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, stream_digest
from oracle import rawboost_oracle as orc

ARGS = orc.make_args()


@pytest.fixture(scope="module")
def P():
    from scl_deepfake_audio_detection_b200 import plans
    return plans


def test_surface_names_and_signatures():
    """Same names and argument lists as datautils/RawBoost.py and the loaders' dispatcher (SURVEY.md 8b)."""
    import inspect
    from scl_deepfake_audio_detection_b200 import RawBoost as rb
    want = {
        "randRange": ["x1", "x2", "integer"],
        "normWav": ["x", "always"],
        "genNotchCoeffs": ["nBands", "minF", "maxF", "minBW", "maxBW", "minCoeff", "maxCoeff", "minG", "maxG", "fs"],
        "filterFIR": ["x", "b"],
        "LnL_convolutive_noise": ["x", "N_f", "nBands", "minF", "maxF", "minBW", "maxBW", "minCoeff", "maxCoeff", "minG", "maxG",
                                  "minBiasLinNonLin", "maxBiasLinNonLin", "fs"],
        "ISD_additive_noise": ["x", "P", "g_sd"],
        "SSI_additive_noise": ["x", "SNRmin", "SNRmax", "nBands", "minF", "maxF", "minBW", "maxBW", "minCoeff", "maxCoeff", "minG",
                               "maxG", "fs"],
        "process_Rawboost_feature": ["feature", "sr", "args", "algo"],
        "RawBoost12": ["x", "args", "sr", "audio_path"],
    }
    for name, params in want.items():
        assert list(inspect.signature(getattr(rb, name)).parameters) == params, name


def test_randrange_and_notch_match_reference_golden(P, golden):
    arrays, meta = golden
    r = meta["ops"]["randRange"]
    np.random.seed(3)
    f = P.randRange(20, 8000, 0)
    assert isinstance(f, np.ndarray) and f.shape == (1,) and float(f[0]) == r["float"]
    assert P.randRange(10, 100, 1) == r["int"]
    assert float(P.randRange(-5, -20, 0)[0]) == r["reversed"]
    assert stream_digest() == r["stream"]
    for u in range(6):
        np.random.seed(orc.seed_for(u))
        b = P.genNotchCoeffs(5, 20, 8000, 100, 1000, 10, 100, 0, 0, 16000)
        assert b.dtype == np.float64 and b.shape[0] == meta["ops"][f"notch_u{u}"]["K"]
        np.testing.assert_allclose(b, arrays[f"notch_u{u}"], rtol=0, atol=1e-15)
        assert stream_digest() == meta["ops"][f"notch_u{u}"]["stream"]


@pytest.mark.parametrize("algo", list(range(1, 9)))
def test_plan_draws_leave_the_reference_stream_state(P, golden, algo):
    """Drawing a plan consumes the global stream exactly as the reference's call does (integer-exact parity)."""
    _, meta = golden
    for loud in (0, 1):
        for u in (0, 1):
            c = meta["cases"][f"algo{algo}_loud{loud}_u{u}"]
            np.random.seed(orc.seed_for(u))
            P.draw_for_algo(c["L"], 16000, ARGS, algo)
            assert stream_digest() == c["stream"]
    for key in (k for k in meta["full"] if k.startswith(f"algo{algo}_")):
        u = int(key.split("_")[2][1:])
        np.random.seed(orc.seed_for(u))
        P.draw_for_algo(64600, 16000, ARGS, algo)
        assert stream_digest() == meta["full"][key]["stream"]


def test_plans_equal_oracle_plans(P):
    np.random.seed(21)
    p = P.draw_for_algo(64600, 16000, ARGS, 4)
    np.random.seed(21)
    q1 = orc.draw_lnl_plan(5, 5, 20, 8000, 100, 1000, 10, 100, 0, 0, 5, 20, 16000)
    q2 = orc.draw_isd_plan(64600, 10)
    q3 = orc.draw_ssi_plan(64600, 10, 40, 5, 20, 8000, 100, 1000, 10, 100, 0, 0, 16000)
    assert all(np.array_equal(a, b) for a, b in zip(p.lnl_taps, q1.taps))
    assert p.isd_idx.dtype == np.int64 and np.array_equal(p.isd_idx, q2.idx) and np.array_equal(p.isd_fr, q2.f_r)
    assert np.array_equal(p.ssi_noise, q3.noise) and np.array_equal(p.ssi_taps, q3.taps) and p.ssi_snr_db == q3.snr_db


def test_pack_builds_csr(P):
    lens = [10, 64600, 333]
    seeds = [5, 6, 7]
    bp = P.draw_batch(lens, 16000, ARGS, 4, seeds=seeds)
    assert bp.B == 3 and bp.ld == 64600 and bp.lengths.dtype == np.int32 and bp.lengths.tolist() == lens
    assert bp.n_f == 5 and bp.lnl_tap_off.shape == (16,) and bp.lnl_tap_off[0] == 0
    assert bp.lnl_taps.dtype == np.float32 and bp.lnl_taps.shape[0] == bp.lnl_tap_off[-1]
    k = np.diff(bp.lnl_tap_off)
    assert np.all(k % 2 == 1) and k.min() >= 51 and k.max() <= 491
    assert bp.isd_off.tolist()[0] == 0 and bp.isd_idx.dtype == np.int32 and bp.isd_fr.dtype == np.float64
    for u, n in enumerate(lens):
        idx = bp.isd_idx[bp.isd_off[u]:bp.isd_off[u + 1]]
        assert len(set(idx.tolist())) == idx.shape[0] and (idx.size == 0 or (idx.min() >= 0 and idx.max() < n))
        assert np.all(bp.ssi_noise[u, n:] == 0)
    assert bp.ssi_noise.shape == (3, 64600) and bp.ssi_snr_db.shape == (3,) and bp.g_sd == 2.0
    # per-utterance re-seeding makes plans independent of batch composition (sharding invariance)
    solo = P.draw_batch([64600], 16000, ARGS, 4, seeds=[6])
    assert np.array_equal(solo.isd_idx, bp.isd_idx[bp.isd_off[1]:bp.isd_off[2]])
    assert np.array_equal(solo.lnl_taps, bp.lnl_taps[bp.lnl_tap_off[5]:bp.lnl_tap_off[10]])
    assert bp.fir_flops() == pytest.approx(2.0 * sum(n * (np.diff(bp.lnl_tap_off)[5 * u:5 * u + 5].sum() + np.diff(bp.ssi_tap_off)[u])
                                                    for u, n in enumerate(lens)))


def test_library_exports_every_header_symbol():
    """The C-ABI library loads and exports exactly what include/rawboost_b200.h declares (no compute calls)."""
    import ctypes
    from scl_deepfake_audio_detection_b200 import _lib
    header = open(os.path.join(ROOT, "include", "rawboost_b200.h")).read()
    declared = set(re.findall(r"RB_API\s+[\w\s\*]+?\b(rb_\w+)\s*\(", header))
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    lib = _lib.load()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.rb_abi_version() == 1
    assert lib.rb_error_string(0) == b"ok" and b"plan" in lib.rb_error_string(-5)
    assert lib.rb_workspace_bytes(0, 64600) == 0
    small, big = lib.rb_workspace_bytes(1, 64600), lib.rb_workspace_bytes(4096, 64600)
    assert 2 * 64600 * 4 <= small and big >= 4096 * 2 * 64600 * 4 and big < 4096 * 2.2 * 64600 * 4  # algo 8: two branch buffers
    assert ctypes.sizeof(_lib.RbPlan) == 88  # matches the C struct layout on LP64
    # argument validation happens before any CUDA call, so it is checkable without a device
    assert lib.rb_process(5, 16, 16, 2, 63, None, 16, 256, 1 << 30, None) == -2
    assert lib.rb_process(5, None, None, 2, 64, None, None, None, 0, None) == -1
    assert lib.rb_process(5, None, None, 0, 64, None, None, None, 0, None) == 0


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("has a GPU")
    from scl_deepfake_audio_detection_b200 import RawBoost as rb, _lib
    from scl_deepfake_audio_detection_b200.engine import Engine
    with pytest.raises(_lib.RawBoostLibraryError):
        Engine(0)
    x = orc.synth_utterance(0, 1000)
    for call in (lambda: rb.normWav(x, 1), lambda: rb.filterFIR(x, np.ones(3)), lambda: rb.process_Rawboost_feature(x, 16000, ARGS, 5),
                 lambda: rb.ISD_additive_noise(x, 10, 2)):
        with pytest.raises(_lib.RawBoostLibraryError):
            call()
    assert rb.process_Rawboost_feature(x, 16000, ARGS, 0) is x  # identity needs no device


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "scl-deepfake-audio-detection_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("SURVEY", ""), f"{f} mentions the oracle"


def test_shard_range_partitions():
    from scl_deepfake_audio_detection_b200.sharding import shard_range
    for total in (0, 1, 7, 4096, 65536, 65537):
        for world in (1, 2, 3, 4, 8):
            rs = [shard_range(total, r, world) for r in range(world)]
            assert rs[0][0] == 0 and rs[-1][1] == total
            assert all(rs[i][1] == rs[i + 1][0] for i in range(world - 1))
            sizes = [b - a for a, b in rs]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        shard_range(10, 2, 2)


_WORKER = r"""
import os, sys
sys.path.insert(0, sys.argv[1])
import numpy as np
import torch.distributed as dist
from scl_deepfake_audio_detection_b200 import sharding, plans
from oracle import rawboost_oracle as orc
sharding.init_process_group("gloo")
rank, _, world = sharding.env_rank_world()
lo, hi = sharding.shard_range(6, rank, world)
# each rank draws only its shard's plans; per-utterance seeding makes them identical to a single-process draw
bp = plans.draw_batch([4000] * (hi - lo), 16000, orc.make_args(), 5, seeds=[orc.seed_for(u) for u in range(lo, hi)])
full = plans.draw_batch([4000] * 6, 16000, orc.make_args(), 5, seeds=[orc.seed_for(u) for u in range(6)])
ok = np.array_equal(bp.isd_idx, full.isd_idx[full.isd_off[lo]:full.isd_off[hi]]) and \
     np.array_equal(bp.lnl_taps, full.lnl_taps[full.lnl_tap_off[5 * lo]:full.lnl_tap_off[5 * hi]])
sharding.barrier()
t = sharding.max_over_ranks(1.0 + rank)
n = sharding.sum_over_ranks(hi - lo)
assert ok and t == float(world) and n == 6.0, (ok, t, n)
dist.destroy_process_group()
print("rank", rank, "ok")
"""


def test_two_rank_gloo_sharding(tmp_path):
    """world_size-2 gloo job on CPU: shards partition the batch, plans match the single-process draw, timing is MAX-reduced."""
    script = tmp_path / "w.py"
    script.write_text(_WORKER)
    port = 29000 + os.getpid() % 2000
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), LOCAL_RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, str(script), ROOT], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    for p in procs:
        out, _ = p.communicate(timeout=180)
        assert p.returncode == 0, out.decode()


# ---------------------------------------------------------------------------------------------------------
# native planner (csrc/rb_planner.cpp): bit-exact with the numpy calls of plans.py
# ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def native():
    from scl_deepfake_audio_detection_b200.native_planner import NativePlanner
    return NativePlanner(threads=2, pinned=False)


def _same_plan(a, b):
    for name in ("lnl_tap_off", "isd_off", "isd_idx", "ssi_tap_off"):
        x, y = getattr(a, name), getattr(b, name)
        assert (x is None) == (y is None), name
        if x is not None:
            assert x.dtype == y.dtype and np.array_equal(x, y), name      # integer work: bit-exact
    for name in ("isd_fr", "ssi_noise", "ssi_snr_db"):
        x, y = getattr(a, name), getattr(b, name)
        if y is not None:
            assert np.array_equal(x, y), name                              # pure MT19937 arithmetic: bit-exact
    for name in ("lnl_taps", "ssi_taps"):
        x, y = getattr(a, name), getattr(b, name)
        if y is not None:                                                  # libm vs numpy SIMD: <= 1 float32 ulp
            np.testing.assert_allclose(x, y, rtol=1.3e-7, atol=1e-12, err_msg=name)
    assert a.n_f == b.n_f and a.g_sd == b.g_sd and a.ld == b.ld


@pytest.mark.parametrize("algo", [1, 2, 3, 4, 5, 6, 7, 8])
def test_native_planner_matches_numpy_per_utterance_seeds(P, native, algo):
    lens = [64600, 1, 2, 37, 4097, 70001, 16000]
    seeds = [orc.seed_for(u) for u in range(len(lens))]
    a = native.draw(lens, 16000, ARGS, algo, seeds=seeds, copy=True)
    b = P.draw_batch(lens, 16000, ARGS, algo, seeds=seeds)
    _same_plan(a, b)


def test_native_planner_continues_the_global_numpy_stream(P, native, golden):
    """Stream mode: consumes np.random's global state exactly as the reference's calls do (digests from the reference)."""
    _, meta = golden
    for algo in (2, 4, 5):
        for u in (0, 1):
            c = meta["cases"][f"algo{algo}_loud0_u{u}"]
            np.random.seed(orc.seed_for(u))
            native.draw([c["L"]], 16000, ARGS, algo, use_global_stream=True)
            assert stream_digest() == c["stream"]
    # mid-block start and a cached gaussian carried in and out
    np.random.seed(5)
    np.random.normal(size=3)
    b = P.draw_batch([3001, 64600], 16000, ARGS, 7)
    ref_state = np.random.get_state()
    np.random.seed(5)
    np.random.normal(size=3)
    a = native.draw([3001, 64600], 16000, ARGS, 7, use_global_stream=True, copy=True)
    got = np.random.get_state()
    _same_plan(a, b)
    assert np.array_equal(ref_state[1], got[1]) and ref_state[2:] == got[2:]
    # algos without SSI exchange the words directly with numpy's bit generator: a pending cached gaussian must survive untouched
    for algo in (1, 2, 5, 8):
        tails = []
        for draw in (lambda: P.draw_batch([777, 64600], 16000, ARGS, algo),
                     lambda: native.draw([777, 64600], 16000, ARGS, algo, use_global_stream=True, copy=True)):
            np.random.seed(11)
            np.random.normal()                      # leaves the second value of the pair cached
            plan = draw()
            st = np.random.get_state()
            assert st[3] == 1                        # still cached
            tails.append((plan, st[1].copy(), st[2:], np.random.normal(), np.random.uniform()))
        _same_plan(tails[1][0], tails[0][0])
        assert np.array_equal(tails[0][1], tails[1][1]) and tails[0][2:] == tails[1][2:]


def test_native_planner_nondefault_args(P, native):
    args = orc.make_args(nBands=7, maxCoeff=300, minCoeff=3, N_f=3, P=37, g_sd=5, SNRmin=0, SNRmax=3, minG=-4, maxG=6, minF=1, maxF=7999)
    a = native.draw([20000, 333], 16000, args, 4, seeds=[9, 10], copy=True)
    b = P.draw_batch([20000, 333], 16000, args, 4, seeds=[9, 10])
    _same_plan(a, b)
    assert np.diff(a.lnl_tap_off).max() > 512  # cascades longer than one staged segment


def test_workload_matches_oracle_workload():
    from scl_deepfake_audio_detection_b200 import workload
    for u in (0, 1, 7):
        for loud in (False, True):
            assert np.array_equal(workload.synth_utterance(u, 5000, loud), orc.synth_utterance(u, 5000, loud))
        assert workload.seed_for(u) == orc.seed_for(u)
    assert vars(workload.default_args()) == vars(orc.make_args())


# ---------------------------------------------------------------------------------------------------------
# property sweep: the native planner against numpy itself over random arguments, lengths, algos and seeds
# ---------------------------------------------------------------------------------------------------------
hypothesis = pytest.importorskip("hypothesis")
from hypothesis import given, settings, strategies as st  # noqa: E402


@st.composite
def _planner_cases(draw):
    min_c = draw(st.integers(2, 40))
    args = orc.make_args(
        N_f=draw(st.integers(1, 6)), nBands=draw(st.integers(1, 6)),
        minF=draw(st.integers(1, 400)), maxF=draw(st.integers(2000, 8000)),
        minBW=draw(st.integers(20, 200)), maxBW=draw(st.integers(300, 1500)),
        minCoeff=min_c, maxCoeff=min_c + draw(st.integers(1, 120)),
        minG=draw(st.integers(-6, 3)), maxG=draw(st.integers(-6, 3)),          # low > high is legal (RawBoost.py:62-64)
        minBiasLinNonLin=draw(st.integers(0, 8)), maxBiasLinNonLin=draw(st.integers(0, 25)),
        P=draw(st.integers(0, 40)), g_sd=draw(st.integers(1, 4)),
        SNRmin=draw(st.integers(0, 20)), SNRmax=draw(st.integers(20, 45)))
    algo = draw(st.integers(1, 8))
    lens = draw(st.lists(st.integers(1, 3000), min_size=1, max_size=3))
    seed = draw(st.integers(0, 2 ** 32 - 1))
    sr = draw(st.sampled_from([16000, 8000, 22050]))
    if args.maxF >= sr // 2:
        args.maxF = sr // 2 - 1
    return args, algo, lens, seed, sr


@settings(max_examples=40, deadline=None)
@given(_planner_cases())
def test_native_planner_property_sweep(case):
    """Seeded and global-stream drawing equal numpy's draws (integers and stream state bit for bit) for arbitrary knobs."""
    from scl_deepfake_audio_detection_b200 import plans as P
    from scl_deepfake_audio_detection_b200.native_planner import NativePlanner
    args, algo, lens, seed, sr = case
    native = NativePlanner(threads=2, pinned=False)
    seeds = [(seed + 7919 * u) % 2 ** 32 for u in range(len(lens))]
    _same_plan(native.draw(lens, sr, args, algo, seeds=seeds, copy=True), P.draw_batch(lens, sr, args, algo, seeds=seeds))
    np.random.seed(seed)
    ref = P.draw_batch(lens, sr, args, algo)
    ref_state = np.random.get_state()
    np.random.seed(seed)
    got = native.draw(lens, sr, args, algo, use_global_stream=True, copy=True)
    got_state = np.random.get_state()
    _same_plan(got, ref)
    assert np.array_equal(ref_state[1], got_state[1]) and ref_state[2:] == got_state[2:]


def test_header_is_plain_c(tmp_path):
    """include/rawboost_b200.h is the C ABI: it must compile as C (no C++ types in the signatures)."""
    src = tmp_path / "use.c"
    src.write_text('#include "rawboost_b200.h"\nint main(void) { rb_plan p; rb_args a; (void)p; (void)a; return RB_ABI_VERSION == 1 ? 0 : 1; }\n')
    out = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr


# -----------------------------------------------------------------------------------------------------------------------------
@pytest.fixture
def cuobjdump_on_path(monkeypatch):
    """The toolkit's cuobjdump on PATH: found there or where csrc/build.sh takes it from, next to $NVCC (default
    /usr/local/cuda/bin/nvcc), so that a shell without the toolkit on PATH still runs the SASS checks against the built library."""
    import shutil
    from scl_deepfake_audio_detection_b200 import _lib
    nvcc = shutil.which(os.environ.get("NVCC") or "/usr/local/cuda/bin/nvcc")
    if shutil.which("cuobjdump") is None and nvcc and os.access(os.path.join(os.path.dirname(nvcc), "cuobjdump"), os.X_OK):
        monkeypatch.setenv("PATH", os.path.dirname(nvcc) + os.pathsep + os.environ.get("PATH", ""))
    if shutil.which("cuobjdump") is None or not os.path.exists(_lib.LIB_PATH):
        pytest.skip("cuobjdump or the built library is not available")


# the compiled FIR-bank kernel keeps its shape: packed FFMA2 body loop, no spills, 4 CTAs per SM worth of registers
def test_fir_kernel_sass_contract(cuobjdump_on_path):
    from scl_deepfake_audio_detection_b200 import _lib
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import sass_loop_stats
    loops, reuse = {}, {}
    for name, ins in sass_loop_stats.functions(_lib.LIB_PATH):
        m = re.search(r"fir_bank_kernelILi(\d)ELi(\d+)E", name)
        if not m:
            continue
        text = [t for _, t, _ in ins]
        assert not any("STL" in t or "LDL" in t for t in text), "local-memory spills in " + name
        body = [t for _, t, _ in (sass_loop_stats.body_loop(ins) or [])]
        loops[int(m.group(1))] = (int(m.group(2)), sum("FFMA2" in t for t in body), sum("LDS.128" in t for t in body), len(body))
        ff = [(t, hi) for _, t, hi in (sass_loop_stats.body_loop(ins) or []) if t.startswith("FFMA2")]
        reuse[int(m.group(1))] = sum(((hi >> 58) & 0xf) != 0 for _, hi in ff) / max(1, len(ff))
    assert set(loops) == {0, 1, 2}, "one instantiation per tail mode"
    assert loops[0][0] == 28 and loops[1][0] == loops[2][0] == 20, "outputs per thread: 28 for the plain filter, 20 with a tail"
    for mode, (kr, ffma2, lds, total) in loops.items():
        # a body covers kr + 4 taps: (kr + 4) / 4 groups of 2 * kr FFMA2 and 3 LDS.128 (240 + 18 at kr = 20, 448 + 24 at 28);
        # the loop holds two bodies (single filters) or four (LnL bank)
        per_body, lds_body = (kr + 4) // 4 * 2 * kr, (kr + 4) // 4 * 3
        assert ffma2 in (2 * per_body, 4 * per_body) and lds == lds_body * ffma2 // per_body, \
            f"tail mode {mode}: body loop changed shape ({ffma2} FFMA2, {lds} LDS.128)"
        assert total - ffma2 - lds <= 8, f"tail mode {mode}: {total - ffma2 - lds} other instructions inside the body loop"
    if not os.environ.get("RB_NO_SASS_PATCH"):
        # the post-link step (csrc/sass_reuse_patch.py) ran: ptxas alone flags ~69 % of the loop's FFMA2 for operand reuse and
        # puts a yield hint on every sixth one; the patched stream carries the flag wherever the next FFMA2 shares the tap pair
        for mode, frac in reuse.items():
            assert frac >= 0.78, f"tail mode {mode}: only {100 * frac:.1f} % of the body loop's FFMA2 carry a reuse flag -- unpatched library?"
    log = os.path.join(os.path.dirname(_lib.LIB_PATH), "librawboost_b200.rb_fir_bank.ptxas.log")
    if os.path.exists(log):
        regs = [int(r) for r in re.findall(r"Used (\d+) registers", open(log).read())]
        assert regs and max(regs) <= 128, f"more than 128 registers: fewer than 4 CTAs of 128 threads per SM ({regs})"


def test_sass_reuse_patch_is_idempotent_and_touches_control_bits_only(tmp_path, cuobjdump_on_path):
    """csrc/sass_reuse_patch.py on the (already patched) built library changes nothing; and against a library linked without it
    (when one can be produced here) it differs only in bits 45 and 58 of FFMA2 control words."""
    import subprocess
    from scl_deepfake_audio_detection_b200 import _lib
    script = os.path.join(os.path.dirname(_lib.LIB_PATH), "..", "csrc", "sass_reuse_patch.py")
    out = tmp_path / "again.so"
    subprocess.run([sys.executable, script, _lib.LIB_PATH, str(out)], check=True, capture_output=True)
    a, b = open(_lib.LIB_PATH, "rb").read(), open(out, "rb").read()
    assert a == b, "patching a patched library must be the identity"
    # rebuild the FIR object's unpatched image from the object file the library was linked from and compare the code bytes
    obj = os.path.join(os.path.dirname(_lib.LIB_PATH), "librawboost_b200.rb_fir_bank.o")
    if not os.path.exists(obj):
        pytest.skip("object file of the FIR kernels not present")
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import sass_loop_stats
    before = {n: ins for n, ins in sass_loop_stats.functions(obj) if "fir_bank_kernel" in n}
    after = {n: ins for n, ins in sass_loop_stats.functions(_lib.LIB_PATH) if "fir_bank_kernel" in n}
    assert set(before) == set(after) and len(before) == 3
    changed = 0
    for n in before:
        assert len(before[n]) == len(after[n])
        for (a0, t0, h0), (a1, t1, h1) in zip(before[n], after[n]):
            assert a0 == a1 and re.sub(r"\.reuse", "", t0) == re.sub(r"\.reuse", "", t1), "an instruction changed"
            if h0 != h1:
                assert t0.startswith("FFMA2") and (h0 ^ h1) & ~((1 << 45) | (1 << 58)) == 0, "a bit other than yield / reuse-A changed"
                changed += 1
    assert changed > 300


def test_sass_reuse_patch_rule_on_a_synthetic_stream():
    """The rule of csrc/sass_reuse_patch.py on a hand-made instruction list: the flag goes on an FFMA2 exactly when the next FFMA2
    of the same straight-line stretch multiplies by the same tap pair and nothing in between (itself included) writes that pair."""
    import importlib.util
    path = os.path.join(ROOT, "scl-deepfake-audio-detection_b200", "csrc", "sass_reuse_patch.py")
    spec = importlib.util.spec_from_file_location("sass_reuse_patch", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    assert mod.tap_operand("FFMA2 R78, R28.reuse.F32x2.HI_LO, R24.F32x2.HI_LO, R78.F32x2.HI_LO") == "R28"
    assert mod.written("FFMA2 R36, R36.F32x2.HI_LO, R34.F32x2.HI_LO, R4.F32x2.HI_LO") == {36, 37}
    assert mod.written("LDS.128 R28, [R84+0x10]") == {28, 29, 30, 31}
    assert mod.written("@!P0 LDS.64 R6, [R2]") == {6, 7}
    assert mod.written("UIADD3 UR6, UPT, UPT, UR6, 0x4, URZ") == set()
    yield_ok = 0  # bit 45 clear = yield hint present
    lo = 0x1234
    text = [
        "FFMA2 R40, R28.F32x2.HI_LO, R8.F32x2.HI_LO, R40.F32x2.HI_LO",    # next shares R28                    -> flag
        "FFMA2 R42, R28.F32x2.HI_LO, R10.F32x2.HI_LO, R42.F32x2.HI_LO",   # an LDS in between, not touching R28 -> flag
        "LDS.128 R48, [R84+0x20]",
        "FFMA2 R44, R28.F32x2.HI_LO, R12.F32x2.HI_LO, R44.F32x2.HI_LO",   # next has another tap               -> no flag
        "FFMA2 R46, R30.F32x2.HI_LO, R8.F32x2.HI_LO, R46.F32x2.HI_LO",    # the LDS in between overwrites R30  -> no flag
        "LDS.128 R28, [R84+0x30]",
        "FFMA2 R40, R30.F32x2.HI_LO, R10.F32x2.HI_LO, R40.F32x2.HI_LO",   # writes its own tap below? no: next -> see below
        "FFMA2 R30, R30.F32x2.HI_LO, R12.F32x2.HI_LO, R42.F32x2.HI_LO",   # overwrites R30 itself              -> no flag
        "FFMA2 R44, R30.F32x2.HI_LO, R14.F32x2.HI_LO, R44.F32x2.HI_LO",   # a barrier before the next FFMA2    -> no flag
        "BAR.SYNC.DEFER_BLOCKING 0x0",
        "FFMA2 R46, R30.F32x2.HI_LO, R16.F32x2.HI_LO, R46.F32x2.HI_LO",   # last FFMA2                          -> no flag
        "EXIT", "NOP", "NOP", "NOP",
    ]
    ins = [(16 * i, t, lo + i, yield_ok) for i, t in enumerate(text)]
    blob = bytearray(b"".join(l.to_bytes(8, "little") + h.to_bytes(8, "little") for _, _, l, h in ins))
    n, r0, r1, y0, y1 = mod.patch(blob, ins)
    flagged = [i for i in range(len(text)) if (int.from_bytes(blob[16 * i + 8:16 * i + 16], "little") >> 58) & 1]
    assert (n, r0, y0) == (8, 0, 8)
    assert flagged == [0, 1, 6], flagged
    for i in flagged:  # a flagged instruction loses its yield hint; the others keep theirs
        assert (int.from_bytes(blob[16 * i + 8:16 * i + 16], "little") >> 45) & 1
    assert y1 == 8 - len(flagged) and r1 == len(flagged)
    assert all(blob[16 * i:16 * i + 8] == (lo + i).to_bytes(8, "little") for i in range(len(text))), "the low words must not change"


def test_fp32_peak_probe_uses_the_uniform_register_form(cuobjdump_on_path):
    """The roofline denominator of the FIR kernels is measured by rb_probe_fp32; its FFMA2 chain must be the fast form
    (multiplier in a uniform register), or the peak -- and with it every reported fraction -- would be off by 2 %."""
    import subprocess
    from scl_deepfake_audio_detection_b200 import _lib
    sass = subprocess.run(["cuobjdump", "-sass", "-fun", "fp32_probe_kernel", _lib.LIB_PATH], capture_output=True, text=True).stdout
    if "FFMA2" not in sass:  # older cuobjdump: no -fun filter on mangled substrings
        sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True).stdout
        sass = sass[sass.index("fp32_probe_kernelILb1"):]
        sass = sass[:sass.index("Function :", 10)] if "Function :" in sass[10:] else sass
    ffma2 = [l for l in sass.splitlines() if "FFMA2" in l]
    assert len(ffma2) >= 1024
    assert sum(" UR" in l for l in ffma2) >= 0.95 * len(ffma2), "the packed probe lost its uniform-register operand"


def test_native_planner_self_check_and_state_layout_guard():
    """The default planner of the drop-in verifies itself against numpy before its first use and leaves the global stream alone;
    the raw-state exchange is only used when numpy's private layout is what it assumes."""
    from scl_deepfake_audio_detection_b200 import native_planner as nplan
    np.random.seed(4321)
    before = np.random.get_state()
    p = nplan.NativePlanner(threads=1, pinned=False)
    p.self_check()
    after = np.random.get_state()
    assert np.array_equal(before[1], after[1]) and before[2:] == after[2:]
    assert nplan._direct_exchange_ok() is True
    # a layout mismatch must switch the exchange off, not corrupt the stream: simulate it
    nplan._direct_ok = False
    try:
        from types import SimpleNamespace
        from scl_deepfake_audio_detection_b200 import plans
        args = SimpleNamespace(**{**dict(N_f=5, nBands=5, minF=20, maxF=8000, minBW=100, maxBW=1000, minCoeff=10, maxCoeff=100, minG=0, maxG=0,
                                         minBiasLinNonLin=5, maxBiasLinNonLin=20, P=10, g_sd=2, SNRmin=10, SNRmax=40)})
        np.random.seed(9)
        got = p.draw([3000], 16000, args, 5, use_global_stream=True, copy=True)
        s1 = np.random.get_state()
        np.random.seed(9)
        want = plans.pack([plans.draw_for_algo(3000, 16000, args, 5)])
        s2 = np.random.get_state()
        assert np.array_equal(got.isd_idx, want.isd_idx) and np.array_equal(s1[1], s2[1]) and s1[2:] == s2[2:]
    finally:
        nplan._direct_ok = None


def test_native_planner_rejects_bad_arguments_instead_of_throwing():
    """rb_planner_draw validates its arguments (no C++ exception may cross the C ABI) and clips like numpy's [:n] for P > 100."""
    from types import SimpleNamespace
    from scl_deepfake_audio_detection_b200 import _lib, native_planner as nplan
    base = dict(N_f=5, nBands=5, minF=20, maxF=8000, minBW=100, maxBW=1000, minCoeff=10, maxCoeff=100, minG=0, maxG=0,
                minBiasLinNonLin=5, maxBiasLinNonLin=20, P=10, g_sd=2, SNRmin=10, SNRmax=40)
    p = nplan.NativePlanner(threads=2, pinned=False)
    for bad in (dict(P=-5), dict(minCoeff=-3), dict(nBands=0), dict(N_f=0)):
        with pytest.raises(_lib.RawBoostLibraryError):
            p.draw([1000, 1200], 16000, SimpleNamespace(**{**base, **bad}), 5, seeds=[1, 2])
    got = p.draw([1000], 16000, SimpleNamespace(**{**base, "P": 400}), 2, seeds=[3], copy=True)  # beta up to 400 %: n clipped to L
    assert 0 <= got.isd_idx.shape[0] <= 1000 and len(set(got.isd_idx.tolist())) == got.isd_idx.shape[0]
    np.random.seed(3)
    from scl_deepfake_audio_detection_b200 import plans
    want_idx, _ = plans.draw_isd(1000, 400)
    assert np.array_equal(got.isd_idx, want_idx.astype(np.int32))


def test_bench_dump_outputs_every_row_or_a_fixed_sample_under_64_mb(tmp_path):
    """``bench.py --dump-outputs``: a small result is written whole; of a 4096 x 64600 one the same seeded rows on every call,
    float32 results and float64 row numbers, under 64 MB; of rows longer than the budget one row's head."""
    import torch
    import bench
    y = torch.arange(3 * 40, dtype=torch.float32).reshape(3, 40)
    bench.dump_outputs(str(tmp_path / "small"), y, 3, 37)
    assert np.array_equal(np.load(tmp_path / "small" / "y.npy"), y[:, :37].numpy())
    assert np.load(tmp_path / "small" / "rows.npy").tolist() == [0.0, 1.0, 2.0]
    B, L = 4096, 64600
    y = torch.arange(B, dtype=torch.float32)[:, None].expand(B, L + 4)  # row u holds u
    for name in ("a", "b"):
        bench.dump_outputs(str(tmp_path / name), y, B, L)
    rows, out = np.load(tmp_path / "a" / "rows.npy"), np.load(tmp_path / "a" / "y.npy")
    assert rows.dtype == np.float64 and out.dtype == np.float32 and out.shape == (rows.shape[0], L)
    assert 100 < rows.shape[0] < B and np.all(np.diff(rows) > 0) and np.array_equal(out[:, 0], rows) and np.all(out == out[:, :1])
    assert np.array_equal(np.load(tmp_path / "b" / "rows.npy"), rows)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in ("y.npy", "rows.npy")) <= 64 * 2 ** 20
    y = torch.ones(1, 1).expand(2, 20_000_000)  # one row alone is larger than the budget: its head, not an empty file
    bench.dump_outputs(str(tmp_path / "long"), y, 2, 20_000_000)
    out = np.load(tmp_path / "long" / "y.npy", mmap_mode="r")
    assert out.shape == (1, bench.DUMP_BYTES // 4) and float(out[0, -1]) == 1.0
    assert os.path.getsize(tmp_path / "long" / "y.npy") <= 64 * 2 ** 20

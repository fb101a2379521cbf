"""The device planner (rb_devplan.cu) and the LnL bank across the whole argument domain rb_devplan_draw accepts.

rb_devplan_draw accepts nBands 1-100, any N_f >= 1, P 0-100, stages of at most 255 taps, nBands * (ceil(cmax) + 1) <= 1024
and any sample rate. Off the defaults its code takes paths the default arguments never reach: LnL draws in several windows of
fpw = max(1, min(624 / per, 32)) filters (per = 2 (3 nBands + 1) stream words per filter), the gain bias across a window
edge, stream words near the end of the two tempered blocks (nBands = 100), the f1 <= 0 / f2 >= fs/2 clamps of genNotchCoeffs
at other sample rates, 255-tap stages and 1024-tap cascades, and LnL banks of more filters than the 16 whose supports the
workspace holds (such a bank runs every tap).

CPU (needs the built library, no device): the refusal rule restated from args_ok against rb_devplan_bytes, on a boundary table
and a seeded sweep; the edge table reaches every regime it names, counted from numpy's own draws; the hand-built rows of the
large banks leave every edge tap visible to the bound.
GPU: per edge set, the device plan against numpy's (integers, gains, SNR and noise bit for bit, taps within 1 ulp(fp32)), the
dispatcher against the float64 reference within its per-sample bound (ISD alone against the oracle bit for bit), trimming on
against off; a hypothesis sweep over the whole domain; Dataset_for items at two non-default argument sets.
"""
import ctypes as C
import dataclasses
import math
import zlib
from dataclasses import dataclass, field
from typing import Tuple

import numpy as np
import pytest

from oracle import rawboost_oracle as orc  # noqa: E402  (checker only)
from scl_deepfake_audio_detection_b200 import _lib, plans

import test_gpu_fir_bank as fir_bank
from test_gpu_fir_bank import C_DENSE, Row, edge_mutations, edge_taps, ratio, reference
from test_gpu_items import Corpus, _same_stream
from test_host_logic import _same_plan
from test_tap_support import EPS, U

MT_N = 624            # words of one MT19937 block
MAX_STAGE = 255       # taps of one firwin stage the device designs
MAX_CASCADE = 1024    # freqz's 1024-point path
SUPPORT_FILTERS = 16  # LnL filters per utterance whose supports the workspace holds


def per_filter(nBands):
    """Stream words one genNotchCoeffs call consumes: (fc, bw, c) per band and the gain, two words per double."""
    return 2 * (3 * nBands + 1)


def filters_per_window(nBands):
    return max(1, min(MT_N // per_filter(nBands), 32))


def windows(a):
    return -(-a.N_f // filters_per_window(a.nBands))


def accepted(a, fs):
    """args_ok (rb_devplan.cu) restated."""
    if a.N_f < 1 or not 1 <= a.nBands <= 100:
        return False
    if not fs > 0 or not 0 <= a.P <= 100:
        return False
    cmax, cmin = max(a.minCoeff, a.maxCoeff), min(a.minCoeff, a.maxCoeff)
    if cmin < 1 or cmax + 1 > MAX_STAGE + 1:
        return False
    return a.nBands * (math.ceil(cmax) + 1) <= MAX_CASCADE


def bank_c(row):
    """Constant of the per-sample bound for a bank of notch cascades. C_DENSE holds for random taps, whose partial sums stay
    small; a notch cascade's large centre tap carries the output into the running sum, so each later tap of a K-tap filter
    rounds relative to |y| (a random walk of sqrt(K) roundings), and the N_f filter sums are added into one accumulator, each
    add rounding relative to the running total. On an NVIDIA B200 at a 1000 W power limit the largest err/tol with this
    constant was below 0.5 on every edge set (C_DENSE alone reached 1.4 at N_f = 17 and on 983-tap cascades)."""
    K = max([t.shape[0] for t in row.lnl] + ([row.ssi_taps.shape[0]] if row.ssi_taps is not None else []) + [1])
    return C_DENSE * max(1.0, math.sqrt(K / 64.0)) + len(row.lnl)


def devplan_bytes(a, fs, algo=5, B=3, ld=64):
    return int(_lib.load().rb_devplan_bytes(C.byref(_lib.args_struct(a, fs)), algo, B, ld))


# ---------------------------------------------------------------------------------------------------------------------------
# A. the refusal rule
# ---------------------------------------------------------------------------------------------------------------------------
BOUNDARY = [
    # (label, overrides, fs)
    ("cmax 255", dict(nBands=4, minCoeff=200, maxCoeff=255), 16000),
    ("cmax 255.5", dict(nBands=3, minCoeff=200, maxCoeff=255.5), 16000),
    ("cmax 256", dict(nBands=3, minCoeff=200, maxCoeff=256), 16000),
    ("cmax 255 as minCoeff", dict(nBands=4, minCoeff=255, maxCoeff=10), 16000),
    ("cmax 256 as minCoeff", dict(nBands=3, minCoeff=256, maxCoeff=10), 16000),
    ("nBands 100", dict(nBands=100, minCoeff=1, maxCoeff=9), 16000),
    ("nBands 101", dict(nBands=101, minCoeff=1, maxCoeff=9), 16000),
    ("P 100", dict(P=100), 16000),
    ("P 100.5", dict(P=100.5), 16000),
    ("P 0", dict(P=0), 16000),
    ("P -0.5", dict(P=-0.5), 16000),
    ("bound 1024", dict(nBands=4, maxCoeff=255), 16000),
    ("bound 1025", dict(nBands=5, maxCoeff=204), 16000),
    ("bound 1024 at 203.5", dict(nBands=5, maxCoeff=203.5), 16000),
    ("minCoeff > maxCoeff", dict(minCoeff=100, maxCoeff=10), 16000),
    ("minCoeff > maxCoeff past the bound", dict(nBands=5, minCoeff=204, maxCoeff=10), 16000),
    ("cmin 1", dict(minCoeff=1, maxCoeff=9), 16000),
    ("cmin 0.5", dict(minCoeff=0.5, maxCoeff=9), 16000),
    ("N_f 0", dict(N_f=0), 16000),
    ("N_f 1000", dict(N_f=1000), 16000),
    ("fs 0", dict(), 0),
    ("fs 48000", dict(maxF=24000), 48000),
]


@pytest.mark.parametrize("label,kw,fs", BOUNDARY, ids=[b[0] for b in BOUNDARY])
def test_refusal_rule_at_the_boundaries(label, kw, fs):
    a = orc.make_args(**kw)
    n = devplan_bytes(a, fs)
    assert (n > 0) == accepted(a, fs), f"{label}: rb_devplan_bytes {n}, restated rule {accepted(a, fs)}"


def test_refusal_table_has_both_sides():
    verdicts = {label: accepted(orc.make_args(**kw), fs) for label, kw, fs in BOUNDARY}
    for yes, no in (("cmax 255", "cmax 256"), ("nBands 100", "nBands 101"), ("P 100", "P 100.5"), ("bound 1024", "bound 1025"),
                    ("cmax 255 as minCoeff", "cmax 256 as minCoeff")):
        assert verdicts[yes] and not verdicts[no], (yes, no)
    assert not verdicts["cmax 255.5"] and not verdicts["minCoeff > maxCoeff past the bound"] and verdicts["minCoeff > maxCoeff"]


def test_refusal_rule_sweep():
    """Seeded arguments on both sides of every boundary: the library refuses exactly what the restated rule refuses."""
    rs = np.random.RandomState(2024)
    seen = {True: 0, False: 0}
    for _ in range(3000):
        nb = int(rs.choice([1, 2, 3, 4, 5, 6, 25, 26, 51, 52, 99, 100, 101, 102], p=[0.08] * 12 + [0.02, 0.02]))
        lim = MAX_CASCADE // nb - 1
        c1 = float(rs.choice([rs.randint(1, min(lim, 255) + 1), 1, min(lim, 255), lim, lim + 0.5, lim + 1, 0.5, 0.99, 254.5, 255,
                              255.5, 256], p=[0.25, 0.1, 0.2, 0.1] + [0.05] * 6 + [0.025, 0.025]))
        c2 = float(rs.choice([rs.randint(1, min(lim, 255) + 1), 1, 2, min(lim, 255)]))
        if rs.rand() < 0.5:
            c1, c2 = c2, c1
        a = orc.make_args(nBands=nb, N_f=int(rs.choice([1, 2, 17, 40, 300, 0], p=[0.2] * 4 + [0.15, 0.05])), minCoeff=c1,
                          maxCoeff=c2, P=float(rs.choice([0, 1e-9, 50, 99.99, 100, 100.0000001, 100.5, -1e-9],
                                                          p=[0.17] * 5 + [0.05] * 3)))
        fs = float(rs.choice([16000, 8000, 44100, 0, -1], p=[0.32, 0.32, 0.32, 0.02, 0.02]))
        want = accepted(a, fs)
        seen[want] += 1
        for algo in (1, 3, 5):
            assert (devplan_bytes(a, fs, algo) > 0) == want, vars(a)
    assert min(seen.values()) > 300, seen


def test_error_string_states_the_domain():
    msg = _lib.load().rb_error_string(-6).decode()
    for part in ("nBands 1-100", "P 0-100", "255", "1024"):
        assert part in msg, msg


# ---------------------------------------------------------------------------------------------------------------------------
# the edge table
# ---------------------------------------------------------------------------------------------------------------------------
SHORT = (7999, 1, 2, 33, 4097, 2561, 641)            # N_f >= 16 or cascades past 512 taps: the host reference is the cost
LENS = (16001, 1, 2, 33, 4097, 7999, 12345)
LONG = (49153, 65537, 1, 3, 2561)
CLAMP_FS = (8000, 22050, 44100, 48000)


@dataclass
class Edge:
    name: str
    kw: dict
    algos: Tuple[int, ...]
    lengths: Tuple[int, ...] = LENS
    sr: int = 16000
    hand: bool = False  # also hand-built rows with edge taps through LnL and algo 5
    args: object = field(init=False)

    def __post_init__(self):
        self.args = orc.make_args(**self.kw)

    def seeds(self):
        base = zlib.crc32(self.name.encode())
        return [(base + 7919 * u) % 2 ** 32 for u in range(len(self.lengths))]


def clamp_kw(fs):
    return dict(minF=0, maxF=fs / 2, minBW=fs / 16, maxBW=fs)


EDGES = [
    Edge("nb5_nf24", dict(N_f=24), (1, 5, 6), SHORT, hand=True),
    Edge("nf16", dict(N_f=16), (1, 5), SHORT, hand=True),
    Edge("nf17", dict(N_f=17), (1, 5), SHORT, hand=True),
    Edge("nb1_nf40", dict(nBands=1, N_f=40), (1, 5, 8), SHORT, hand=True),
    Edge("nb26_nf7", dict(nBands=26, minCoeff=1, maxCoeff=37, N_f=7), (1, 4), SHORT),
    Edge("nb60", dict(nBands=60, minCoeff=1, maxCoeff=15, N_f=3), (1, 3, 5), SHORT),
    Edge("nb100", dict(nBands=100, minCoeff=1, maxCoeff=9, N_f=2), (3, 4, 6), SHORT),
    Edge("stage255", dict(nBands=4, minCoeff=200, maxCoeff=255), (1, 3), SHORT),
] + [Edge(f"clamps_{fs}", clamp_kw(fs), (1, 3), LENS, sr=fs) for fs in CLAMP_FS] + [
    Edge(f"gains_gsd{g}", dict(minG=3, maxG=-2, minBiasLinNonLin=10, maxBiasLinNonLin=30, SNRmin=12, SNRmax=12, g_sd=g),
         (1, 2, 4, 5, 7), LENS) for g in (0, 10)
] + [
    Edge("p0", dict(P=0), (2, 5), LONG),
    Edge("p100", dict(P=100), (2, 5, 8), LONG),
]
EDGE_IDS = [e.name for e in EDGES]
EDGE = {e.name: e for e in EDGES}


def lnl_bands(a, fs, seed):
    """numpy's draws of the LnL filters right after np.random.seed(seed): per filter the (f1, f2, c) of every band, before the
    clamps, and the clamp hits (f1 <= 0, f2 >= fs/2)."""
    rs = np.random.RandomState(seed)
    filters, lo_hits, hi_hits = [], 0, 0
    for _ in range(a.N_f):
        bands = []
        for _ in range(a.nBands):
            fc, bw, c = rs.uniform(a.minF, a.maxF), rs.uniform(a.minBW, a.maxBW), int(rs.uniform(a.minCoeff, a.maxCoeff))
            c += c % 2 == 0
            bands.append((fc - bw / 2, fc + bw / 2, c))
            lo_hits += fc - bw / 2 <= 0
            hi_hits += fc + bw / 2 >= fs / 2
        rs.uniform()  # the gain
        filters.append(bands)
    return filters, lo_hits, hi_hits


def clamp_hits(e):
    lo = hi = 0
    for s in e.seeds():
        _, a, b = lnl_bands(e.args, e.sr, s)
        lo, hi = lo + a, hi + b
    return lo, hi


# ---------------------------------------------------------------------------------------------------------------------------
# E. the edge table reaches what it claims (CPU)
# ---------------------------------------------------------------------------------------------------------------------------
def test_edge_sets_are_accepted():
    for e in EDGES:
        assert accepted(e.args, e.sr), e.name
        assert devplan_bytes(e.args, e.sr) > 0, e.name
        assert max(e.args.maxF, e.args.minF) <= e.sr / 2, e.name


def test_edge_table_reaches_its_regimes():
    lnl = [e for e in EDGES if set(e.algos) & plans.ALGO_USES_LNL]
    regimes = {filters_per_window(e.args.nBands) for e in lnl if e.args.N_f > filters_per_window(e.args.nBands)}
    assert 1 in regimes and 32 in regimes and any(2 <= r <= 19 for r in regimes), regimes
    assert windows(EDGE["nb5_nf24"].args) == 2 and windows(EDGE["nb1_nf40"].args) == 2 and windows(EDGE["nb26_nf7"].args) == 3
    assert {e.args.N_f for e in lnl} >= {16, 17}
    assert EDGE["nf16"].args.N_f == SUPPORT_FILTERS and EDGE["nf17"].args.N_f == SUPPORT_FILTERS + 1
    # the last word the SSI draw reads, word(per + 1), at nBands = 100: 603 of the 624 a window may address
    assert per_filter(EDGE["nb100"].args.nBands) + 1 == 603 and set(EDGE["nb100"].algos) >= {3, 4, 6}
    a = EDGE["stage255"].args
    assert a.nBands * (math.ceil(max(a.minCoeff, a.maxCoeff)) + 1) == MAX_CASCADE
    stages = [c for s in EDGE["stage255"].seeds() for bands in lnl_bands(a, 16000, s)[0] for _, _, c in bands]
    assert max(stages) == MAX_STAGE, "no 255-tap stage drawn"
    assert {EDGE["p0"].args.P, EDGE["p100"].args.P} == {0, 100}
    assert max(EDGE["p100"].lengths) > 65536 and 49153 in EDGE["p100"].lengths


@pytest.mark.parametrize("fs", CLAMP_FS)
def test_clamp_sets_hit_both_branches(fs):
    e = EDGE[f"clamps_{fs}"]
    lo, hi = clamp_hits(e)
    total = len(e.seeds()) * e.args.N_f * e.args.nBands
    print(f"clamps at {fs} Hz: f1 <= 0 in {lo}, f2 >= fs/2 in {hi} of {total} bands")
    assert lo > 0 and hi > 0 and lo + hi > total // 2


def test_band_replay_is_numpys_draw():
    """The replay behind the counts above gives numpy's own tap counts (sum of the stages minus the overlaps)."""
    for e in EDGES:
        if not set(e.algos) & plans.ALGO_USES_LNL:
            continue
        s = e.seeds()[0]
        filters, _, _ = lnl_bands(e.args, e.sr, s)
        bp = plans.draw_batch([5], e.sr, e.args, 1, seeds=[s])
        want = [sum(c for _, _, c in bands) - (e.args.nBands - 1) for bands in filters]
        assert np.diff(bp.lnl_tap_off).tolist() == want, e.name


# ---- hand-built rows: every edge tap of a bank of more than 16 filters --------------------------------------------------
HAND_AMP = 1.2
HAND_KS = (1, 2, 3, 5, 24, 25, 48, 49, 97, 161)


def hand_rows(e):
    """Rows of amplitude 1.2 whose filter f has edge taps scaled by 1.2^-(f+1), so that every power contributes alike."""
    rs = np.random.RandomState(zlib.crc32(e.name.encode()) % 2 ** 31)
    rows = []
    for r, L in enumerate((1201, 97, 640)):
        x = (HAND_AMP * rs.uniform(-1, 1, L)).astype(np.float32)
        lnl = [(edge_taps(rs, HAND_KS[(3 * r + f) % len(HAND_KS)]) * HAND_AMP ** -(f + 1)).astype(np.float32).astype(np.float64)
               for f in range(e.args.N_f)]
        row = Row(x=x, lnl=lnl)
        n = int(rs.randint(1, L // 3 + 2))
        row.isd_idx = rs.permutation(L)[:n].astype(np.int64)
        row.isd_fr = (2 * rs.rand(n) - 1) * (2 * rs.rand(n) - 1)
        rows.append(row)
    return rows


@pytest.mark.parametrize("name", [e.name for e in EDGES if e.hand])
def test_hand_rows_bound_sees_every_edge_tap(name):
    """Zeroing the first or the last tap of any filter of the bank moves the float64 LnL reference by at least 10 tol."""
    weakest, checked = np.inf, 0
    for row in hand_rows(EDGE[name])[:2]:
        y, tol = reference(row, 1, bank_c(row))
        for label, raw, _ in edge_mutations(row, 1):
            ym, _ = reference(row, 1, bank_c(row), raw=raw)
            weakest = min(weakest, ratio(np.abs(ym - y), tol))
            checked += 1
    print(f"{name}: {checked} edge taps, weakest moves the reference by {weakest:.1f} tol")
    assert checked >= 2 * EDGE[name].args.N_f and weakest >= 10.0


# ---------------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def eng():
    torch = pytest.importorskip("torch")
    from scl_deepfake_audio_detection_b200.engine import Engine
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    e = Engine(0)
    yield e
    e.set_tap_trim(True)


@pytest.fixture
def g_sd(monkeypatch):
    """Sets the ISD gain the float64 reference of test_gpu_fir_bank applies."""
    return lambda v: monkeypatch.setattr(fir_bank, "G_SD", float(v))


def waves_for(lengths, seed):
    rs = np.random.RandomState(seed)
    return [((0.9 if u % 2 else 0.3) * rs.uniform(-1, 1, n)).astype(np.float32) for u, n in enumerate(lengths)]


def device_plan(eng, lengths, seeds, sr, args, algo):
    import torch
    ld = plans.padded_ld(max(lengths))
    ln = torch.tensor(list(lengths), dtype=torch.int32, device=eng.device)
    dp = eng.draw_device_plan(ln, np.asarray(seeds, np.uint32), sr, args, algo, ld)
    torch.cuda.synchronize()
    return dp, eng.download_plan(dp)


def same_plan(got, ref, algo, tap_tol=None):
    """_same_plan; the ISD gain only where the plan carries impulses (a device plan always holds the argument, numpy's plan
    only once ISD drew). tap_tol (per tap, see design_tolerance) replaces the 1-ulp rule for the taps."""
    if algo not in plans.ALGO_USES_ISD:
        ref = dataclasses.replace(ref, g_sd=got.g_sd)
    if tap_tol is not None:
        for name, tol in tap_tol.items():
            err = np.abs(getattr(got, name).astype(np.float64) - getattr(ref, name))
            assert np.all(err <= tol), f"{name}: {np.max(err / tol):.3g} x the tolerance"
            ref = dataclasses.replace(ref, **{name: getattr(got, name)})
    _same_plan(got, ref)


def _design(bands, gain_db, fs, exact):
    """genNotchCoeffs on drawn bands; `exact` takes each stage's DC sum with math.fsum instead of numpy's pairwise sum."""
    from scipy import signal
    casc = np.ones(1)
    for lo, hi, c in bands:
        h = signal.firwin(c, [lo, hi], window="hamming", fs=fs, scale=False)
        casc = np.convolve(h / (math.fsum(h) if exact else np.sum(h)), casc)
    _, resp = signal.freqz(casc, 1, fs=fs)
    return 10.0 ** (gain_db / 20) * casc / np.amax(np.abs(resp))


def _draw_bands(rs, a, fs, minG, maxG):
    bands = []
    for _ in range(a.nBands):
        fc, bw, c = rs.uniform(a.minF, a.maxF), rs.uniform(a.minBW, a.maxBW), int(rs.uniform(a.minCoeff, a.maxCoeff))
        c += c % 2 == 0
        lo, hi = fc - bw / 2, fc + bw / 2
        bands.append((lo if lo > 0 else 1 / 1000, hi if hi < fs / 2 else fs / 2 - 1 / 1000, c))
    return bands, rs.uniform(minG, maxG)


def design_tolerance(lengths, fs, a, algo, seeds):
    """Per-tap tolerance of the device's float64 design against numpy's: one float32 ulp of the filter's largest tap, plus 32
    times the most any tap of numpy's own design of the filter moves by when its stages' DC sums are taken exactly. Far from the
    defaults a cascade of many nearly all-stop stages (wide bands, few taps: DC sums down to 1e-7) turns the rounding order of
    those sums into visible tap differences; there numpy itself does not determine the taps any better, and the device
    (sequential sums) was found within 8 times that spread of numpy (pairwise sums) on 400 random plans. Well-conditioned
    plans keep one ulp of the peak."""
    tol = {"lnl_taps": [], "ssi_taps": []}

    def add(name, bands, g):
        t, e = _design(bands, g, fs, False), _design(bands, g, fs, True)
        tol[name].append(np.full(t.shape, np.spacing(np.float32(np.abs(t).max())) + 32.0 * np.abs(t - e).max()))

    for L, s in zip(lengths, seeds):
        rs = np.random.RandomState(int(s))
        if algo in plans.ALGO_USES_LNL:
            for f in range(a.N_f):
                lo, hi = (a.minG, a.maxG) if f == 0 else (a.minG - a.minBiasLinNonLin, a.maxG - a.maxBiasLinNonLin)
                add("lnl_taps", *_draw_bands(rs, a, fs, lo, hi))
        if algo in plans.ALGO_USES_ISD:
            n = int(L * (rs.uniform(0, a.P) / 100))
            rs.permutation(L)
            rs.rand(n), rs.rand(n)
        if algo in plans.ALGO_USES_SSI:
            rs.normal(0, 1, L)
            add("ssi_taps", *_draw_bands(rs, a, fs, a.minG, a.maxG))
    return {k: np.concatenate(v) for k, v in tol.items() if v}


def rows_of(bp, waves):
    """Rows of the fir-bank reference holding exactly what the device plan holds."""
    rows = []
    for u, x in enumerate(waves):
        L = x.shape[0]
        row = Row(x=x)
        if bp.lnl_tap_off is not None:
            o = bp.lnl_tap_off
            row.lnl = [bp.lnl_taps[o[u * bp.n_f + f]:o[u * bp.n_f + f + 1]].astype(np.float64) for f in range(bp.n_f)]
        if bp.isd_off is not None:
            row.isd_idx = bp.isd_idx[bp.isd_off[u]:bp.isd_off[u + 1]].astype(np.int64)
            row.isd_fr = bp.isd_fr[bp.isd_off[u]:bp.isd_off[u + 1]]
        if bp.ssi_tap_off is not None:
            row.noise = bp.ssi_noise[u, :L].copy()
            row.ssi_taps = bp.ssi_taps[bp.ssi_tap_off[u]:bp.ssi_tap_off[u + 1]].astype(np.float64)
            row.snr = float(bp.ssi_snr_db[u])
        rows.append(row)
    return rows


def run_plan(eng, algo, waves, dp):
    import torch
    x, ln = eng.pack_waveforms(waves, ld=dp.ld)
    y = eng.process(algo, x, ln, dp)
    torch.cuda.synchronize()
    y = y.cpu().numpy()
    return [y[u, :w.shape[0]] for u, w in enumerate(waves)]


def check_results(eng, algo, args, sr, waves, seeds, dp, bp):
    """The dispatcher on a device plan: ISD alone bit for bit against the oracle, the FIR algos within the per-sample bound
    of the float64 reference on the same plan, algos 7 and 8 within the suite's 1e-5 of the oracle. Returns the largest
    err/tol."""
    got = run_plan(eng, algo, waves, dp)
    worst = 0.0
    if algo in (2, 7, 8):
        for u, (x, g) in enumerate(zip(waves, got)):
            np.random.seed(int(seeds[u]))
            want = orc.process(x, sr, args, algo)
            if algo == 2:
                assert np.array_equal(g, want), f"algo 2 row {u}: ISD must equal the oracle bit for bit"
            else:
                assert np.max(np.abs(g - want)) <= 1e-5 * max(1.0, float(np.abs(want).max())), f"algo {algo} row {u}"
        return worst
    for u, (row, g) in enumerate(zip(rows_of(bp, waves), got)):
        y, tol = reference(row, algo, bank_c(row))
        q = ratio(np.abs(g.astype(np.float64) - y), tol)
        assert q <= 1.0, f"algo {algo} row {u} (L={row.x.shape[0]}): err/tol {q:.3g}"
        worst = max(worst, q)
    return worst


def check_trim(eng, algo, waves, dp, bp):
    """Trimming on against off: bit-identical past 16 filters (the bank must not trim), within the bound of
    test_tap_support.test_trim_on_against_off up to 16. Returns whether the two runs differ."""
    eng.set_tap_trim(False)
    try:
        full = run_plan(eng, algo, waves, dp)
    finally:
        eng.set_tap_trim(True)
    trim = run_plan(eng, algo, waves, dp)
    n_f = bp.n_f
    K = np.diff(bp.lnl_tap_off).reshape(bp.B, n_f)
    l1 = np.add.reduceat(np.abs(bp.lnl_taps.astype(np.float64)), bp.lnl_tap_off[:-1]).reshape(bp.B, n_f)
    l1[K == 0] = 0.0
    differs = False
    for u, (f, t) in enumerate(zip(full, trim)):
        diff = np.abs(t.astype(np.float64) - f)
        differs |= bool(np.any(diff > 0))
        if n_f > SUPPORT_FILTERS:
            assert np.array_equal(t, f), f"row {u}: a bank of {n_f} filters must run every tap"
            continue
        amax = float(np.abs(waves[u]).max())
        S = sum(l1[u, k] * amax ** (k + 1) for k in range(n_f))
        assert diff.max() <= 3.0 * 2.0 * (EPS + 2 * C_DENSE * U) * S, (u, diff.max())
        assert diff.max() <= 1e-5 * max(1.0, float(np.abs(f).max()))
    return differs


@pytest.mark.gpu
@pytest.mark.parametrize("name", EDGE_IDS)
def test_edge_set(eng, g_sd, name):
    e = EDGE[name]
    a, seeds = e.args, e.seeds()
    g_sd(a.g_sd)
    waves = waves_for(e.lengths, seeds[0])
    lo, hi = clamp_hits(e)
    report = []
    for algo in e.algos:
        dp, got = device_plan(eng, e.lengths, seeds, e.sr, a, algo)
        ref = plans.draw_batch(list(e.lengths), e.sr, a, algo, seeds=seeds, ld=dp.ld)
        same_plan(got, ref, algo)
        worst = check_results(eng, algo, a, e.sr, waves, seeds, dp, got)
        trimmed = ""
        if algo in (1, 5):
            trimmed = f", trim on/off {'differ' if check_trim(eng, algo, waves, dp, got) else 'identical'}"
        report.append(f"algo {algo}: err/tol {worst:.3f}{trimmed}")
    if e.hand:
        import torch
        for algo in (1, 5):
            rows = hand_rows(e)
            got = fir_bank.run_rows(eng, algo, rows)
            worst = 0.0
            for r, (row, g) in enumerate(zip(rows, got)):
                y, tol = reference(row, algo, bank_c(row))
                q = ratio(np.abs(g.astype(np.float64) - y), tol)
                assert q <= 1.0, f"hand-built row {r}, algo {algo}: err/tol {q:.3g}"
                worst = max(worst, q)
            torch.cuda.synchronize()
            report.append(f"hand algo {algo}: err/tol {worst:.3f}")
    wn = windows(a) if set(e.algos) & plans.ALGO_USES_LNL else 0
    print(f"{name}: {wn} LnL window(s) of {filters_per_window(a.nBands)}, bank "
          f"{'trims' if a.N_f <= SUPPORT_FILTERS else 'runs every tap'}, clamp hits f1 {lo} f2 {hi}; " + "; ".join(report))


# ---- C. property sweep over the whole domain ------------------------------------------------------------------------------
hypothesis = pytest.importorskip("hypothesis")
from hypothesis import HealthCheck, given, settings, strategies as st  # noqa: E402

SWEEP_FS = (16000,) + CLAMP_FS


@st.composite
def _domain_cases(draw):
    fs = draw(st.sampled_from(SWEEP_FS))
    nb = draw(st.integers(1, 100))
    lim = min(MAX_STAGE, MAX_CASCADE // nb - 1)
    outside = draw(st.sampled_from([None] * 7 + ["nBands", "cmax", "P", "bound"]))
    c1, c2 = draw(st.integers(1, lim)), draw(st.integers(1, lim))
    P = draw(st.integers(0, 100))
    if outside == "nBands":
        nb = 101
        c1 = c2 = draw(st.integers(1, 9))
    elif outside == "cmax":
        c1 = draw(st.sampled_from([255.5, 256, 300]))
        nb = min(nb, 3)
    elif outside == "P":
        P = draw(st.sampled_from([100.5, 101, 150]))
    elif outside == "bound":
        nb = max(nb, 5)
        c1 = MAX_CASCADE // nb  # nb * (c1 + 1) > 1024
    minF = draw(st.integers(0, fs // 2 - 1))
    minBW = draw(st.integers(1, fs // 4))
    args = orc.make_args(
        N_f=draw(st.integers(1, 40)), nBands=nb, minF=minF, maxF=draw(st.integers(minF + 1, fs // 2)),
        minBW=minBW, maxBW=draw(st.integers(minBW, fs)), minCoeff=c1, maxCoeff=c2,
        minG=draw(st.integers(-10, 10)), maxG=draw(st.integers(-10, 10)),
        minBiasLinNonLin=draw(st.integers(0, 30)), maxBiasLinNonLin=draw(st.integers(0, 30)),
        P=P, g_sd=draw(st.integers(0, 10)), SNRmin=draw(st.integers(-5, 40)), SNRmax=draw(st.integers(-5, 40)))
    lens = draw(st.lists(st.integers(1, 20000), min_size=1, max_size=4))
    algo = draw(st.integers(1, 8))
    seed = draw(st.integers(0, 2 ** 32 - 1))
    return args, fs, lens, algo, seed, outside


@pytest.mark.gpu
@settings(max_examples=50, deadline=None, derandomize=True, suppress_health_check=list(HealthCheck))
@given(_domain_cases())
def test_device_planner_property_sweep(eng, g_sd, case):
    """Device plans equal numpy's over the whole accepted domain; the dispatcher matches the oracle where the float64 reference
    is cheap; arguments outside the domain are refused although numpy draws them."""
    args, fs, lens, algo, seed, outside = case
    seeds = [(seed + 7919 * u) % 2 ** 32 for u in range(len(lens))]
    assert accepted(args, fs) == (outside is None)
    ref = plans.draw_batch(lens, fs, args, algo, seeds=seeds, ld=plans.padded_ld(max(lens)))
    if outside is not None:
        with pytest.raises(_lib.RawBoostLibraryError):
            device_plan(eng, lens, seeds, fs, args, algo)
        return
    dp, got = device_plan(eng, lens, seeds, fs, args, algo)
    same_plan(got, ref, algo, design_tolerance(lens, fs, args, algo, seeds))
    cost = sum(L * (np.diff(ref.lnl_tap_off).reshape(ref.B, -1)[u].sum() if ref.lnl_tap_off is not None else 0)
               + L * (np.diff(ref.ssi_tap_off)[u] if ref.ssi_tap_off is not None else 0) for u, L in enumerate(lens))
    if cost <= 2e8:
        g_sd(args.g_sd)
        check_results(eng, algo, args, fs, waves_for(lens, seed % 2 ** 31), seeds, dp, got)


# ---- D. items at non-default arguments ------------------------------------------------------------------------------------
ITEM_SETS = {"nb5_nf24": (dict(N_f=24), 16000), "nb60": (dict(nBands=60, minCoeff=1, maxCoeff=15, N_f=3), 22050)}


def _check_item_views(data, labels, out_len, items, n_add, nvoc):
    data, labels, out_len = data.cpu().numpy(), labels.cpu().numpy(), out_len.cpu().numpy()
    for g, (_, ref, lab) in enumerate(items):
        n = ref.shape[0]
        assert int(out_len[g]) == n, g
        assert np.max(np.abs(data[g][:n].astype(np.float64) - ref), initial=0.0) <= 1e-5, g
        copies = [0] + list(range(2, 2 + n_add + nvoc))
        assert np.array_equal(data[g][:n, copies], ref[:, copies]), g
        assert not np.any(data[g][n:]), "nothing is written past out_len"
        assert np.array_equal(labels[g], lab), g


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(ITEM_SETS))
def test_items_at_nondefault_arguments(eng, name):
    """SeededItemBatcher and StreamItemBatcher against Dataset_for items replayed by the oracle at the set's arguments and
    sample rate: views, labels and the stream state after each item / stream."""
    import torch
    from scl_deepfake_audio_detection_b200 import multiview
    kw, sr = ITEM_SETS[name]
    args = orc.make_args(**kw)
    nvoc, n_add, trim = 1, 1, 1000
    c = Corpus([1500, 2200, 900, 3001, 1000], nvoc, seed=len(name))
    dc = multiview.DeviceCorpus(c.ids, "/data", c.load, c.vocoders, engine=eng)
    ref_item = lambda idx: orc.dataset_item(idx, c.ids, c.load, args, c.vocoders, n_add, trim, sr=sr)  # noqa: E731

    seeded = multiview.SeededItemBatcher(args, dc, num_additional_real=n_add, trim_length=trim, wav_samp_rate=sr)
    indices, seeds = [0, 4, 2, 3, 1, 3], [11, 2 ** 32 - 1, 0, 77, 5, 1234]
    end = torch.empty((len(indices), 625), dtype=torch.int32, device=eng.device)
    _, data, labels, out_len = seeded.items(indices, seeds, end_state=end)
    torch.cuda.synchronize()
    items, states = [], []
    for idx, s in zip(indices, seeds):
        np.random.seed(s)
        items.append(ref_item(idx))
        states.append(np.random.get_state())
    _check_item_views(data, labels, out_len, items, n_add, nvoc)
    end = end.cpu().numpy()
    for g, st_ in enumerate(states):
        assert _same_stream(end[g], st_), g

    stream = multiview.StreamItemBatcher(args, dc, num_additional_real=n_add, trim_length=trim, wav_samp_rate=sr)
    index_lists = [[3, 0, 4], [1], [2, 2]]
    starts = [np.random.RandomState(900 + q).get_state() for q in range(len(index_lists))]
    ids, data, labels, out_len, ends = stream.items_streams(index_lists, starts)
    torch.cuda.synchronize()
    saved = np.random.get_state()
    items, finals = [], []
    try:
        for ix, st_ in zip(index_lists, starts):
            np.random.set_state(st_)
            items += [ref_item(i) for i in ix]
            finals.append(np.random.get_state())
    finally:
        np.random.set_state(saved)
    assert ids == [c.ids[i] for ix in index_lists for i in ix]
    _check_item_views(data, labels, out_len, items, n_add, nvoc)
    ends = ends.cpu().numpy()
    for q, st_ in enumerate(finals):
        assert _same_stream(ends[q], st_), q

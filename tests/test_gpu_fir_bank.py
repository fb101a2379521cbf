"""The FIR-bank kernel's LnL and SSI instantiations (rb_fir_bank.cu, TAIL_AFFINE and TAIL_SSI: 20 outputs per thread, six 4-tap
groups per body, their own segment reach and power staging, the fused tails) against the float64 oracle, with taps whose edges
matter; and every batched launcher across the 65 535-row grid split.

Why hand-built taps: the notch cascades of genNotchCoeffs are products of Hamming-windowed stages, so their first and last
taps are ~1e-20 of the largest, and a kernel that drops, duplicates or misaligns the taps at either end of a filter stays far
inside any tolerance with them. Here every filter gets random taps of unit variance scaled by 1/sqrt(K), with the first and last
at least half that size, at tap counts around the 4-tap group, the 24-tap body, the 512-tap segment and the restaged segments.

The bound is per sample and follows each stage's float32 arithmetic to first order from the float64 reference (u = 2^-24):
  LnL  tol = c u (S + mean S + |y| (S[p] + mean S)) / D + 2u |y|,  S = sum_f |b_f| * |x^p_f| in the closed-form alignment,
       D the normWav divisor (1 when idle), p the sample that sets it (the |y| term is the divisor's own error);
  ISD  the incoming bound times |1 + g_sd f_r| at an impulse (the gain it applies), over the second divisor, plus its roundings;
  SSI  the incoming bound, plus c u S_noise times the noise gain, plus the gain's relative error (from both norms) times the
       noise term, plus the roundings of the gain and of the final FMA.
c is 4 for the impulse probes (every output is a sum of at most N_f products) and 8 for dense inputs. On an NVIDIA B200 at a
1000 W power limit the largest err/tol per case was 0.19-0.34 for the probes, 0.15-0.29 for dense LnL and its chains, 0.64
for dense SSI and 0.19 for LnL -> ISD.
The CPU-only tests check, for every adversarial case, that zeroing the first or the last tap of any single filter moves the
float64 reference by at least 10 tol at some sample: the bound is tight enough to see every edge tap.
"""
import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np
import pytest

from oracle import rawboost_oracle as orc  # noqa: E402  (checker only)

U = 2.0 ** -24
C_PROBE = 4.0
C_DENSE = 8.0
G_SD = 2.0
TOL = 1e-5  # the suite's max-abs FIR tolerance, kept beside the per-sample bound
KS = [1, 2, 3, 4, 5, 7, 8, 9, 23, 24, 25, 27, 28, 29, 47, 48, 49, 511, 512, 513, 514, 1024, 1025, 1537, 2049]
DENSE_LENS = [1, 2, 5, 19, 20, 21, 2559, 2560, 2561, 5121, 7680, 64600, 70001]
SPLIT = 65535  # rows per launch of every batched launcher (gridDim.y)


# ---------------------------------------------------------------------------------------------------------------------------
# cases: one row = one utterance with its waveform and plan, float32 values held as float64 (what the kernel sees)
# ---------------------------------------------------------------------------------------------------------------------------
@dataclass
class Row:
    x: np.ndarray                                   # float32 [L]
    lnl: List[np.ndarray] = field(default_factory=list)
    isd_idx: Optional[np.ndarray] = None
    isd_fr: Optional[np.ndarray] = None
    noise: Optional[np.ndarray] = None              # float32 [L]
    ssi_taps: Optional[np.ndarray] = None
    snr: float = 0.0                                # float32-rounded


@dataclass
class Case:
    name: str
    algo: int
    rows: List[Row]
    c: float


def edge_taps(rs, K):
    """Unit-variance taps scaled by 1/sqrt(K), rounded to float32; the first and last are at least half the typical size."""
    b = rs.standard_normal(K)
    for i in (0, K - 1):
        if abs(b[i]) < 0.5:
            b[i] = 0.5 + rs.rand() if rs.rand() < 0.5 else -0.5 - rs.rand()
    return (b / np.sqrt(K)).astype(np.float32).astype(np.float64)


def probe_positions(L):
    """Spike positions of the impulse probes: the ends, the thread span (20), the warp span (640), the tile (2560), and
    positions whose response straddles a tile boundary or runs off either end of the row."""
    pos = [0, 1, L - 1, 19, 20, 21, 639, 640, 2559, 2560, 2561, 2560 - 300, 2560 + 300, 5120 - 700, 5120, 5121, 150, L - 151]
    return sorted({p for p in pos if 0 <= p < L})


def probe_cases():
    """Item 1: rows that are zero except for +-2 spikes spaced more than the row's longest filter apart, N_f in {1, 2, 5, 7}
    with tap counts mixed inside each utterance; every third row has its taps scaled by a power of two so that normWav idles."""
    cases = []
    lens = (7681, 5120, 2561, 7680)
    for n_f in (1, 2, 5, 7):
        rs = np.random.RandomState(1000 + n_f)
        rows, todo, r = [], {L: set(probe_positions(L)) for L in lens}, 0
        while r < -(-len(KS) // n_f) or any(todo.values()):  # every tap count, and every position at every length
            L = lens[r % 4]
            taps = [edge_taps(rs, KS[(r * n_f + f) % len(KS)]) for f in range(n_f)]
            reach = max(t.shape[0] for t in taps)
            spikes = []
            for p in sorted(todo[L]) + probe_positions(L):
                if all(abs(p - q) > reach for q in spikes):
                    spikes.append(p)
            todo[L] -= set(spikes)
            x = np.zeros(L, np.float32)
            x[spikes] = np.where(rs.rand(len(spikes)) < 0.5, -2.0, 2.0)
            row = Row(x=x, lnl=taps)
            if r % 3 == 2:  # normWav idle: exact power-of-two scaling keeps the float32 taps exact
                raw = lnl_raw(row)[0]
                s = 2.0 ** np.floor(np.log2(0.25 / max(np.abs(raw).max(), 1e-30)))
                row.lnl = [t * s for t in taps]
            rows.append(row)
            r += 1
        cases.append(Case(f"probe_nf{n_f}", 1, rows, C_PROBE))
    return cases


def dense_cases():
    """Item 2: dense inputs of amplitude 1.1-1.3 over the ragged lengths, for LnL, SSI and the chains. Filters of 1025 taps and
    more only on rows up to 7680 samples (the float64 host reference is the cost)."""
    cases = []
    for algo, n_f in ((1, 7), (3, 0), (4, 5), (5, 5), (6, 2)):
        rs = np.random.RandomState(2000 + algo)
        rows = []
        for r, L in enumerate(DENSE_LENS):
            def k_at(i):
                K = KS[i % len(KS)]
                return K if L <= 7680 or K <= 514 else KS[i % 17]
            amp = 1.1 + 0.2 * rs.rand()
            x = (amp * rs.uniform(-1, 1, L)).astype(np.float32)
            row = Row(x=x, lnl=[edge_taps(rs, k_at(r * max(n_f, 1) + 3 * f + algo)) for f in range(n_f)])
            if algo in (4, 5):
                n = int(rs.randint(0, max(1, L // 4)) if L > 1 else 1)
                row.isd_idx = rs.permutation(L)[:n].astype(np.int64)
                row.isd_fr = (2 * rs.rand(n) - 1) * (2 * rs.rand(n) - 1)
            if algo in (3, 4, 6):
                Ks = k_at(5 * r + 11)
                if r % 2:  # spike-train noise
                    noise = np.zeros(L)
                    noise[rs.rand(L) < 0.02] = 3.0
                    noise[0] = noise[L - 1] = -3.0
                    noise *= np.sign(rs.standard_normal(L))
                else:
                    noise = rs.standard_normal(L)
                row.noise = noise.astype(np.float32)
                row.ssi_taps = edge_taps(rs, Ks)
                row.snr = float(np.float32(rs.uniform(0, 20)))
            rows.append(row)
        cases.append(Case(f"dense_algo{algo}", algo, rows, C_DENSE))
    return cases


def isd_cases():
    """Item 3: LnL -> ISD (algo 5, the fused tail's in-place keep_hits path) on inputs with a large DC offset, so that the mean the
    tail removes and its first divisor are far from 0 and 1; impulses at mask-word, thread-span and tile boundaries, the ends and
    the LnL peak; a short row with every sample but the peak an impulse, and one with every sample."""
    rs = np.random.RandomState(3000)
    rows = []
    for r, (L, dc) in enumerate(((7681, 0.9), (5121, -0.8), (2561, 1.0), (97, 0.9), (61, -0.9))):
        x = (dc + 0.25 * rs.uniform(-1, 1, L)).astype(np.float32)
        row = Row(x=x, lnl=[edge_taps(rs, KS[(7 * r + 3 * f) % len(KS)] if L > 100 else 1 + (5 * r + 7 * f) % 48) for f in range(5)])
        y, _ = reference(row, 1, C_DENSE)
        peak = int(np.argmax(np.abs(y)))
        if L == 97:
            idx = np.array([p for p in range(L) if p != peak])
        elif L == 61:
            idx = np.arange(L)
        else:
            s = {31, 32, 63, 64, 0, L - 1, peak, 2559, 2560, 2561, 5119, 5120, 5121}
            s |= {p for k in range(20, L + 1, 20) for p in (k - 1, k)}
            idx = np.array(sorted(p for p in s if 0 <= p < L))
        idx = rs.permutation(idx)
        row.isd_idx = idx.astype(np.int64)
        row.isd_fr = (2 * rs.rand(idx.shape[0]) - 1) * (2 * rs.rand(idx.shape[0]) - 1)
        rows.append(row)
    return [Case("isd_dc", 5, rows, C_DENSE)]


# ---------------------------------------------------------------------------------------------------------------------------
# float64 reference with a per-sample bound
# ---------------------------------------------------------------------------------------------------------------------------
def _fir(x, b):
    return orc.filter_fir_closed_form(x, b)


def lnl_raw(row):
    """(sum_f FIR(x^p_f, b_f), S): powers in float32 as the oracle forms them, filters and the sums in float64."""
    raw, S = np.zeros(row.x.shape[0]), np.zeros(row.x.shape[0])
    for f, t in enumerate(row.lnl):
        xp = np.power(row.x, f + 1)
        raw += _fir(xp, t)
        S += _fir(np.abs(xp.astype(np.float64)), np.abs(t))
    return raw, S


def lnl_stage(raw, S, c):
    cen = raw - raw.mean()
    pk = int(np.argmax(np.abs(cen))) if cen.size else 0
    D = abs(cen[pk]) if cen.size and abs(cen[pk]) > 1 else 1.0
    y = cen / D
    e = c * U * (S + (S.mean() if S.size else 0.0))
    if D > 1:
        e = e + np.abs(y) * e[pk]
    return y, e / D + 2 * U * np.abs(y)


def isd_stage(y, e, idx, fr):
    z = y.copy()
    z[idx] = y[idx] + G_SD * y[idx] * fr
    G = np.ones_like(y)
    G[idx] = np.abs(1 + G_SD * fr)
    ez = e * G
    ez[idx] += U * G_SD * np.abs(fr) * np.abs(y[idx])
    pk = int(np.argmax(np.abs(z)))
    D = abs(z[pk]) if abs(z[pk]) > 1 else 1.0
    out = z / D
    if D > 1:
        ez = ez + np.abs(out) * ez[pk]
    return out, ez / D + U * np.abs(z) / D + U * np.abs(out)


def ssi_stage(y, e, col, Sn, snr, c):
    """y + g col, g = ||y|| / (||col|| 10^(snr/20)): apply_ssi's peak normalisation of the coloured noise cancels in g."""
    g = np.linalg.norm(y) / (np.linalg.norm(col) * 10.0 ** (0.05 * snr))
    out = y + g * col
    ec = c * U * Sn
    rel = np.sum(np.abs(col) * ec) / np.sum(col * col) + np.sum(np.abs(y) * e) / max(np.sum(y * y), 1e-300) + 16 * U
    return out, e + g * ec + g * np.abs(col) * (rel + U) + U * np.abs(out)


def ssi_col(row):
    return _fir(row.noise, row.ssi_taps), _fir(np.abs(row.noise.astype(np.float64)), np.abs(row.ssi_taps))


def reference(row, algo, c, raw=None, col=None):
    """float64 result of `algo` on one row and its bound; `raw` / `col` replace the LnL sum / the coloured noise."""
    if algo in (1, 4, 5, 6):
        r, S = lnl_raw(row)
        y, e = lnl_stage(r if raw is None else raw, S, c)
    else:
        y, e = row.x.astype(np.float64), np.zeros(row.x.shape[0])
    if algo in (4, 5):
        y, e = isd_stage(y, e, row.isd_idx, row.isd_fr)
    if algo in (3, 4, 6):
        cl, Sn = ssi_col(row)
        y, e = ssi_stage(y, e, cl if col is None else col, Sn, row.snr, c)
    return y, e


def edge_delta(x, t, k):
    """Change of FIR(x, t) when tap k is zeroed: -t[k] x[n + (K+1)//2 - k]."""
    L, K = x.shape[0], t.shape[0]
    src = np.arange(L) + (K + 1) // 2 - k
    d = np.zeros(L)
    ok = (src >= 0) & (src < L)
    d[ok] = -t[k] * x[src[ok]].astype(np.float64)
    return d


def edge_mutations(row, algo):
    """(label, raw or None, col or None) for every filter whose first and last taps both reach an output of the row."""
    L = row.x.shape[0]
    reach = lambda K: (K + 1) // 2 < L and K - 1 - (K + 1) // 2 < L
    if algo in (1, 4, 5, 6):
        raw, _ = lnl_raw(row)
        for f, t in enumerate(row.lnl):
            if reach(t.shape[0]):
                for k in (0, t.shape[0] - 1):
                    yield f"lnl f{f} K={t.shape[0]} tap {k}", raw + edge_delta(np.power(row.x, f + 1), t, k), None
    if algo in (3, 4, 6) and reach(row.ssi_taps.shape[0]):
        col, _ = ssi_col(row)
        t = row.ssi_taps
        for k in (0, t.shape[0] - 1):
            yield f"ssi K={t.shape[0]} tap {k}", None, col + edge_delta(row.noise, t, k)


def ratio(err, tol):
    """max err / tol; a sample with zero tolerance must be exact."""
    err, tol = np.asarray(err, np.float64), np.asarray(tol, np.float64)
    if err.size == 0:
        return 0.0
    with np.errstate(divide="ignore", invalid="ignore"):
        q = np.where(tol > 0, err / tol, np.where(err > 0, np.inf, 0.0))
    return float(q.max())


CASES = probe_cases() + dense_cases() + isd_cases()
CASE_IDS = [c.name for c in CASES]


# ---------------------------------------------------------------------------------------------------------------------------
# CPU only: the reference is the oracle, and the bound sees every edge tap
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_reference_is_the_oracle(case):
    """The restated reference equals the oracle's apply_lnl / apply_isd / apply_ssi chain on the float32 values."""
    for row in case.rows[:: max(1, len(case.rows) // 6)]:
        if row.x.shape[0] > 20000:
            continue
        y, _ = reference(row, case.algo, case.c)
        # SSI alone: float64 input, so that ||x|| is not rounded to float32 (the kernel sums its squares in double);
        # LnL keeps the float32 input: its powers are float32, as the kernel forms them
        want = row.x.astype(np.float64)
        if case.algo in (1, 4, 5, 6):
            want = orc.apply_lnl(row.x, orc.LnLPlan(taps=row.lnl))
        if case.algo in (4, 5):
            want = orc.apply_isd(want, orc.ISDPlan(idx=row.isd_idx, f_r=row.isd_fr), G_SD)
        if case.algo in (3, 4, 6):
            want = orc.apply_ssi(want, orc.SSIPlan(noise=row.noise.astype(np.float64), taps=row.ssi_taps, snr_db=row.snr))
        assert np.max(np.abs(y - want)) <= 1e-12 * max(1.0, np.abs(want).max())


@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_bound_sees_every_edge_tap(case):
    """Zeroing the first or the last tap of any single filter moves the float64 reference by at least 10 tol at some sample
    (filters whose edge taps cannot reach an output of the row are skipped: nothing can see them)."""
    checked, weakest = 0, (np.inf, "")
    for r, row in enumerate(case.rows):
        y, tol = reference(row, case.algo, case.c)
        for label, raw, col in edge_mutations(row, case.algo):
            ym, _ = reference(row, case.algo, case.c, raw=raw, col=col)
            q = ratio(np.abs(ym - y), tol)
            weakest = min(weakest, (q, f"row {r} (L={row.x.shape[0]}) {label}"))
            checked += 1
    print(f"{case.name}: {checked} edge taps, weakest moves the reference by {weakest[0]:.1f} tol at {weakest[1]}")
    assert checked >= len(case.rows)
    assert weakest[0] >= 10.0, weakest


def test_probe_cases_cover_the_tap_counts_and_positions():
    for case in CASES[:4]:
        assert {t.shape[0] for row in case.rows for t in row.lnl} == set(KS), case.name
        for row in case.rows:
            spikes = np.flatnonzero(row.x)
            reach = max(t.shape[0] for t in row.lnl)
            assert spikes.size and np.all(np.diff(spikes) > reach) and np.all(np.abs(row.x[spikes]) == 2.0)
    probes = CASES[:4]
    hit = {(row.x.shape[0], int(p)) for case in probes for row in case.rows for p in np.flatnonzero(row.x)}
    for L in (7681, 5120, 2561, 7680):
        assert {(L, p) for p in probe_positions(L)} <= hit, L
    peaks = [np.abs(raw - raw.mean()).max() for raw in (lnl_raw(row)[0] for case in probes for row in case.rows)]
    assert min(peaks) < 1 < max(peaks)  # rows where normWav idles and rows where it divides


# ---------------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def eng():
    torch = pytest.importorskip("torch")
    from scl_deepfake_audio_detection_b200.engine import Engine
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return Engine(0)


def pack_rows(rows, ld=None):
    from scl_deepfake_audio_detection_b200 import plans
    ups = []
    for row in rows:
        up = plans.UtterancePlan(length=row.x.shape[0], g_sd=G_SD)
        if row.lnl:
            up.lnl_taps = row.lnl
        if row.isd_idx is not None:
            up.isd_idx, up.isd_fr = row.isd_idx, row.isd_fr
        if row.noise is not None:
            up.ssi_noise, up.ssi_taps, up.ssi_snr_db = row.noise, row.ssi_taps, row.snr
        ups.append(up)
    return plans.pack(ups, ld=ld)


def run_rows(eng, algo, rows, ld=None):
    import torch
    bp = pack_rows(rows, ld)
    x, ln = eng.pack_waveforms([r.x for r in rows], ld=bp.ld)
    y = eng.process(algo, x, ln, eng.upload_plan(bp))
    torch.cuda.synchronize()
    y = y.cpu().numpy()
    return [y[u, :r.x.shape[0]] for u, r in enumerate(rows)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_fir_bank_within_bound(eng, case):
    """Every sample of every row within the per-sample bound of the float64 reference, and within the suite's 1e-5."""
    got = run_rows(eng, case.algo, case.rows)
    worst = (0.0, -1)
    for r, (row, g) in enumerate(zip(case.rows, got)):
        y, tol = reference(row, case.algo, case.c)
        q = ratio(np.abs(g.astype(np.float64) - y), tol)
        worst = max(worst, (q, r))
        assert q <= 1.0, f"{case.name} row {r} (L={row.x.shape[0]}): err/tol {q:.3g}"
        assert np.max(np.abs(g - y), initial=0.0) <= TOL * max(1.0, np.abs(y).max(initial=0.0))
    print(f"{case.name}: largest err/tol {worst[0]:.3f} (row {worst[1]})")


# ---- item 4: batches past the grid split --------------------------------------------------------------------------------
B_BIG = SPLIT + 3
LD_BIG = 64


@pytest.fixture(scope="module")
def big():
    """B = 65 538 rows of ld 64: lengths 1-64, distinct content, N_f = 2 filters of 1-40 taps, impulses, SSI noise and taps."""
    rs = np.random.RandomState(4000)
    B, ld = B_BIG, LD_BIG
    d = {"len": rs.randint(1, ld + 1, B).astype(np.int32)}
    d["len"][[0, 1, B - 1]] = [ld, 1, ld - 1]
    d["x"] = rs.uniform(-1.3, 1.3, (B, ld)).astype(np.float32)
    k = rs.randint(1, 41, 2 * B)
    d["lnl_off"] = np.concatenate([[0], np.cumsum(k)]).astype(np.int32)
    d["lnl_taps"] = (rs.standard_normal(int(k.sum())) / np.sqrt(np.repeat(k, k))).astype(np.float32)
    hit = (rs.rand(B, ld) < 0.2) & (np.arange(ld)[None, :] < d["len"][:, None])
    rr, cc = np.nonzero(hit)
    d["isd_off"] = np.concatenate([[0], np.cumsum(hit.sum(axis=1))]).astype(np.int32)
    d["isd_idx"] = cc.astype(np.int32)
    d["isd_fr"] = (2 * rs.rand(rr.size) - 1) * (2 * rs.rand(rr.size) - 1)
    d["noise"] = rs.standard_normal((B, ld)).astype(np.float32)
    ks = rs.randint(1, 41, B)
    d["ssi_off"] = np.concatenate([[0], np.cumsum(ks)]).astype(np.int32)
    d["ssi_taps"] = (rs.standard_normal(int(ks.sum())) / np.sqrt(np.repeat(ks, ks))).astype(np.float32)
    d["snr"] = rs.uniform(5, 30, B).astype(np.float32)
    d["rows"] = sorted({0, 1, *range(SPLIT - 2, B)} | set(rs.randint(0, B, 8).tolist()))
    return d


def big_row(d, u):
    L = int(d["len"][u])
    o, i, s = d["lnl_off"], d["isd_off"], d["ssi_off"]
    return Row(x=d["x"][u, :L].copy(), lnl=[d["lnl_taps"][o[2 * u + f]:o[2 * u + f + 1]].astype(np.float64) for f in range(2)],
               isd_idx=d["isd_idx"][i[u]:i[u + 1]].astype(np.int64), isd_fr=d["isd_fr"][i[u]:i[u + 1]],
               noise=d["noise"][u, :L].copy(), ssi_taps=d["ssi_taps"][s[u]:s[u + 1]].astype(np.float64), snr=float(d["snr"][u]))


def big_plan(d):
    from scl_deepfake_audio_detection_b200 import plans
    return plans.BatchPlan(B=B_BIG, ld=LD_BIG, lengths=d["len"], n_f=2, lnl_taps=d["lnl_taps"], lnl_tap_off=d["lnl_off"],
                           isd_off=d["isd_off"], isd_idx=d["isd_idx"], isd_fr=d["isd_fr"], g_sd=G_SD, ssi_noise=d["noise"],
                           ssi_taps=d["ssi_taps"], ssi_tap_off=d["ssi_off"], ssi_snr_db=d["snr"])


def _beyond_untouched(out, ln, sentinel):
    import torch
    past = torch.arange(out.shape[1], device=out.device)[None, :] >= ln[:, None].long()
    return bool(torch.all(out[past] == sentinel))


@pytest.mark.gpu
def test_filter_fir_past_the_grid_split(eng, big):
    import torch
    d = big
    x, ln = torch.from_numpy(d["x"]).cuda(), torch.from_numpy(d["len"]).cuda()
    taps, off = torch.from_numpy(d["ssi_taps"]).cuda(), torch.from_numpy(d["ssi_off"]).cuda()
    out = torch.full_like(x, 7.0)
    eng.filter_fir(x, ln, taps, off, out=out)
    torch.cuda.synchronize()
    assert _beyond_untouched(out, ln, 7.0)
    y = out.cpu().numpy()
    rows = d["rows"]
    sub = np.ascontiguousarray(d["x"][rows])
    sk = [d["ssi_taps"][d["ssi_off"][u]:d["ssi_off"][u + 1]] for u in rows]
    small = eng.filter_fir(torch.from_numpy(sub).cuda(), torch.from_numpy(d["len"][rows]).cuda(), torch.from_numpy(np.concatenate(sk)).cuda(),
                           torch.from_numpy(np.concatenate([[0], np.cumsum([t.size for t in sk])]).astype(np.int32)).cuda()).cpu().numpy()
    for j, u in enumerate(rows):
        L, t = int(d["len"][u]), sk[j].astype(np.float64)
        assert np.array_equal(y[u, :L], small[j, :L]), u
        ref = _fir(d["x"][u, :L], t)
        S = _fir(np.abs(d["x"][u, :L].astype(np.float64)), np.abs(t))
        assert ratio(np.abs(y[u, :L] - ref), C_DENSE * U * S) <= 1.0, u


@pytest.mark.gpu
@pytest.mark.parametrize("algo", [1, 3, 5])
def test_process_past_the_grid_split(eng, big, algo):
    """Rows on both sides of the split equal the same rows run as a small batch, bit for bit, and the oracle within the bound;
    nothing beyond a row's length is written."""
    import torch
    d = big
    x, ln = torch.from_numpy(d["x"]).cuda(), torch.from_numpy(d["len"]).cuda()
    out = torch.full_like(x, 7.0)
    eng.process(algo, x, ln, eng.upload_plan(big_plan(d)), out=out)
    torch.cuda.synchronize()
    assert _beyond_untouched(out, ln, 7.0)
    y = out.cpu().numpy()
    rows = [big_row(d, u) for u in d["rows"]]
    small = run_rows(eng, algo, rows, ld=LD_BIG)
    for u, row, s in zip(d["rows"], rows, small):
        L = row.x.shape[0]
        assert np.array_equal(y[u, :L], s), f"algo {algo} row {u}: differs from the same row in a small batch"
        ref, tol = reference(row, algo, C_DENSE)
        assert ratio(np.abs(y[u, :L] - ref), tol) <= 1.0, f"algo {algo} row {u}"


@pytest.mark.gpu
@pytest.mark.parametrize("repeat_pad,layout", [(False, 1), (True, 0)])
def test_multiview_assemble_past_the_grid_split(eng, big, repeat_pad, layout):
    import torch
    from scl_deepfake_audio_detection_b200 import multiview
    d = big
    G, V, length = SPLIT + 2, 2, 48
    rs = np.random.RandomState(4100)
    a = torch.from_numpy(d["x"][:G].copy()).cuda()
    b = torch.from_numpy(d["noise"][:G].copy()).cuda()
    lens = d["len"][:G]
    other = (np.arange(G, dtype=np.int64) * 7919) % G
    view_row = np.stack([-1 - np.arange(G), other], axis=1).reshape(-1).astype(np.int32)
    first = lens[np.arange(G)]
    starts = np.where(first >= length, (rs.rand(G) * (first - length + 1)).astype(np.int64), 0).astype(np.int32)
    shape = (G, length, V) if layout == 0 else (G, V, length)
    out = torch.full(shape, 7.0, dtype=torch.float32, device="cuda")
    out, out_len, _ = multiview.assemble_ex(eng, a, b, torch.from_numpy(view_row).cuda(), torch.from_numpy(lens).cuda(), V, starts,
                                            length, repeat_pad, layout, out=out)
    got, got_len = out.cpu().numpy(), out_len.cpu().numpy()
    for g in d["rows"][:-1] + [G - 1]:
        fl = int(first[g])
        _, olen, wrap = orc.multiview_crop_plan(fl, length, False, repeat_pad)
        views = [d["noise"][g, :fl], d["x"][other[g], :lens[other[g]]]]
        want = orc.multiview_gather(views, fl, int(starts[g]), olen, wrap, repeat_pad).astype(np.float32)
        item = got[g] if layout == 0 else got[g].T
        assert got_len[g] == olen, g
        assert np.array_equal(item[:olen], want), g
        assert np.all(item[olen:] == 7.0), g


@pytest.mark.gpu
def test_reverb_past_the_grid_split(eng, big):
    import torch
    d = big
    B, ld_out = SPLIT + 2, 80
    rs = np.random.RandomState(4200)
    k = rs.randint(1, 17, B)
    rir = rs.standard_normal(int(k.sum())).astype(np.float32)
    off = np.concatenate([[0], np.cumsum(k)]).astype(np.int32)
    x, ln = torch.from_numpy(d["x"][:B].copy()).cuda(), torch.from_numpy(d["len"][:B].copy()).cuda()
    out = torch.full((B, ld_out), 7.0, dtype=torch.float32, device="cuda")
    y, out_len = eng.reverb(x, ln, torch.from_numpy(rir).cuda(), torch.from_numpy(off).cuda(), out=out, max_taps=16)
    assert _beyond_untouched(y, out_len, 7.0)
    y, n = y.cpu().numpy(), out_len.cpu().numpy()
    assert np.array_equal(n, d["len"][:B] + k - 1)
    rows = [u for u in d["rows"] if u < B]
    hs = [rir[off[u]:off[u + 1]] for u in rows]
    sx, sln = eng.pack_waveforms([d["x"][u, :d["len"][u]] for u in rows], ld=LD_BIG)
    sh = np.concatenate([[0], np.cumsum([h.size for h in hs])]).astype(np.int32)
    small, _ = eng.reverb(sx, sln, torch.from_numpy(np.concatenate(hs)).cuda(), torch.from_numpy(sh).cuda(), ld_out=ld_out, max_taps=16)
    small = small.cpu().numpy()
    for j, (u, h) in enumerate(zip(rows, hs)):
        ref = orc.reverb_convolve(d["x"][u, :d["len"][u]], h)
        assert np.array_equal(y[u, :n[u]], small[j, :n[u]]), u
        assert np.max(np.abs(y[u, :n[u]] - ref)) <= TOL, u


# ---- item 6: the per-operator ABI entries --------------------------------------------------------------------------------
@pytest.mark.gpu
def test_operator_entries_equal_process(eng):
    """rb_lnl, rb_isd and rb_ssi are rb_process(1 / 2 / 3), bit for bit."""
    import torch
    rows = dense_cases()[2].rows[6:10]  # algo 4 rows: LnL, ISD and SSI plans
    bp = pack_rows(rows)
    x, ln = eng.pack_waveforms([r.x for r in rows], ld=bp.ld)
    dp = eng.upload_plan(bp)
    ws = eng.workspace(bp.B, bp.ld)
    for algo, name in ((1, "rb_lnl"), (2, "rb_isd"), (3, "rb_ssi")):
        want = eng.process(algo, x, ln, dp)
        got = torch.zeros_like(x)
        rc = getattr(eng.lib, name)(C.c_void_p(x.data_ptr()), C.c_void_p(ln.data_ptr()), bp.B, bp.ld, C.byref(dp.struct),
                                    C.c_void_p(got.data_ptr()), C.c_void_p(eng._ws_ptr(ws)), ws.numel() - 256,
                                    C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0, name
        torch.cuda.synchronize()
        assert torch.equal(got, want), name

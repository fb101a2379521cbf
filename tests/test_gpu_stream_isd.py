"""The streaming normWav / ISD pass (norm_stream_kernel in rb_dense.cu) on hand-placed inputs, the chained algos by composition,
the impulse mask past its shared-memory limit, and the pipelined host entry with its device planner.

norm_stream_kernel runs algo 2, the ISD stage of algo 7, the ISD branch and the final sum of algo 8, rb_normwav and the last
normalisation of rb_reverb. Tile CTAs copy 32 768 samples each and take their peak; a finisher CTA per row applies the impulses
and finds the row's peak in one of three ways (rb_dense.cu, after the impulse rounds):
  * max(M, mt)   when no impulse replaced the peak sample (mx < M) or a new value reaches it (mt >= M);
  * no rescale   when M <= 1;
  * a rescan     of the row when the peak sample was hit, shrank, and M > 1.
Seeded random plans almost never reach the rescan, so the rows here are built by hand to steer every branch, at the tile edges,
the ragged last float4 chunk and the 4 096-impulse round boundary, with ties and special values.

The reference is numpy in float32: orc.apply_isd and orc.norm_wav on float32 rows follow the reference's operation order and
precision (g_sd * x in float32, times f_r and plus x in float64, rounded once), which is what isd_value computes. Results are
compared as bit patterns, so -0.0 against +0.0 is a difference. Where a NaN is expected only the NaN masks are compared: the
device writes the canonical NaN, numpy propagates the payload of the NaN it started from.
"""
import ctypes as C
import functools
import os
import subprocess
import sys
from collections import Counter
from dataclasses import dataclass

import numpy as np
import pytest

from oracle import rawboost_oracle as orc  # noqa: E402  (checker only)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARGS = orc.make_args()
SR = 16000
T = 32768        # samples per tile CTA (RB_STREAM_THREADS * RB_STREAM_CHUNKS * RB_STREAM_SUBTILES * 4)
ROUND = 4096     # impulses per finisher round (RB_STREAM_IMP_U * RB_STREAM_THREADS)
ONE_BITS = 0x3F800000
ABOVE_ONE = float(np.nextafter(np.float32(1), np.float32(2)))
SENTINEL = np.float32(-7.5)
MASK_SMEM_WORDS = 12 * 1024  # kMaskSmemWords: longer strides build the impulse mask with global atomics


# ---------------------------------------------------------------------------------------------------------------------------
# float32 reference and bit comparison
# ---------------------------------------------------------------------------------------------------------------------------
def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def abs_bits(a):
    return bits(a) & np.uint32(0x7FFFFFFF)


def assert_same_bits(got, want, what):
    """Bit patterns equal; where numpy has a NaN only NaN-ness is compared (canonical NaN on the device, payload in numpy)."""
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    gn, wn = np.isnan(got), np.isnan(want)
    if not np.array_equal(gn, wn):
        i = int(np.flatnonzero(gn != wn)[0])
        raise AssertionError(f"{what}: NaN mask differs first at {i}: got {got[i]!r}, want {want[i]!r}")
    diff = (bits(got) != bits(want)) & ~wn
    if diff.any():
        i = int(np.flatnonzero(diff)[0])
        raise AssertionError(f"{what}: {int(diff.sum())} samples differ, first at {i}: got {got[i]!r} ({int(bits(got)[i]):#010x}), "
                             f"want {want[i]!r} ({int(bits(want)[i]):#010x})")


def norm_wav_f32(x, always):
    x = np.asarray(x, np.float32)
    if x.size == 0:
        return x.copy()
    with np.errstate(all="ignore"):
        return np.asarray(orc.norm_wav(x, always), np.float32)


def isd_f32(x, idx, fr, g_sd):
    with np.errstate(all="ignore"):
        y = orc.apply_isd(np.asarray(x, np.float32), orc.ISDPlan(idx=np.asarray(idx, np.int64), f_r=np.asarray(fr, np.float64)),
                          np.float32(g_sd))
    assert y.dtype == np.float32
    return y


def isd_new_values(x, idx, fr, g_sd):
    """The values the impulses write, before normWav: float32(x + float64(float32(g_sd * x)) * f_r)."""
    h = np.asarray(x, np.float32)[idx]
    with np.errstate(all="ignore"):
        return (h.astype(np.float64) + (np.float32(g_sd) * h).astype(np.float64) * np.asarray(fr, np.float64)).astype(np.float32)


# ---------------------------------------------------------------------------------------------------------------------------
# hand-built ISD rows
# ---------------------------------------------------------------------------------------------------------------------------
@dataclass
class IsdRow:
    name: str
    x: np.ndarray    # float32 [L]
    idx: np.ndarray  # int64, distinct positions of [0, L)
    fr: np.ndarray   # float64
    g_sd: float = 2.0


def quiet(rs, L, amp):
    return (amp * rs.uniform(-1.0, 1.0, L)).astype(np.float32)


def impulses(rs, L, n, exclude=(), amp_fr=1.0):
    """n distinct random positions of [0, L) outside `exclude`, with gains uniform in (-amp_fr, amp_fr)."""
    free = np.setdiff1d(np.arange(L), np.asarray(sorted(exclude), np.int64))
    idx = rs.permutation(free)[:n].astype(np.int64)
    return idx, amp_fr * (2 * rs.rand(idx.size) - 1)


def make_row(rs, name, x, idx, fr, g_sd=2.0):
    """A row with its impulse list in random order."""
    idx, fr = np.asarray(idx, np.int64), np.asarray(fr, np.float64)
    order = rs.permutation(idx.size)
    return IsdRow(name, np.asarray(x, np.float32), idx[order], fr[order], g_sd)


def finisher_rows(rs):
    """Rows that steer the finisher's peak logic (g_sd = 2)."""
    rows = []
    # the peak sample is hit and shrinks, M > 1: the row's new peak is the second-largest sample, in the same tile, another
    # tile or the ragged tail (L = 98 307: three full tiles and a ragged float4 chunk of 3 samples)
    L = 3 * T + 3
    for f_hit in (-0.5, -0.25):  # -1/g_sd (the new value is exactly +0) and a shrink to half
        for pM, p2 in ((40000, 50000), (32768, 70000), (65535, 1000), (40000, L - 2), (L - 1, 5), (L - 3, L - 1)):
            x = quiet(rs, L, 0.3)
            s = 1.0 if rs.rand() < 0.5 else -1.0
            x[pM], x[p2] = 1.75 * s, -1.5 * s
            idx, fr = impulses(rs, L, 200, exclude=(pM, p2))
            rows.append(make_row(rs, f"shrink{f_hit}_M@{pM}_second@{p2}", x, np.append(idx, pM), np.append(fr, f_hit)))
    # M <= 1, M == 1 and M = nextafter(1, 2), hit or untouched (L = 32 769: the second tile holds one sample)
    L = T + 1
    for name, M, hit, f_hit, pM in (("M0.9_hit", 0.9, True, -0.25, 32767), ("M1_hit", 1.0, True, -0.25, 32768),
                                    ("M1_untouched", 1.0, False, 0.0, 100), ("Mnext_hit", ABOVE_ONE, True, -0.25, 32768),
                                    ("Mnext_hit_fr0", ABOVE_ONE, True, 0.0, 32767), ("Mnext_untouched", ABOVE_ONE, False, 0.0, 32768)):
        x = quiet(rs, L, 0.25)
        x[pM], x[7] = -M, 0.8
        idx, fr = impulses(rs, L, 100, exclude=(pM, 7))
        if hit:
            idx, fr = np.append(idx, pM), np.append(fr, f_hit)
        rows.append(make_row(rs, name, x, idx, fr))
    # the only sample above 1 lies in the ragged last float4 chunk of the tile CTA
    for L in (T + 1, 2 * T + 2, 3 * T + 3, 4 * T + 3):
        r = L % 4
        for p in range(L - r, L):
            x = quiet(rs, L, 0.5)
            x[p] = 1.25 if p % 2 else -1.25
            idx, fr = impulses(rs, L, 50, exclude=(p,), amp_fr=0.5)
            rows.append(make_row(rs, f"tail_only_above_one_L{L}_p{p}", x, idx, fr))
    L = 2 * T + 2
    x = quiet(rs, L, 0.5)
    x[10], x[L - 1] = 1.2, 0.6  # an impulse in the ragged chunk grows past the peak: 0.6 * (1 + 2 * 0.9) = 1.68
    idx, fr = impulses(rs, L, 50, exclude=(10, L - 1), amp_fr=0.5)
    rows.append(make_row(rs, "tail_impulse_grows_past_M", x, np.append(idx, L - 1), np.append(fr, 0.9)))
    # ties and whole-row cases
    L = 70001
    for name, hits in (("tie_one_hit", (1000,)), ("tie_both_hit", (1000, 69999))):
        x = quiet(rs, L, 0.3)
        x[1000], x[69999] = 1.5, -1.5
        idx, fr = impulses(rs, L, 300, exclude=(1000, 69999))
        rows.append(make_row(rs, name, x, np.append(idx, hits), np.append(fr, [-0.25] * len(hits))))
    x = quiet(rs, L, 0.3)
    x[100], x[5000] = 1.5, 0.6
    idx, fr = impulses(rs, L, 300, exclude=(100, 5000))
    rows.append(make_row(rs, "impulse_grows_past_M", x, np.append(idx, 5000), np.append(fr, 0.9)))
    rows.append(make_row(rs, "peak_shrinks_other_grows_past_M", x, np.append(idx, [100, 5000]), np.append(fr, [-0.5, 0.9])))
    x = x.copy()
    x[5000] = 0.5  # 0.5 + 2 * 0.5 * 1.0 = 1.5: a new value equal to M
    rows.append(make_row(rs, "peak_shrinks_other_reaches_M", x, np.append(idx, [100, 5000]), np.append(fr, [-0.25, 1.0])))
    for L in (5001, 3):
        x = quiet(rs, L, 1.2)
        rows.append(make_row(rs, f"every_sample_an_impulse_L{L}", x, np.arange(L), 2 * rs.rand(L) - 1))
    rows.append(make_row(rs, "no_impulses", quiet(rs, 7001, 1.3), [], []))
    idx, fr = impulses(rs, 4100, 30)
    rows.append(make_row(rs, "zero_row_with_impulses", np.zeros(4100, np.float32), idx, fr))
    # impulse counts around the 4 096-impulse rounds; the deciding impulse is the last of the list
    L = 20001
    for n in (ROUND - 1, ROUND, ROUND + 1, 2 * ROUND + 1, 3 * ROUND + 1):
        x = quiet(rs, L, 0.4)
        x[7] = 1.5
        idx, fr = impulses(rs, L, n, exclude=(7,), amp_fr=0.3)
        x[idx[-1]], fr[-1] = 0.9, 0.9  # 2.52: the row's peak comes from the last round
        rows.append(IsdRow(f"count{n}_grows_at_last", x, idx, fr))
        x = quiet(rs, L, 0.4)
        x[idx[-1]], x[7] = 1.5, 1.25
        fr = fr.copy()
        fr[-1] = -0.25  # the peak sample is hit in the last round and shrinks: the rescan finds 1.25
        rows.append(IsdRow(f"count{n}_peak_hit_at_last", x, idx, fr))
    return rows


def position_row(rs, g_sd):
    """Impulses at 0, L-1, the tile edges and inside the ragged last chunk (L = 131 075 = 4 tiles + 3)."""
    L = 4 * T + 3
    x = quiet(rs, L, 0.7)
    x[100] = 1.3
    special = sorted({0, L - 1, T - 1, T, 2 * T - 1, 2 * T, 3 * T - 1, 3 * T, 4 * T - 1, L - 3, L - 2})
    x[special] = np.where(rs.rand(len(special)) < 0.5, -0.9, 0.9)
    fr_s = np.where(rs.rand(len(special)) < 0.5, -1, 1) * rs.uniform(0.5, 1.0, len(special))
    idx, fr = impulses(rs, L, 500, exclude=special + [100])
    return make_row(rs, f"positions_g{g_sd}", x, np.append(idx, special), np.append(fr, fr_s), g_sd)


def parameter_rows(rs, g_sd):
    """fr in {-1, -0.5, 0, 1, random} at this g_sd, and the special values."""
    rows = []
    L = 4099
    for f in (-1.0, -0.5, 0.0, 1.0, None):
        x = quiet(rs, L, 1.1)
        idx, fr = impulses(rs, L, 400)
        if f is not None:
            fr[:] = f
        rows.append(make_row(rs, f"g{g_sd}_fr{f if f is not None else 'random'}", x, idx, fr, g_sd))
    L = 3001
    x = quiet(rs, L, 0.5)  # the peak (<= 1) is hit and shrinks: no rescale either way
    x[9] = 0.95
    idx, fr = impulses(rs, L, 30, exclude=(9,))
    rows.append(make_row(rs, f"g{g_sd}_idle_peak_hit", x, np.append(idx, 9), np.append(fr, -0.75 / g_sd if g_sd else 0.0), g_sd))
    inf_fr = -1.5 / g_sd if g_sd else -0.5  # below -1/g_sd: x + g_sd x f_r = inf - inf = NaN (g_sd = 0: 0 * inf = NaN)
    for name, p, val, hit, f in (("nan_at_impulse", 10, np.nan, True, 0.3), ("nan_untouched", 20, np.nan, False, 0.0),
                                 ("inf_hit_to_nan", 30, np.inf, True, inf_fr), ("inf_hit_grows", 40, np.inf, True, 0.5),
                                 ("minus_inf_untouched", 50, -np.inf, False, 0.0)):
        x = quiet(rs, L, 1.2)
        x[p] = val
        idx, fr = impulses(rs, L, 30, exclude=(p,))
        if hit:
            idx, fr = np.append(idx, p), np.append(fr, f)
        rows.append(make_row(rs, f"g{g_sd}_{name}", x, idx, fr, g_sd))
    for amp in (1.3, 0.5):  # -0.0 and +0.0, at impulses and not, in a rescaled row and in an idle one
        x = quiet(rs, L, amp)
        z = rs.permutation(L)[:80]
        x[z[:40]], x[z[40:]] = -0.0, 0.0
        idx, fr = impulses(rs, L, 60, exclude=set(z.tolist()))
        rows.append(make_row(rs, f"g{g_sd}_signed_zeros_amp{amp}", x, np.append(idx, z[::2]), np.append(fr, 2 * rs.rand(40) - 1), g_sd))
    x = quiet(rs, L, 1.3)  # subnormal samples, divided by the peak (gradual underflow, no flush to zero)
    sub = rs.permutation(L)[:80]
    x[sub] = (rs.randint(1, 1 << 23, 80) * np.where(rs.rand(80) < 0.5, -1, 1)).astype(np.int64).astype(np.float64) * 2.0 ** -149
    idx, fr = impulses(rs, L, 60, exclude=set(sub.tolist()))
    rows.append(make_row(rs, f"g{g_sd}_subnormals", x, np.append(idx, sub[::2]), np.append(fr, 2 * rs.rand(40) - 1), g_sd))
    return rows


RAGGED_LENS = [1, 2, 3, 4, 5, T - 1, T, T + 1, 2 * T, 3 * T + 1, 4 * T + 3]


def ragged_rows(rs):
    rows = []
    for L in RAGGED_LENS:
        x = quiet(rs, L, 1.2)
        idx, fr = impulses(rs, L, max(1, L // 20))
        rows.append(make_row(rs, f"ragged_L{L}", x, idx, fr))
    return rows


G_SDS = (0.0, 0.1, 2.0, 2.5)


@functools.lru_cache(maxsize=None)
def isd_batches():
    """g_sd -> rows (g_sd is one value per batch)."""
    rs = np.random.RandomState(7000)
    out = {}
    for g in G_SDS:
        rows = parameter_rows(rs, g) + [position_row(rs, g)]
        if g == 2.0:
            rows = finisher_rows(rs) + ragged_rows(rs) + rows
        else:  # one rescan row at every g_sd: the peak is hit and shrinks to a quarter at most
            L = 2 * T + 5
            x = quiet(rs, L, 0.3)
            x[T + 3], x[L - 1] = 1.75, 1.5
            idx, fr = impulses(rs, L, 100, exclude=(T + 3, L - 1), amp_fr=0.5)
            f_hit = -0.75 / g if g else 0.0
            rows.append(make_row(rs, f"g{g}_shrink", x, np.append(idx, T + 3), np.append(fr, f_hit), g))
        out[g] = rows
    return out


def all_isd_rows():
    return [r for rows in isd_batches().values() for r in rows]


def finisher_branch(row):
    """The finisher's rule, from float32 bit patterns: which way it finds the row's peak."""
    M = int(abs_bits(row.x).max()) if row.x.size else 0
    if row.idx.size:
        mx = int(abs_bits(row.x[row.idx]).max())
        mt = int(abs_bits(isd_new_values(row.x, row.idx, row.fr, row.g_sd)).max())
    else:
        mx = mt = 0
    if mx < M:
        return "mx<M"
    if mt >= M:
        return "mt>=M"
    if M <= ONE_BITS:
        return "M<=1"
    return "rescan"


def rescan_place(row):
    """Where a rescanned row's new peak lies: the ragged last chunk, the replaced peak's tile, or another tile."""
    y = row.x.copy()
    y[row.idx] = isd_new_values(row.x, row.idx, row.fr, row.g_sd)
    pM, py = int(np.argmax(abs_bits(row.x))), int(np.argmax(abs_bits(y)))
    L = row.x.shape[0]
    if L % 4 and py >= L - L % 4:
        return "tail"
    return "same" if py // T == pM // T else "other"


# ---------------------------------------------------------------------------------------------------------------------------
# CPU only
# ---------------------------------------------------------------------------------------------------------------------------
def test_hand_rows_are_valid_plans():
    for row in all_isd_rows():
        L = row.x.shape[0]
        assert row.idx.shape == row.fr.shape, row.name
        assert np.unique(row.idx).size == row.idx.size, f"{row.name}: repeated impulse position"
        assert row.idx.size == 0 or (row.idx.min() >= 0 and row.idx.max() < L), row.name


def test_hand_rows_reach_every_finisher_branch():
    """Every branch of the finisher's peak logic is taken by several rows, and the rescan by rows whose new peak lies in the
    replaced peak's tile, in another tile and in the ragged last chunk -- so an edit that drops a case shows here."""
    rows = all_isd_rows()
    branch = Counter(finisher_branch(r) for r in rows)
    print(dict(branch))
    for b in ("mx<M", "mt>=M", "M<=1", "rescan"):
        assert branch[b] >= 3, (b, dict(branch))
    places = Counter(rescan_place(r) for r in rows if finisher_branch(r) == "rescan")
    print(dict(places))
    assert all(places[p] >= 1 for p in ("same", "other", "tail")), dict(places)
    # the rescan must matter: rows where max(M, mt) would give another result than the row's true peak
    matter = [r for r in rows if finisher_branch(r) == "rescan" and np.isfinite(r.x).all()
              and not np.array_equal(bits(isd_f32(r.x, r.idx, r.fr, r.g_sd)), bits(_shortcut(r)))]
    assert len(matter) >= 3
    # impulse rounds: rows whose deciding impulse is the first of a later round
    assert {r.idx.size for r in rows} >= {ROUND - 1, ROUND, ROUND + 1, 2 * ROUND + 1, 3 * ROUND + 1}
    # only sample above 1 in the ragged chunk, at every offset inside it
    tails = {(r.x.shape[0], r.x.shape[0] - int(np.argmax(np.abs(r.x)))) for r in rows if r.name.startswith("tail_only")}
    assert {d for _, d in tails} == {1, 2, 3}


def _shortcut(row):
    """What y / max(M, mt) would be (a finisher without the rescan): y scaled by the wrong peak when that exceeds 1."""
    y = row.x.copy()
    y[row.idx] = isd_new_values(row.x, row.idx, row.fr, row.g_sd)
    pk = max(np.float32(np.abs(row.x).max()), np.float32(np.abs(y[row.idx]).max()) if row.idx.size else np.float32(0))
    return y / pk if pk > 1 else y


def test_mask_stride_threshold():
    """The stride pair of the boundary test straddles the shared-memory mask limit (mask_ld_for in rb_api.cu)."""
    mask_ld = lambda ld: (ld // 32 + 2 + 3) // 4 * 4
    assert mask_ld(393180) == MASK_SMEM_WORDS and mask_ld(393184) > MASK_SMEM_WORDS
    assert mask_ld(64600) <= MASK_SMEM_WORDS < mask_ld(400000)


# ---------------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def eng():
    torch = pytest.importorskip("torch")
    from scl_deepfake_audio_detection_b200.engine import Engine
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return Engine(0)


def loud_batch(rs, waves, ld=None):
    """[B, ld] float32 host array: each row's samples, then +-100 garbage in the padding."""
    from scl_deepfake_audio_detection_b200 import plans
    lengths = np.array([w.shape[0] for w in waves], np.int32)
    ld = ld or plans.padded_ld(int(lengths.max()))
    x = np.where(rs.rand(len(waves), ld) < 0.5, -100.0, 100.0).astype(np.float32)
    for u, w in enumerate(waves):
        x[u, :w.shape[0]] = w
    return x, lengths


def hand_plan(rows, ld):
    from scl_deepfake_audio_detection_b200 import plans
    n = np.array([r.idx.size for r in rows], np.int64)
    return plans.BatchPlan(B=len(rows), ld=ld, lengths=np.array([r.x.shape[0] for r in rows], np.int32),
                           isd_off=np.concatenate([[0], np.cumsum(n)]).astype(np.int32),
                           isd_idx=np.concatenate([r.idx for r in rows]).astype(np.int32),
                           isd_fr=np.concatenate([r.fr for r in rows]).astype(np.float64), g_sd=float(rows[0].g_sd))


def to_dev(*arrays):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


def assert_untouched_past(out, lengths, what, fill=None):
    """Nothing past a row's length was written: the sentinel (or the row's own padding, `fill`) is still there."""
    for u, L in enumerate(lengths):
        want = np.full(out.shape[1] - L, SENTINEL, np.float32) if fill is None else fill[u, L:]
        assert np.array_equal(bits(out[u, L:]), bits(want)), f"{what}: row {u} (L={L}) written past its length"


@pytest.mark.gpu
@pytest.mark.parametrize("g_sd", G_SDS)
def test_isd_hand_rows_bit_exact(eng, g_sd):
    """rb_process(2) on the hand-built rows equals orc.apply_isd in float32, bit for bit, and writes nothing past a row."""
    import torch
    rows = isd_batches()[g_sd]
    x, lengths = loud_batch(np.random.RandomState(7100), [r.x for r in rows])
    bp = hand_plan(rows, x.shape[1])
    xd, ln = to_dev(x, lengths)
    out = torch.full_like(xd, float(SENTINEL))
    eng.process(2, xd, ln, eng.upload_plan(bp), out=out)
    torch.cuda.synchronize()
    y = out.cpu().numpy()
    for u, r in enumerate(rows):
        assert_same_bits(y[u, :r.x.shape[0]], isd_f32(r.x, r.idx, r.fr, g_sd), f"g_sd={g_sd} row {u} {r.name} [{finisher_branch(r)}]")
    assert_untouched_past(y, lengths, f"g_sd={g_sd}")


# ---- the sum and plain passes around the 48-row lag ---------------------------------------------------------------------------
LAG_BS = [1, 47, 48, 49, 130]
LAG_LENS = [4097, 32769, 1, 65537, 3, 32768, 40000, 5, 32767, 12000, 2]
SUM_LEN = 40000


def sum_row(rs, L, above):
    """x of multiples of 2^-8 with x[0] = 0 and an exactly zero sum. Under the LnL taps [0.5], [0], [0], ... its LnL branch is
    exactly 0.5 x[n+1] (zero mean, peak 0.375: no division), its ISD branch without impulses is x itself (peak <= 1), and
    their sum peaks at exactly 1.0 (or 1 + 2^-8) at n = L/3 and at minus that at n = 2L/3."""
    x = np.zeros(L, np.float32)
    k, j = L // 3, 2 * L // 3
    free = rs.permutation(np.setdiff1d(np.arange(L), [0, k, k + 1, j, j + 1]))
    npair = free.size // 2
    v = rs.randint(-64, 65, npair) / 256.0
    x[free[:npair]], x[free[npair:2 * npair]] = v, -v
    top = 0.75 + (2.0 ** -8 if above else 0.0)
    x[k], x[k + 1], x[j], x[j + 1] = top, 0.5, -top, -0.5
    return x


@functools.lru_cache(maxsize=None)
def lag_batch(B):
    """Ragged rows around the lag: row 0 (and 1) sum to a peak of exactly 1.0 (just above 1), rows 2 / 3 peak at exactly 1.0 /
    nextafter(1, 2) themselves, row B/2 is empty; the rest carry seeded algo-8 plans of the default arguments."""
    from scl_deepfake_audio_detection_b200 import plans
    rs = np.random.RandomState(8000 + B)
    kinds = ["sum_above"] if B == 1 else ["sum_one", "sum_above", "x_one", "x_above"] + ["random"] * (B - 4)
    ups, waves = [], []
    for u, kind in enumerate(kinds):
        L = SUM_LEN if kind.startswith("sum") else LAG_LENS[(3 * u + B) % len(LAG_LENS)]
        if B > 1 and u == B // 2:
            L = 0
        np.random.seed(8100 + 1000 * B + u)
        up = plans.draw_for_algo(L, SR, ARGS, 8)
        if kind.startswith("sum"):
            x = sum_row(rs, L, kind == "sum_above")
            up.lnl_taps = [np.array([0.5])] + [np.zeros(1)] * (ARGS.N_f - 1)
            up.isd_idx, up.isd_fr = np.zeros(0, np.int64), np.zeros(0)
        else:
            x = quiet(rs, L, 0.6 if kind.startswith("x_") else rs.uniform(0.2, 1.4))
            if kind.startswith("x_") and L:
                x[rs.randint(L)] = -1.0 if kind == "x_one" else -ABOVE_ONE
        ups.append(up)
        waves.append(x)
    x, lengths = loud_batch(rs, waves)
    return x, lengths, plans.pack(ups, ld=x.shape[1]), kinds


@pytest.mark.gpu
@pytest.mark.parametrize("B", LAG_BS)
def test_sum_pass_is_normwav_of_the_branches(eng, B):
    """rb_process(8) == normWav(rb_process(1) + rb_process(2), 0), the add and the division done in numpy float32 on the device's
    own stage outputs with the same plan; an empty row stays untouched."""
    import torch
    x, lengths, bp, kinds = lag_batch(B)
    xd, ln = to_dev(x, lengths)
    dp = eng.upload_plan(bp)
    y = {}
    for algo in (1, 2, 8):
        out = torch.full_like(xd, float(SENTINEL))
        eng.process(algo, xd, ln, dp, out=out)
        torch.cuda.synchronize()
        y[algo] = out.cpu().numpy()
        assert_untouched_past(y[algo], lengths, f"B={B} algo {algo}")
    for u, L in enumerate(lengths):
        s = y[1][u, :L] + y[2][u, :L]
        if kinds[u] == "sum_one":
            assert np.abs(s).max() == 1.0
        elif kinds[u] == "sum_above":
            assert np.abs(s).max() == 1.0 + 2.0 ** -8
        assert_same_bits(y[8][u, :L], norm_wav_f32(s, 0), f"B={B} row {u} ({kinds[u]}, L={L})")


@pytest.mark.gpu
def test_batch_without_any_impulse(eng):
    """A batch whose utterances have no impulse at all (empty isd_idx / isd_fr) runs every ISD algo: algo 2 is normWav(x, 0),
    algo 5 is algo 1 and algo 8 is normWav(1 + 2), bit for bit, through the device and the host-buffer entries."""
    from scl_deepfake_audio_detection_b200 import plans
    rs = np.random.RandomState(8500)
    lengths = [5, 4097, 32769, 12000]
    ups, waves = [], []
    for u, L in enumerate(lengths):
        np.random.seed(8600 + u)
        up = plans.draw_for_algo(L, SR, ARGS, 4)
        up.isd_idx, up.isd_fr = np.zeros(0, np.int64), np.zeros(0)
        ups.append(up)
        waves.append(quiet(rs, L, 0.5 + 0.3 * u))
    x, ln_h = loud_batch(rs, waves)
    bp = plans.pack(ups, ld=x.shape[1])
    assert bp.isd_idx.size == 0 and bp.isd_fr.size == 0
    xd, ln = to_dev(x, ln_h)
    dp = eng.upload_plan(bp)
    inside = np.arange(x.shape[1])[None, :] < ln_h[:, None]
    y = {}
    for algo in range(1, 9):
        y[algo] = eng.process(algo, xd, ln, dp).cpu().numpy()
        host = eng.process_host(algo, x, bp)
        assert np.array_equal(bits(host)[inside], bits(y[algo])[inside]), f"algo {algo}: host entry differs"
    for u, L in enumerate(lengths):
        assert_same_bits(y[2][u, :L], norm_wav_f32(x[u, :L], 0), f"algo 2 row {u}")
        assert_same_bits(y[5][u, :L], y[1][u, :L], f"algo 5 row {u}")
        assert_same_bits(y[8][u, :L], norm_wav_f32(y[1][u, :L] + y[2][u, :L], 0), f"algo 8 row {u}")


def run_normwav(eng, x, lengths, always, in_place):
    import torch
    xd, ln = to_dev(x, lengths)
    out = xd if in_place else torch.full_like(xd, float(SENTINEL))
    eng.normwav(xd, ln, bool(always), out=out)
    torch.cuda.synchronize()
    return out.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("B", LAG_BS)
@pytest.mark.parametrize("always", [0, 1])
@pytest.mark.parametrize("in_place", [False, True], ids=["out_of_place", "in_place"])
def test_normwav_around_the_lag(eng, B, always, in_place):
    x, lengths, _, kinds = lag_batch(B)
    y = run_normwav(eng, x, lengths, always, in_place)
    for u, L in enumerate(lengths):
        assert_same_bits(y[u, :L], norm_wav_f32(x[u, :L], always), f"B={B} row {u} ({kinds[u]}, L={L})")
    assert_untouched_past(y, lengths, f"B={B}", fill=x if in_place else None)


LAG_SCRIPT = r"""
import sys
import numpy as np
import torch
from scl_deepfake_audio_detection_b200 import plans
from scl_deepfake_audio_detection_b200.engine import Engine
d = np.load(sys.argv[1])
eng = Engine(0)
x, ln = torch.from_numpy(d["x"]).cuda(), torch.from_numpy(d["len"]).cuda()
res = {}
for a in (0, 1):
    out = torch.full_like(x, float(d["sentinel"]))
    eng.normwav(x, ln, bool(a), out=out)
    res["normwav%d" % a] = out.cpu().numpy()
bp = plans.BatchPlan(B=x.shape[0], ld=x.shape[1], lengths=d["len"], n_f=int(d["n_f"]), lnl_taps=d["lnl_taps"],
                     lnl_tap_off=d["lnl_tap_off"], isd_off=d["isd_off"], isd_idx=d["isd_idx"], isd_fr=d["isd_fr"], g_sd=float(d["g_sd"]))
out = torch.full_like(x, float(d["sentinel"]))
eng.process(8, x, ln, eng.upload_plan(bp), out=out)
res["algo8"] = out.cpu().numpy()
np.savez(sys.argv[2], **res)
"""


@pytest.mark.gpu
def test_stream_lag_override_changes_no_bit(eng, tmp_path):
    """RAWBOOST_B200_STREAM_LAG (read once per process) moves the finishers of the plain and the sum pass 0 or 192 rows behind
    their tiles; the outputs must not change by a bit."""
    import torch
    x, lengths, bp, _ = lag_batch(130)
    xd, ln = to_dev(x, lengths)
    want = {f"normwav{a}": run_normwav(eng, x, lengths, a, False) for a in (0, 1)}
    out = torch.full_like(xd, float(SENTINEL))
    eng.process(8, xd, ln, eng.upload_plan(bp), out=out)
    want["algo8"] = out.cpu().numpy()
    src = tmp_path / "in.npz"
    np.savez(src, x=x, len=lengths, sentinel=SENTINEL, n_f=bp.n_f, lnl_taps=bp.lnl_taps, lnl_tap_off=bp.lnl_tap_off,
             isd_off=bp.isd_off, isd_idx=bp.isd_idx, isd_fr=bp.isd_fr, g_sd=bp.g_sd)
    for lag in ("0", "192"):
        dst = tmp_path / f"out{lag}.npz"
        env = dict(os.environ, RAWBOOST_B200_STREAM_LAG=lag)
        r = subprocess.run([sys.executable, "-s", "-c", LAG_SCRIPT, str(src), str(dst)], cwd=ROOT, env=env, capture_output=True,
                           text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        got = np.load(dst)
        for k, v in want.items():
            assert np.array_equal(bits(got[k]), bits(v)), f"lag {lag}: {k} differs from the default lag"


# ---- chained algos by composition ---------------------------------------------------------------------------------------------
COMP_LENS = [64600, 1, 5, 4097, 32769, 70001, 12000, 98307]


@functools.lru_cache(maxsize=None)
def comp_batch():
    """Seeded LnL and SSI draws of the default arguments with hand-placed impulses (tile edges, the ends, the ragged chunk);
    row 3 has a DC offset of 0.9."""
    from scl_deepfake_audio_detection_b200 import plans
    rs = np.random.RandomState(9000)
    ups, waves = [], []
    for u, L in enumerate(COMP_LENS):
        np.random.seed(9100 + u)
        up = plans.draw_for_algo(L, SR, ARGS, 4)
        special = {p for p in (0, L - 1, L - 2, L - 3, T - 1, T, 2 * T - 1, 2 * T, 3 * T - 1, 3 * T) if 0 <= p < L}
        extra, _ = impulses(rs, L, L // 25, exclude=special)
        idx = rs.permutation(np.array(sorted(special | set(extra.tolist())), np.int64))
        fr = 2 * rs.rand(idx.size) - 1
        fr[:3] = [-0.5, 0.0, 1.0][:idx.size]
        up.isd_idx, up.isd_fr = idx, fr[:idx.size]
        ups.append(up)
        waves.append((0.9 + 0.2 * rs.uniform(-1, 1, L)).astype(np.float32) if u == 3 else quiet(rs, L, rs.uniform(0.3, 1.3)))
    x, lengths = loud_batch(rs, waves)
    return x, lengths, plans.pack(ups, ld=x.shape[1])


@pytest.mark.gpu
def test_chained_algos_equal_their_stages(eng):
    """4 == 3(5(x)), 6 == 3(1(x)), 7 == 3(2(x)) and 8 == normWav(1(x) + 2(x), 0), bit for bit; every algo on a fresh workspace
    (filled with 0xff bytes) and again on one workspace right after a different algo, so stale tile statistics, stream state or
    arrival counters would show."""
    import torch
    x, lengths, bp = comp_batch()
    xd, ln = to_dev(x, lengths)
    dp = eng.upload_plan(bp)
    B, ld = x.shape
    need = int(eng.lib.rb_workspace_bytes(B, ld))
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def fresh():
        return torch.full((need + 256,), 0xFF, dtype=torch.uint8, device="cuda")

    def run(algo, src, ws):
        out = torch.full_like(xd, float(SENTINEL))
        rc = eng.lib.rb_process(algo, C.c_void_p(src.data_ptr()), C.c_void_p(ln.data_ptr()), B, ld, C.byref(dp.struct),
                                C.c_void_p(out.data_ptr()), C.c_void_p(eng._ws_ptr(ws)), ws.numel() - 256, stream)
        assert rc == 0, (algo, rc)
        torch.cuda.synchronize()
        return out

    stage = {a: run(a, xd, fresh()) for a in (1, 2, 3, 5)}
    fresh_out = {a: run(a, xd, fresh()) for a in (4, 6, 7, 8)}
    composed = {4: run(3, stage[5], fresh()), 6: run(3, stage[1], fresh()), 7: run(3, stage[2], fresh())}
    for a in (4, 6, 7):
        got, want = fresh_out[a].cpu().numpy(), composed[a].cpu().numpy()
        for u, L in enumerate(lengths):
            assert_same_bits(got[u, :L], want[u, :L], f"algo {a} row {u} (L={L}) against its stages")
        assert_untouched_past(got, lengths, f"algo {a}")
    y1, y2, y8 = stage[1].cpu().numpy(), stage[2].cpu().numpy(), fresh_out[8].cpu().numpy()
    for u, L in enumerate(lengths):
        assert_same_bits(y8[u, :L], norm_wav_f32(y1[u, :L] + y2[u, :L], 0), f"algo 8 row {u} (L={L}) against its branches")
    results = {**{a: t.cpu().numpy() for a, t in stage.items()}, **{a: t.cpu().numpy() for a, t in fresh_out.items()}}
    shared = fresh()
    for algo in (4, 5, 6, 1, 7, 2, 8, 3, 4, 8, 6, 7, 5, 2):
        got = run(algo, xd, shared).cpu().numpy()
        assert np.array_equal(bits(got), bits(results[algo])), f"algo {algo} on a used workspace differs from a fresh one"


# ---- the impulse mask past its shared-memory limit ---------------------------------------------------------------------------
MASK_ROWS = {  # name: (length, seed, DC offset)
    "L400000": (400000, 11, 0.0), "L393300": (393300, 12, 0.0), "L393180": (393180, 13, 0.0), "L64600": (64600, 14, 0.0),
    "L4097": (4097, 15, 0.0), "L1": (1, 16, 0.0), "dc300000": (300000, 17, 0.9),
}


def mask_wave(name):
    L, seed, dc = MASK_ROWS[name]
    rs = np.random.RandomState(seed)
    return ((dc + 0.25 * rs.uniform(-1, 1, L)) if dc else 0.4 * rs.standard_normal(L)).astype(np.float32)


def run_seeded_rows(eng, algo, names, ld):
    import torch
    from scl_deepfake_audio_detection_b200 import plans
    lengths = [MASK_ROWS[n][0] for n in names]
    seeds = [MASK_ROWS[n][1] for n in names]
    bp = plans.draw_batch(lengths, SR, ARGS, algo, seeds=seeds, ld=ld)
    x, ln = eng.pack_waveforms([mask_wave(n) for n in names], ld=ld)
    y = eng.process(algo, x, ln, eng.upload_plan(bp))
    torch.cuda.synchronize()
    y = y.cpu().numpy()
    return {n: y[u, :L] for u, (n, L) in enumerate(zip(names, lengths))}


@pytest.mark.gpu
@pytest.mark.parametrize("algo", [4, 5])
def test_global_impulse_mask(eng, algo):
    """ld = 400 000 builds the impulse mask with global atomics (every row, short ones too): every row within 1e-5 of the
    float64 oracle, and the short rows bit for bit what the same rows and plans give at ld = 64 600 (shared-memory mask)."""
    names = ["L400000", "L393300", "L64600", "L4097", "L1", "dc300000"]
    got = run_seeded_rows(eng, algo, names, 400000)
    for n in names:
        np.random.seed(MASK_ROWS[n][1])
        ref = orc.process(mask_wave(n), SR, ARGS, algo)
        err = float(np.max(np.abs(got[n].astype(np.float64) - ref)))
        assert err <= 1e-5, f"algo {algo} {n}: max-abs error {err:.3g} against the oracle"
    small = run_seeded_rows(eng, algo, ["L64600", "L4097", "L1"], 64600)
    for n, v in small.items():
        assert np.array_equal(bits(got[n]), bits(v)), f"algo {algo} {n}: ld 400000 differs from ld 64600"


@pytest.mark.gpu
@pytest.mark.parametrize("algo", [4, 5])
def test_mask_path_boundary_gives_identical_bits(eng, algo):
    """ld = 393 180 is the longest stride of the shared-memory mask, 393 184 the shortest of the global one; the fused tail
    reads only a row's active tiles, so the same rows and plans give the same bits."""
    names = ["L393180", "L64600", "L4097", "L1", "dc300000"]
    a = run_seeded_rows(eng, algo, names, 393180)
    b = run_seeded_rows(eng, algo, names, 393184)
    for n in names:
        assert np.array_equal(bits(a[n]), bits(b[n])), f"algo {algo} {n}: ld 393180 and 393184 differ"


def ulp_err(got, ref):
    got, ref = np.asarray(got, np.float32), np.asarray(ref, np.float32)
    if ref.size == 0:
        return 0.0
    return float(np.max(np.abs(got.astype(np.float64) - ref.astype(np.float64)) / np.spacing(np.maximum(np.abs(ref), np.float32(1e-30)))))


@pytest.mark.gpu
@pytest.mark.parametrize("algo", [2, 3, 5])
def test_device_plan_on_rows_past_the_shared_mask(eng, algo):
    import torch
    from scl_deepfake_audio_detection_b200 import plans
    names = ["L400000", "L393300", "L64600", "L4097", "L1", "dc300000"]
    lengths = [MASK_ROWS[n][0] for n in names]
    seeds = [MASK_ROWS[n][1] for n in names]
    ln = torch.tensor(lengths, dtype=torch.int32, device="cuda")
    dp = eng.draw_device_plan(ln, seeds, SR, ARGS, algo, 400000)
    torch.cuda.synchronize()
    got = eng.download_plan(dp)
    ref = plans.draw_batch(lengths, SR, ARGS, algo, seeds=seeds, ld=400000)
    for name in ("lnl_tap_off", "isd_off", "isd_idx", "isd_fr", "ssi_tap_off", "ssi_snr_db"):
        r = getattr(ref, name)
        if r is not None:
            assert np.array_equal(r, getattr(got, name)), f"algo {algo}: {name} differs from numpy"
    for name in ("lnl_taps", "ssi_taps", "ssi_noise"):
        r = getattr(ref, name)
        if r is not None:
            assert ulp_err(getattr(got, name), r) <= 1.0, f"algo {algo}: {name} more than 1 ulp(fp32) from numpy"


# ---- the pipelined host entry with the device planner -------------------------------------------------------------------------
HOST_B, HOST_LD, HOST_CHUNK = 8192, 2000, 1024  # 8 chunks; without SSI the planner runs in 4 pieces (1, 1, 4 and 2 chunks)


@pytest.fixture(scope="module")
def host_batch():
    rs = np.random.RandomState(10000)
    amp = rs.uniform(0.2, 1.3, (HOST_B, 1))
    x = (amp * rs.uniform(-1, 1, (HOST_B, HOST_LD))).astype(np.float32)
    lengths = np.where(rs.rand(HOST_B) < 0.25, rs.randint(1, HOST_LD + 1, HOST_B), HOST_LD).astype(np.int32)
    lengths[:4] = [1, 2, 3, HOST_LD - 1]
    seeds = rs.randint(0, 2 ** 32, HOST_B, dtype=np.uint64).astype(np.uint32)
    return x, lengths, seeds


@pytest.mark.gpu
@pytest.mark.parametrize("algo", range(9))
def test_pipelined_host_entry_matches_rb_process(eng, host_batch, algo):
    """rb_process_host_seeded, its device planner issued in pieces beside the kernels, == rb_process on host-drawn plans:
    bit-exact for algos 0 and 2, within 1e-5 otherwise (taps and noise may differ by 1 ulp)."""
    import torch
    from scl_deepfake_audio_detection_b200.native_planner import NativePlanner
    x, lengths, seeds = host_batch
    eng.set_host_chunk(HOST_CHUNK)
    try:
        got = eng.process_host_seeded(algo, x, lengths, seeds, SR, ARGS)
    finally:
        eng.set_host_chunk(0)
    inside = np.arange(HOST_LD)[None, :] < lengths[:, None]
    plan = NativePlanner(threads=0, pinned=False).draw(lengths, SR, ARGS, algo, seeds=seeds, ld=HOST_LD, copy=True) if algo else None
    xd, ln = to_dev(x, lengths)
    ref = eng.process(algo, xd, ln, eng.upload_plan(plan) if plan is not None else None)
    torch.cuda.synchronize()
    ref = ref.cpu().numpy()
    if algo in (0, 2):
        assert np.array_equal(bits(got)[inside], bits(ref)[inside]), f"algo {algo}: seeded host entry differs from rb_process"
    else:
        err = float(np.max(np.abs(got[inside].astype(np.float64) - ref[inside])))
        assert err <= 1e-5, f"algo {algo}: seeded host entry {err:.3g} from rb_process"

"""The fused LnL -> ISD tail of the FIR-bank kernel (algo 5) against its two stages, on hand-built plans.

Algo 5 runs the LnL bank and, in the tail of the CTA that finishes an utterance, normWav, the impulses and the second normWav.
Its result must equal algo 2 (the streaming ISD pass) applied to algo 1's result, bit for bit. The tail keeps the impulses'
new values in the CTA's idle shared memory between the gather and the scatter (ISD_CAP of them) and gathers the rest again,
so the rows here sit on both sides of that capacity: n = 0, 1, cap - 1, cap, cap + 1, every impulse inside one tile, impulses
at both ends, loud rows (both normalisations fire), and 100 000- and 211 000-sample rows with more impulses than the capacity.
"""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import rawboost_oracle as orc  # noqa: E402  (argument defaults only)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARGS = orc.make_args()
SR = 16000
ISD_CAP = 2 * 3136 + 2 * 528  # x1, xp, he and ho of the kernel's shared memory, in floats
TILE = 2560                   # outputs per FIR-bank CTA
SENTINEL = np.float32(-7.5)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def row(name, L, n, seed, loud=False, where=None, ends=False):
    """(name, x, impulse positions, f_r): a distinct permutation prefix of positions, as the planner draws them."""
    rs = np.random.RandomState(seed)
    x = (0.9 * rs.uniform(-1, 1, L) * 3.0 if loud else 0.1 * rs.standard_normal(L)).astype(np.float32)
    lo, hi = where if where else (0, L)
    if ends:  # 0 and L - 1 among n positions, in a random place of the list
        idx = rs.permutation(np.concatenate([[0, L - 1], 1 + rs.permutation(L - 2)[:n - 2]]))
    else:
        idx = lo + rs.permutation(hi - lo)[:n]
    fr = 2 * rs.rand(idx.size) - 1
    return name, x, idx.astype(np.int64), fr


CASES = {
    "n0": lambda: [row("n0", 64600, 0, 1)],
    "n1": lambda: [row("n1", 64600, 1, 2)],
    "cap_minus_1": lambda: [row("cap_minus_1", 64600, ISD_CAP - 1, 3)],
    "cap": lambda: [row("cap", 64600, ISD_CAP, 4)],
    "cap_plus_1": lambda: [row("cap_plus_1", 64600, ISD_CAP + 1, 5)],
    "one_tile": lambda: [row("one_tile", 64600, 2000, 6, where=(2 * TILE, 3 * TILE))],
    "ends": lambda: [row("ends", 64600, 500, 7, ends=True), row("ends_short", 7, 2, 8, ends=True)],
    "loud": lambda: [row("loud", 64600, 3000, 9, loud=True), row("loud_cap_plus_1", 64600, ISD_CAP + 1, 10, loud=True)],
    "long": lambda: [row("L100000", 100000, 10000, 11), row("L211000", 211000, 21100, 12, loud=True)],
    "ragged": lambda: [row("r_n0", 5, 0, 13), row("r_cap", 64600, ISD_CAP, 14, loud=True), row("r_one", 1, 1, 15),
                       row("r_long", 211000, 21100, 16), row("r_n1", 3000, 1, 17), row("r_capm1", 70001, ISD_CAP - 1, 18),
                       row("r_ends", 4097, 300, 19, ends=True), row("r_capp1", 100000, ISD_CAP + 1, 20)],
}


def batch(rows):
    """Device input with +-100 garbage past each row, and a packed plan: seeded LnL draws, the rows' own impulses."""
    from scl_deepfake_audio_detection_b200 import plans
    lengths = np.array([r[1].shape[0] for r in rows], np.int32)
    ld = plans.padded_ld(int(lengths.max()))
    rs = np.random.RandomState(99)
    x = np.where(rs.rand(len(rows), ld) < 0.5, -100.0, 100.0).astype(np.float32)
    ups = []
    for u, (name, w, idx, fr) in enumerate(rows):
        x[u, :w.shape[0]] = w
        np.random.seed(7000 + u)
        up = plans.draw_for_algo(w.shape[0], SR, ARGS, 5)
        up.isd_idx, up.isd_fr = idx, fr
        ups.append(up)
    return x, lengths, plans.pack(ups, ld=ld)


@pytest.fixture(scope="module")
def eng():
    torch = pytest.importorskip("torch")
    from scl_deepfake_audio_detection_b200.engine import Engine
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return Engine(0)


def test_cases_are_valid_plans():
    """Positions are distinct and inside the row, and the cases reach both sides of the shared-memory capacity."""
    counts = set()
    for make in CASES.values():
        for name, x, idx, fr in make():
            assert idx.size == fr.size and np.unique(idx).size == idx.size, name
            assert idx.size == 0 or (idx.min() >= 0 and idx.max() < x.shape[0]), name
            counts.add(idx.size)
    assert {0, 1, ISD_CAP - 1, ISD_CAP, ISD_CAP + 1} <= counts and max(counts) > 2 * ISD_CAP


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_algo5_is_algo2_of_algo1(eng, case):
    """rb_process(5) == rb_process(2) on rb_process(1)'s result, bit for bit, and nothing past a row is written."""
    import torch
    rows = CASES[case]()
    x, lengths, bp = batch(rows)
    xd = torch.from_numpy(x).cuda()
    ln = torch.from_numpy(lengths).cuda()
    dp = eng.upload_plan(bp)

    def run(algo, src):
        out = torch.full_like(xd, float(SENTINEL))
        eng.process(algo, src, ln, dp, out=out)
        torch.cuda.synchronize()
        return out

    y5 = run(5, xd).cpu().numpy()
    y1 = run(1, xd)
    y2 = run(2, y1).cpu().numpy()
    for u, (name, w, idx, fr) in enumerate(rows):
        L = w.shape[0]
        got, want = bits(y5[u, :L]), bits(y2[u, :L])
        diff = np.flatnonzero(got != want)
        assert diff.size == 0, (f"{case}/{name} (L={L}, n={idx.size}): {diff.size} samples differ, first at {diff[0]}: "
                                f"algo 5 {y5[u, diff[0]]!r}, algo 2(1) {y2[u, diff[0]]!r}")
        assert np.all(bits(y5[u, L:]) == bits(SENTINEL)), f"{case}/{name}: written past its length"
    if case == "loud":  # both normalisations fire: the first on the loud input, the second on the impulses past full scale
        y1h = y1.cpu().numpy()
        for u, (name, w, idx, fr) in enumerate(rows):
            assert np.max(np.abs(y1h[u, :w.shape[0]])) == 1.0 and np.max(np.abs(y5[u, :w.shape[0]])) == 1.0, name
            assert not np.array_equal(y5[u, :w.shape[0]][np.setdiff1d(np.arange(w.shape[0]), idx)],
                                      y1h[u, :w.shape[0]][np.setdiff1d(np.arange(w.shape[0]), idx)]), name

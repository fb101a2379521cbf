"""Effective support of the LnL and SSI filters: the edge taps the kernels skip (plans.tap_support, rb_tap_support, rb_set_tap_trim).

A filter b[0..K) runs over b[lo:hi): lo is the largest count whose |b| sum to at most eps/2 * sum|b|, hi the same rule from the
other end, eps = 2^-30. Dropping taps of total mass delta moves every output by at most delta * ||x^p||_inf, so trimming changes a
filter's output by at most eps * ||b||_1 * ||x^p||_inf: 1/64 of what rounding the taps to float32 already allows.

CPU: the numpy rule (symmetric on the symmetric notch cascades, never trims taps whose edges matter, the share it trims at the
default arguments, the float64 operator bound). GPU: the device rule equals numpy's bit for bit on drawn plans; hand-built filters
with tiny, asymmetric edges run aligned; trim on against trim off on the bench workload.
"""
import numpy as np
import pytest

from oracle import rawboost_oracle as orc  # noqa: E402  (checker only)
from scl_deepfake_audio_detection_b200 import plans, workload

from test_gpu_fir_bank import C_DENSE, Row, edge_taps, ratio, reference, run_rows

EPS = plans.TAP_TRIM_EPS
U = 2.0 ** -24


def notch_bank(n_utt, seed0=1234):
    """Taps of the default-args LnL filters of n_utt utterances, as float32 rounds them: a list of float64 arrays."""
    a = orc.make_args()
    out = []
    for u in range(n_utt):
        np.random.seed(seed0 + u)
        for _ in range(a.N_f):
            b = orc.draw_notch_taps(a.nBands, a.minF, a.maxF, a.minBW, a.maxBW, a.minCoeff, a.maxCoeff, a.minBiasLinNonLin,
                                    a.maxBiasLinNonLin, workload.SAMPLE_RATE)
            out.append(np.asarray(b, np.float32).astype(np.float64))
    return out


def csr(filters):
    off = np.concatenate([[0], np.cumsum([f.shape[0] for f in filters])]).astype(np.int32)
    return np.concatenate(filters).astype(np.float32), off


def fir(x, b):
    return orc.filter_fir_closed_form(x, b)


# ---------------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------------
def test_support_is_symmetric_on_notch_cascades():
    bank = notch_bank(60)
    taps, off = csr(bank)
    sup = plans.tap_support(taps, off)
    K = np.diff(off)
    assert np.array_equal(sup[:, 0], K - sup[:, 1])
    assert np.all(sup[:, 0] < sup[:, 1])


def test_support_trims_a_quarter_of_the_default_taps():
    bank = notch_bank(200)
    taps, off = csr(bank)
    sup = plans.tap_support(taps, off)
    share = 1.0 - float((sup[:, 1] - sup[:, 0]).sum()) / float(taps.shape[0])
    print(f"default-args notch taps trimmed at eps = 2^-30: {100 * share:.1f} %")
    assert 0.22 <= share <= 0.27


def test_support_never_trims_taps_whose_edges_matter():
    rs = np.random.RandomState(7)
    filters = [edge_taps(rs, K) for K in (1, 2, 3, 4, 5, 7, 24, 25, 48, 511, 512, 513, 1025, 2049) for _ in range(8)]
    taps, off = csr(filters)
    sup = plans.tap_support(taps, off)
    assert np.array_equal(sup[:, 0], np.zeros(len(filters))) and np.array_equal(sup[:, 1], np.diff(off))


def test_support_rule_at_the_edges():
    """Exact zeros at the ends go, an all-zero filter keeps nothing, a non-finite one keeps everything, and the rule follows the
    taps rather than assuming symmetry."""
    taps, off = csr([np.array([0.0, 0.0, 1.0, 0.0]), np.zeros(5), np.array([1e-12, 1.0, np.inf, 1e-12]),
                     np.array([1e-13] * 7 + [1.0] * 20 + [1e-13] * 3), np.array([1.0, 1e-9, 1.0])])
    sup = plans.tap_support(taps, off)
    assert sup.tolist() == [[2, 3], [0, 0], [0, 4], [7, 27], [0, 3]]


def test_trimmed_filter_within_the_operator_bound():
    """float64: ||FIR(x, b) - FIR(x, b_kept)||_inf <= eps ||b||_1 ||x||_inf on random rows."""
    rs = np.random.RandomState(11)
    bank = notch_bank(8, seed0=77)
    taps, off = csr(bank)
    sup = plans.tap_support(taps, off)
    for b, (lo, hi) in zip(bank, sup):
        x = rs.uniform(-1, 1, 3000) * rs.uniform(0.1, 3)
        kept = np.zeros_like(b)
        kept[lo:hi] = b[lo:hi]
        d = np.max(np.abs(fir(x, b) - fir(x, kept)))
        assert d <= EPS * np.abs(b).sum() * np.abs(x).max()


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


def _bench_batch(eng, algo, B):
    import torch
    lens = np.full(B, workload.UTT_LEN, np.int32)
    seeds = np.array([workload.seed_for(u) for u in range(B)], np.uint32)
    waves = [workload.synth_utterance(u, workload.UTT_LEN, bool(u % 2)) for u in range(B)]
    x, ln = eng.pack_waveforms(waves)
    dp = eng.draw_device_plan(torch.from_numpy(lens).to(eng.device), seeds, workload.SAMPLE_RATE, workload.default_args(), algo,
                              int(x.shape[1]))
    return waves, x, ln, dp


@pytest.mark.gpu
@pytest.mark.parametrize("planner", ["native", "device"])
def test_device_support_equals_numpy(eng, planner):
    """rb_tap_support against plans.tap_support on the LnL and SSI taps of 4096 default plans (the taps each planner drew)."""
    import torch
    B = 4096
    if planner == "device":
        lens = torch.full((B,), workload.UTT_LEN, dtype=torch.int32, device=eng.device)
        seeds = np.arange(B, dtype=np.uint32) + 99
        bp = eng.download_plan(eng.draw_device_plan(lens, seeds, workload.SAMPLE_RATE, workload.default_args(), 4, workload.UTT_LEN))
    else:
        from scl_deepfake_audio_detection_b200.native_planner import NativePlanner
        bp = NativePlanner().draw(np.full(B, workload.UTT_LEN, np.int32), workload.SAMPLE_RATE, workload.default_args(), 4,
                                  seeds=np.arange(B) + 99, copy=True)  # the planner's own buffers go with it
    for taps, off in ((bp.lnl_taps, bp.lnl_tap_off), (bp.ssi_taps, bp.ssi_tap_off)):
        want = plans.tap_support(taps, off)
        got = eng.tap_support(torch.from_numpy(np.ascontiguousarray(taps)).to(eng.device),
                              torch.from_numpy(np.ascontiguousarray(off)).to(eng.device)).cpu().numpy()
        assert np.array_equal(got, want), np.flatnonzero(np.any(got != want, axis=1))[:10]
        trimmed = 1.0 - float((want[:, 1] - want[:, 0]).sum()) / float(off[-1])
        print(f"{planner}: {want.shape[0]} filters, {100 * trimmed:.1f} % of the taps trimmed")


ALIGN_KS = [14, 23, 24, 25, 27, 28, 29, 47, 48, 49, 511, 512, 513, 514, 521, 1024, 1025, 1537]


def tiny_edges(rs, K, lead=7, trail=3):
    """edge_taps with the first `lead` and last `trail` taps scaled by 1e-13 and unit-size taps next to them."""
    b = edge_taps(rs, K)
    for i in (lead, K - 1 - trail):
        if abs(b[i]) * np.sqrt(K) < 0.5:
            b[i] = np.sign(b[i] or 1.0) * 0.5 / np.sqrt(K)
    b[:lead] *= 1e-13
    b[K - trail:] *= 1e-13
    return b.astype(np.float32).astype(np.float64)


def kept(b):
    lo, hi = plans.tap_support(b, [0, b.shape[0]])[0]
    out = np.zeros_like(b)
    out[lo:hi] = b[lo:hi]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("algo", [1, 3, 5])
def test_trimmed_filters_run_aligned(eng, algo):
    """Filters with tiny edges of unequal length across the 4-tap group, 24-tap body and 512-tap segment boundaries: within the
    per-sample bound of the float64 reference over the kept taps, and within eps ||b||_1 ||x^p||_inf of the full-tap one."""
    rs = np.random.RandomState(4000 + algo)
    rows = []
    for r, K in enumerate(ALIGN_KS):
        L = (7681, 2561, 5121)[r % 3]
        x = ((1.1 + 0.2 * rs.rand()) * rs.uniform(-1, 1, L)).astype(np.float32)
        row = Row(x=x)
        if algo in (1, 5):
            row.lnl = [tiny_edges(rs, K), tiny_edges(rs, ALIGN_KS[(r + 5) % len(ALIGN_KS)], lead=2, trail=9)]
        if algo == 5:
            n = int(rs.randint(1, L // 4))
            row.isd_idx = rs.permutation(L)[:n].astype(np.int64)
            row.isd_fr = (2 * rs.rand(n) - 1) * (2 * rs.rand(n) - 1)
        if algo == 3:
            row.noise = rs.standard_normal(L).astype(np.float32)
            row.ssi_taps = tiny_edges(rs, K, lead=1 + r % 9, trail=1 + (r * 5) % 9)
            row.snr = float(np.float32(rs.uniform(0, 20)))
        rows.append(row)
    got = run_rows(eng, algo, rows)
    for r, (row, g) in enumerate(zip(rows, got)):
        trimmed = Row(x=row.x, lnl=[kept(b) for b in row.lnl], isd_idx=row.isd_idx, isd_fr=row.isd_fr, noise=row.noise,
                      ssi_taps=None if row.ssi_taps is None else kept(row.ssi_taps), snr=row.snr)
        assert all(not np.array_equal(k, b) for k, b in zip(trimmed.lnl, row.lnl))
        y, tol = reference(trimmed, algo, C_DENSE)
        q = ratio(np.abs(g.astype(np.float64) - y), tol)
        assert q <= 1.0, f"row {r}: err/tol {q:.3g} against the kept taps"
        yf, tolf = reference(row, algo, C_DENSE)
        if algo == 3:
            delta = EPS * np.abs(row.ssi_taps).sum() * np.abs(row.noise).max() * np.abs(yf - row.x).max() / max(
                np.abs(fir(row.noise, row.ssi_taps)).max(), 1e-30)
        else:
            delta = EPS * sum(np.abs(b).sum() * np.abs(np.power(row.x, f + 1)).max() for f, b in enumerate(row.lnl)) * 3.0
        assert np.max(np.abs(g - yf)) <= np.max(tolf) + 4 * delta, f"row {r}"


@pytest.mark.gpu
@pytest.mark.parametrize("algo", [1, 3, 5])
def test_trim_on_against_off(eng, algo):
    """The bench workload (B = 4096, default arguments, device plans) with tap trimming on and off: per row, the difference is
    within the float32 rounding of the filter sums plus the trimmed mass (the two runs round differently where the trimmed
    taps shift the pairing of taps into the kernel's even / odd accumulators), and within the suite's 1e-5."""
    import torch
    B = 4096
    waves, x, ln, dp = _bench_batch(eng, algo, B)
    eng.set_tap_trim(False)
    full = eng.process(algo, x, ln, dp).clone()
    eng.set_tap_trim(True)
    trim = eng.process(algo, x, ln, dp).clone()
    torch.cuda.synchronize()
    full, trim = full.cpu().numpy(), trim.cpu().numpy()
    diff = np.abs(trim.astype(np.float64) - full)
    assert np.max(diff) <= 1e-5 * max(1.0, float(np.abs(full).max()))
    if algo in (1, 5):
        bp = eng.download_plan(dp)
        K = np.diff(bp.lnl_tap_off).reshape(B, bp.n_f)
        l1 = np.add.reduceat(np.abs(bp.lnl_taps.astype(np.float64)), bp.lnl_tap_off[:-1]).reshape(B, bp.n_f)
        l1[K == 0] = 0.0
        for u in range(0, B, 7):
            amax = float(np.abs(waves[u]).max())
            S = sum(l1[u, f] * amax ** (f + 1) for f in range(bp.n_f))
            bound = 3.0 * 2.0 * (EPS + 2 * C_DENSE * U) * S  # mean removal, ISD gain <= 1 + g_sd; normWav only divides
            assert diff[u].max() <= bound, (u, diff[u].max(), bound)
    same = float(np.mean(trim == full))
    print(f"algo {algo}: max |trim - full| {diff.max():.3e}, {100 * same:.2f} % of samples bit-identical")

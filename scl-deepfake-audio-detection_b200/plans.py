"""Host-side random parameters ("plans") of the RawBoost operators.

Everything random in the reference comes from the process-global legacy ``np.random`` stream
(``/root/reference/datautils/RawBoost.py:15,79,80,90``). The functions here issue *the same numpy calls in the
same order*, so after a plan is drawn the global stream is in exactly the state the reference would have left
it in, and the taps / impulse positions / noise are the very numbers the reference would have used. The CUDA
side (``engine``) only does arithmetic on them.

A :class:`BatchPlan` packs the per-utterance draws of a batch into the CSR arrays of ``struct rb_plan``
(``include/rawboost_b200.h``).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np
from scipy import signal

ALGO_USES_LNL = {1, 4, 5, 6, 8}
ALGO_USES_ISD = {2, 4, 5, 7, 8}
ALGO_USES_SSI = {3, 4, 6, 7}


# ------------------------------------------------------------------------------------------------------
# single draws (reference surface: randRange, genNotchCoeffs)
# ------------------------------------------------------------------------------------------------------
def randRange(x1, x2, integer):
    """``randRange`` (RawBoost.py:14-18): one size-(1,) uniform; ``int(...)`` truncation when ``integer``.

    Returns a shape-(1,) float64 array for the non-integer case, like the reference."""
    y = np.random.uniform(low=x1, high=x2, size=(1,))
    if integer:
        return int(y[0])
    return y


def genNotchCoeffs(nBands, minF, maxF, minBW, maxBW, minCoeff, maxCoeff, minG, maxG, fs):
    """``genNotchCoeffs`` (RawBoost.py:28-48): taps of a cascade of ``nBands`` random band-stop FIRs.

    Host float64, by design (SURVEY.md 8a-3): both sides must see identical coefficients. Per band the stream
    yields centre frequency, bandwidth and tap count (forced odd); the stages are Hamming-windowed two-cutoff
    ``firwin`` designs convolved together; one more uniform gives the gain in dB; the cascade is normalised by
    its peak magnitude response on ``freqz``'s default grid."""
    half = fs / 2
    cascade = np.array([1.0])
    for _ in range(int(nBands)):
        fc = float(randRange(minF, maxF, 0)[0])
        bw = float(randRange(minBW, maxBW, 0)[0])
        n = randRange(minCoeff, maxCoeff, 1)
        n += (n % 2 == 0)
        lo, hi = fc - bw / 2, fc + bw / 2
        lo = lo if lo > 0 else 1 / 1000
        hi = hi if hi < half else half - 1 / 1000
        cascade = np.convolve(signal.firwin(n, [lo, hi], window="hamming", fs=fs), cascade)
    gain_db = float(randRange(minG, maxG, 0)[0])
    _, response = signal.freqz(cascade, 1, fs=fs)
    return pow(10, gain_db / 20) * cascade / np.amax(np.abs(response))


# ------------------------------------------------------------------------------------------------------
# per-utterance plans
# ------------------------------------------------------------------------------------------------------
@dataclass
class UtterancePlan:
    """The draws one ``process_Rawboost_feature`` call makes, in order; unused parts stay ``None``."""
    length: int
    lnl_taps: Optional[List[np.ndarray]] = None   # N_f float64 tap vectors
    isd_idx: Optional[np.ndarray] = None          # int64 positions
    isd_fr: Optional[np.ndarray] = None           # float64 gains
    ssi_noise: Optional[np.ndarray] = None        # float64 white noise, length ``length``
    ssi_taps: Optional[np.ndarray] = None
    ssi_snr_db: Optional[float] = None
    g_sd: float = 0.0                             # ISD gain (an argument, not a draw)


def draw_lnl(N_f, nBands, minF, maxF, minBW, maxBW, minCoeff, maxCoeff, minG, maxG, minBiasLinNonLin, maxBiasLinNonLin, fs):
    """The N_f cascades of LnL (RawBoost.py:61-65). The gain window moves down once, before the 2nd order."""
    taps = []
    for order in range(int(N_f)):
        if order == 1:
            minG, maxG = minG - minBiasLinNonLin, maxG - maxBiasLinNonLin
        taps.append(genNotchCoeffs(nBands, minF, maxF, minBW, maxBW, minCoeff, maxCoeff, minG, maxG, fs))
    return taps


def draw_isd(length, P):
    """Impulse positions and gains of ISD (RawBoost.py:74,77-80)."""
    beta = float(randRange(0, P, 0)[0])
    n = int(length * (beta / 100))
    idx = np.random.permutation(length)[:n]
    f_r = np.multiply((2 * np.random.rand(idx.shape[0])) - 1, (2 * np.random.rand(idx.shape[0])) - 1)
    return idx, f_r


def draw_ssi(length, SNRmin, SNRmax, nBands, minF, maxF, minBW, maxBW, minCoeff, maxCoeff, minG, maxG, fs):
    """White noise, one cascade and the SNR of SSI (RawBoost.py:90-91,94)."""
    noise = np.random.normal(0, 1, length)
    taps = genNotchCoeffs(nBands, minF, maxF, minBW, maxBW, minCoeff, maxCoeff, minG, maxG, fs)
    snr = float(randRange(SNRmin, SNRmax, 0)[0])
    return noise, taps, snr


def draw_for_algo(length: int, sr, args, algo: int) -> UtterancePlan:
    """All draws of ``process_Rawboost_feature(feature, sr, args, algo)`` for one utterance of ``length``
    samples, in the dispatcher's order (asvspoof_2019_augall_3.py:377-439): LnL, then ISD, then SSI."""
    a = args
    plan = UtterancePlan(length=int(length))
    if algo in ALGO_USES_LNL:
        plan.lnl_taps = draw_lnl(a.N_f, a.nBands, a.minF, a.maxF, a.minBW, a.maxBW, a.minCoeff, a.maxCoeff, a.minG, a.maxG,
                                 a.minBiasLinNonLin, a.maxBiasLinNonLin, sr)
    if algo in ALGO_USES_ISD:
        plan.isd_idx, plan.isd_fr = draw_isd(plan.length, a.P)
        plan.g_sd = float(a.g_sd)
    if algo in ALGO_USES_SSI:
        plan.ssi_noise, plan.ssi_taps, plan.ssi_snr_db = draw_ssi(plan.length, a.SNRmin, a.SNRmax, a.nBands, a.minF, a.maxF,
                                                                  a.minBW, a.maxBW, a.minCoeff, a.maxCoeff, a.minG, a.maxG, sr)
    return plan


# ------------------------------------------------------------------------------------------------------
# batch packing
# ------------------------------------------------------------------------------------------------------
def padded_ld(max_len: int) -> int:
    """Row stride for a batch whose longest utterance has ``max_len`` samples (multiple of 4, >= 4)."""
    return max(4, (int(max_len) + 3) // 4 * 4)


@dataclass
class BatchPlan:
    """CSR-packed plans of a batch, host numpy arrays laid out as ``struct rb_plan`` expects."""
    B: int
    ld: int
    lengths: np.ndarray                       # int32 [B]
    n_f: int = 0
    lnl_taps: Optional[np.ndarray] = None     # float32 [sum K]
    lnl_tap_off: Optional[np.ndarray] = None  # int32 [B*n_f+1]
    isd_off: Optional[np.ndarray] = None      # int32 [B+1]
    isd_idx: Optional[np.ndarray] = None      # int32 [sum n]
    isd_fr: Optional[np.ndarray] = None       # float64 [sum n]
    g_sd: float = 0.0
    ssi_noise: Optional[np.ndarray] = None    # float32 [B, ld]
    ssi_taps: Optional[np.ndarray] = None     # float32
    ssi_tap_off: Optional[np.ndarray] = None  # int32 [B+1]
    ssi_snr_db: Optional[np.ndarray] = None   # float32 [B]

    # -- workload figures used by bench.py's roofline arithmetic (actual taps / impulses, never padded) --
    def fir_flops(self) -> float:
        """Algorithmic FLOPs of the FIR work: sum over filters of 2 * len * K."""
        total = 0.0
        if self.lnl_tap_off is not None:
            k = np.diff(self.lnl_tap_off.astype(np.int64)).reshape(self.B, self.n_f).sum(axis=1)
            total += float(2.0 * (k * self.lengths.astype(np.int64)).sum())
        if self.ssi_tap_off is not None:
            k = np.diff(self.ssi_tap_off.astype(np.int64))
            total += float(2.0 * (k * self.lengths.astype(np.int64)).sum())
        return total

    def io_bytes(self) -> float:
        """Algorithmic HBM bytes: waveform in + out (+ noise in, + 8 B... per impulse: idx + f_r)."""
        n = float(self.lengths.astype(np.int64).sum())
        total = 8.0 * n
        if self.ssi_noise is not None:
            total += 4.0 * n
        if self.isd_idx is not None:
            total += 12.0 * float(self.isd_idx.shape[0])
        return total


def pack(plans: Sequence[UtterancePlan], ld: Optional[int] = None) -> BatchPlan:
    """Pack per-utterance plans (all drawn for the same algo and arguments) into one :class:`BatchPlan`."""
    B = len(plans)
    lengths = np.array([p.length for p in plans], dtype=np.int32)
    if ld is None:
        ld = padded_ld(int(lengths.max()) if B else 0)
    bp = BatchPlan(B=B, ld=int(ld), lengths=lengths, g_sd=float(plans[0].g_sd) if B else 0.0)
    if B == 0:
        return bp
    first = plans[0]
    if first.lnl_taps is not None:
        bp.n_f = len(first.lnl_taps)
        flat = [t for p in plans for t in p.lnl_taps]
        if any(len(p.lnl_taps) != bp.n_f for p in plans):
            raise ValueError("all utterances of a batch must use the same N_f")
        sizes = np.array([t.shape[0] for t in flat], dtype=np.int64)
        bp.lnl_tap_off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
        bp.lnl_taps = np.concatenate(flat).astype(np.float32)
    if first.isd_idx is not None:
        sizes = np.array([p.isd_idx.shape[0] for p in plans], dtype=np.int64)
        bp.isd_off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
        bp.isd_idx = np.concatenate([p.isd_idx for p in plans]).astype(np.int32)
        bp.isd_fr = np.concatenate([p.isd_fr for p in plans]).astype(np.float64)
    if first.ssi_noise is not None:
        noise = np.zeros((B, bp.ld), dtype=np.float32)
        for u, p in enumerate(plans):
            noise[u, :p.length] = p.ssi_noise
        bp.ssi_noise = noise
        sizes = np.array([p.ssi_taps.shape[0] for p in plans], dtype=np.int64)
        bp.ssi_tap_off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
        bp.ssi_taps = np.concatenate([p.ssi_taps for p in plans]).astype(np.float32)
        bp.ssi_snr_db = np.array([p.ssi_snr_db for p in plans], dtype=np.float32)
    return bp


def _offsets(sizes) -> np.ndarray:
    return np.concatenate([[0], np.cumsum(np.asarray(sizes, dtype=np.int64))]).astype(np.int32)


def concat(parts: Sequence[BatchPlan], ld: Optional[int] = None) -> BatchPlan:
    """Concatenate packed plans (all drawn for the same algo, ``N_f`` and ``g_sd``) into one :class:`BatchPlan` of stride
    ``ld`` (default: the largest stride of the parts). Every field is carried; the SSI noise rows are re-laid to ``ld``."""
    if not parts:
        raise ValueError("nothing to concatenate")
    first = parts[0]
    ld = int(ld if ld is not None else max(p.ld for p in parts))
    if any(p.n_f != first.n_f or p.g_sd != first.g_sd for p in parts):
        raise ValueError("all plans of a batch must share N_f and g_sd")
    lengths = np.concatenate([np.asarray(p.lengths, dtype=np.int32) for p in parts])
    if lengths.size and int(lengths.max()) > ld:
        raise ValueError(f"an utterance of {int(lengths.max())} samples does not fit the stride ld={ld}")
    out = BatchPlan(B=int(lengths.shape[0]), ld=ld, lengths=lengths, n_f=first.n_f, g_sd=first.g_sd)
    for name in ("lnl_tap_off", "isd_off", "ssi_tap_off"):
        if any((getattr(p, name) is None) != (getattr(first, name) is None) for p in parts):
            raise ValueError(f"{name} is set in some plans of the batch and missing in others")
    if first.lnl_tap_off is not None:
        out.lnl_taps = np.concatenate([p.lnl_taps for p in parts]).astype(np.float32, copy=False)
        out.lnl_tap_off = _offsets(np.concatenate([np.diff(p.lnl_tap_off) for p in parts]))
    if first.isd_off is not None:
        out.isd_idx = np.concatenate([p.isd_idx for p in parts]).astype(np.int32, copy=False)
        out.isd_fr = np.concatenate([p.isd_fr for p in parts]).astype(np.float64, copy=False)
        out.isd_off = _offsets(np.concatenate([np.diff(p.isd_off) for p in parts]))
    if first.ssi_tap_off is not None:
        out.ssi_noise = np.zeros((out.B, ld), dtype=np.float32)
        row = 0
        for p in parts:
            for u in range(p.B):
                n = int(p.lengths[u])
                out.ssi_noise[row, :n] = p.ssi_noise[u, :n]
                row += 1
        out.ssi_taps = np.concatenate([p.ssi_taps for p in parts]).astype(np.float32, copy=False)
        out.ssi_tap_off = _offsets(np.concatenate([np.diff(p.ssi_tap_off) for p in parts]))
        out.ssi_snr_db = np.concatenate([p.ssi_snr_db for p in parts]).astype(np.float32, copy=False)
    return out


def draw_batch(lengths: Sequence[int], sr, args, algo: int, seeds: Optional[Sequence[int]] = None,
               ld: Optional[int] = None) -> BatchPlan:
    """Draw and pack the plans of a batch. With ``seeds`` the global stream is re-seeded before each utterance
    (the benchmark's convention, SURVEY.md 8d); without, utterances simply consume the stream one after another,
    which is what a loader calling the reference once per view does."""
    plans = []
    for u, n in enumerate(lengths):
        if seeds is not None:
            np.random.seed(int(seeds[u]))
        plans.append(draw_for_algo(int(n), sr, args, algo))
    return pack(plans, ld=ld)

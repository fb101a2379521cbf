"""Drop-in for the reference's ``datautils/RawBoost.py`` operator surface, computed on a B200.

Same names, argument order and RNG behaviour as ``/root/reference/datautils/RawBoost.py:14-97`` and the
``process_Rawboost_feature`` / ``RawBoost12`` pair every loader defines
(``/root/reference/datautils/asvspoof_2019_augall_3.py:359-439``):

* every random number is drawn on the host from the process-global legacy ``np.random`` stream by the same
  numpy calls in the same order (see :mod:`plans`), so downstream draws of the loader stay bit-identical;
* inputs are 1-D numpy arrays of any length and are never mutated; results are NEW 1-D arrays of the same
  length (``algo`` 0 returns the input object itself, as the reference does);
* the arithmetic runs in the CUDA library. Results are float32 -- the reference returns float64 for every
  algo but 0 and 2 and its loaders cast to float32 immediately (asvspoof_2019_augall_3.py:142). ISD and
  normWav on float32 input are bit-exact; the FIR-based operators agree within 1e-5 max-abs.

These per-utterance calls pay a host->device->host round trip each; the loaders' throughput path is the batched
API in :mod:`engine` (draw plans in the workers, apply them on the collated batch in the main process).
There is no CPU fallback: without the built library and a CUDA device these functions raise.

In a DataLoader worker forked after the parent initialised CUDA, CUDA cannot be used. When the parent serves the workers
(``dropin.serve_workers``, :mod:`broker`), such a process routes ``normWav``, ``filterFIR`` and every RawBoost application to
it: the draws stay here, on this process's numpy stream in the reference's order, and only the waveform and the drawn plan
travel; the result comes back as float32, with the same values and the same object rules as a call in the parent. Without a
broker these functions raise ``RawBoostLibraryError`` in such a process.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from . import _lib, broker as _broker, plans as _plans
from .engine import default_engine
from .plans import genNotchCoeffs, randRange  # noqa: F401  (part of the reference surface)

__all__ = [
    "randRange", "normWav", "genNotchCoeffs", "filterFIR", "LnL_convolutive_noise", "ISD_additive_noise",
    "SSI_additive_noise", "process_Rawboost_feature", "RawBoost12",
]

_DEVICE = None  # engine.default_device(): RAWBOOST_B200_DEVICE, shared with multiview / reverb
# Who issues the draws of the dispatcher: "native" (default) = the library's bit-exact C++ replica of the numpy calls, run
# on numpy's own global stream state (about 7x faster than numpy + scipy per utterance; integers, impulse gains, noise and the
# stream state after the call are identical, taps agree to ~1e-15 before the float32 cast); "numpy" = the numpy / scipy calls
# themselves (plans.py).
_PLANNER = os.environ.get("RAWBOOST_B200_PLANNER", "native")
_native = None


_ZERO_ARGS = dict(N_f=1, nBands=1, minF=0, maxF=0, minBW=0, maxBW=0, minCoeff=0, maxCoeff=0, minG=0, maxG=0, minBiasLinNonLin=0,
                  maxBiasLinNonLin=0, P=0, g_sd=0, SNRmin=0, SNRmax=0)


def _draw_native(length, fs, algo, **knobs):
    """One operator's draws by the native planner on numpy's global stream (only the knobs the operator reads matter)."""
    from types import SimpleNamespace
    kw = dict(_ZERO_ARGS)
    kw.update(knobs)
    return _native_planner().draw([length], fs, SimpleNamespace(**kw), algo, use_global_stream=True)


def _native_planner():
    global _native
    if _native is None or _native[0] != os.getpid():
        from .native_planner import NativePlanner
        if _native is not None:
            _native[1]._h = None  # inherited through fork: this process makes its own (no CUDA call) and leaves the parent's be
        planner = NativePlanner(threads=1, pinned=False)
        planner.self_check()  # once per process: refuse loudly if this numpy's stream is not the one the replica implements
        _native = (os.getpid(), planner)
    return _native[1]


def _engine():
    """The process's engine; refused with a pointer to the broker in a process forked after CUDA was initialised."""
    if torch.cuda._is_in_bad_fork():
        raise _lib.RawBoostLibraryError(
            "CUDA cannot be used in a process forked after its parent initialised CUDA (a DataLoader worker); call "
            "dropin.serve_workers() in the parent before the loader starts its workers, so that this process sends its "
            "RawBoost calls there, or run the loader with num_workers=0 or multiprocessing_context='spawn'")
    return default_engine(_DEVICE)


def _as_wave(x):
    x = np.asarray(x)
    if x.ndim != 1:
        raise ValueError(f"RawBoost operators take 1-D waveforms, got shape {x.shape}")
    return x


def _run_single(algo, x, plan):
    """One utterance through the host-buffer entry (``rb_process_host``: ONE C call copies the waveform and the plan in, runs
    the kernels and copies the result out): returns a new float32 array of x's length. ``plan``: an ``UtterancePlan`` or an
    already packed one-utterance ``BatchPlan``. Routed to the broker in a worker process (:mod:`broker`)."""
    n = x.shape[0]
    if n == 0:
        return np.zeros(0, dtype=np.float32)
    bp = plan if isinstance(plan, _plans.BatchPlan) else (_plans.pack([plan]) if plan is not None else None)
    if _broker.routed():
        if bp is None:
            raise ValueError(f"algo {algo} needs a plan")
        key = ("rb", int(algo), int(bp.n_f), float(bp.g_sd), bp.ld > _broker.MASK_SMEM_MAX_LD)
        return _broker.request(key, np.ascontiguousarray(x, dtype=np.float32), bp)
    eng = _engine()
    ld = bp.ld if bp is not None else _plans.padded_ld(n)
    xh = np.zeros((1, ld), dtype=np.float32)
    xh[0, :n] = x  # (float64 input is rounded to float32 here, see the module docstring)
    y = eng.process_host(algo, xh, bp)
    return y[0, :n].copy()


def normWav(x, always):
    """``normWav`` (RawBoost.py:20-25). Returns the input object itself when no scaling applies, like numpy."""
    x = _as_wave(x)
    if x.shape[0] == 0:
        return x
    if _broker.routed():
        y = _broker.request(("norm", bool(always)), np.ascontiguousarray(x, dtype=np.float32), None)
    else:
        eng = _engine()
        xd, ld = eng.pack_waveforms([x])
        y = eng.normwav(xd, ld, bool(always))[0, :x.shape[0]].cpu().numpy()
    if not always and x.dtype == np.float32 and np.array_equal(y, x):
        return x
    return y


def filterFIR(x, b):
    """``filterFIR`` (RawBoost.py:51-56): y[n] = sum_k b[k] x[n + (K+1)//2 - k], zero-extended x."""
    x = _as_wave(x)
    b = np.asarray(b, dtype=np.float64).reshape(-1)
    if x.shape[0] == 0:
        return np.zeros(0, dtype=np.float32)
    if _broker.routed():
        return _broker.request(("fir",), np.ascontiguousarray(x, dtype=np.float32), b.astype(np.float32))
    eng = _engine()
    xd, ld = eng.pack_waveforms([x])
    taps = torch.from_numpy(b.astype(np.float32)).to(eng.device)
    off = torch.tensor([0, b.shape[0]], dtype=torch.int32, device=eng.device)
    return eng.filter_fir(xd, ld, taps, off)[0, :x.shape[0]].cpu().numpy()


def LnL_convolutive_noise(x, N_f, nBands, minF, maxF, minBW, maxBW, minCoeff, maxCoeff, minG, maxG, minBiasLinNonLin,
                          maxBiasLinNonLin, fs):
    """Linear and non-linear convolutive noise (RawBoost.py:59-69)."""
    x = _as_wave(x)
    if _PLANNER == "native" and x.shape[0] > 0:
        return _run_single(1, x, _draw_native(x.shape[0], fs, 1, N_f=N_f, nBands=nBands, minF=minF, maxF=maxF, minBW=minBW, maxBW=maxBW,
                                              minCoeff=minCoeff, maxCoeff=maxCoeff, minG=minG, maxG=maxG,
                                              minBiasLinNonLin=minBiasLinNonLin, maxBiasLinNonLin=maxBiasLinNonLin))
    plan = _plans.UtterancePlan(length=x.shape[0])
    plan.lnl_taps = _plans.draw_lnl(N_f, nBands, minF, maxF, minBW, maxBW, minCoeff, maxCoeff, minG, maxG, minBiasLinNonLin,
                                    maxBiasLinNonLin, fs)
    return _run_single(1, x, plan)


def ISD_additive_noise(x, P, g_sd):
    """Impulsive signal-dependent noise (RawBoost.py:73-84)."""
    x = _as_wave(x)
    if _PLANNER == "native" and x.shape[0] > 0:
        return _run_single(2, x, _draw_native(x.shape[0], 16000, 2, P=P, g_sd=g_sd))
    plan = _plans.UtterancePlan(length=x.shape[0])
    plan.isd_idx, plan.isd_fr = _plans.draw_isd(x.shape[0], P)
    plan.g_sd = float(g_sd)
    return _run_single(2, x, plan)


def SSI_additive_noise(x, SNRmin, SNRmax, nBands, minF, maxF, minBW, maxBW, minCoeff, maxCoeff, minG, maxG, fs):
    """Stationary signal-independent coloured noise (RawBoost.py:89-97)."""
    x = _as_wave(x)
    if _PLANNER == "native" and x.shape[0] > 0:
        return _run_single(3, x, _draw_native(x.shape[0], fs, 3, SNRmin=SNRmin, SNRmax=SNRmax, nBands=nBands, minF=minF, maxF=maxF,
                                              minBW=minBW, maxBW=maxBW, minCoeff=minCoeff, maxCoeff=maxCoeff, minG=minG, maxG=maxG))
    plan = _plans.UtterancePlan(length=x.shape[0])
    plan.ssi_noise, plan.ssi_taps, plan.ssi_snr_db = _plans.draw_ssi(x.shape[0], SNRmin, SNRmax, nBands, minF, maxF, minBW, maxBW,
                                                                     minCoeff, maxCoeff, minG, maxG, fs)
    return _run_single(3, x, plan)


def process_Rawboost_feature(feature, sr, args, algo):
    """The loaders' 9-way dispatcher (asvspoof_2019_augall_3.py:377-439), one fused device call per utterance.

    ``args`` needs the attributes of main.py:258-298 (N_f, nBands, minF, maxF, minBW, maxBW, minCoeff, maxCoeff,
    minG, maxG, minBiasLinNonLin, maxBiasLinNonLin, P, g_sd, SNRmin, SNRmax)."""
    if algo not in (1, 2, 3, 4, 5, 6, 7, 8):
        return feature
    x = _as_wave(feature)
    if _PLANNER == "native" and x.shape[0] > 0:
        plan = _native_planner().draw([x.shape[0]], sr, args, algo, use_global_stream=True)
    else:
        plan = _plans.draw_for_algo(x.shape[0], sr, args, algo)
    return _run_single(algo, x, plan)


def RawBoost12(x, args, sr=16000, audio_path=None):
    """Algo-5 wrapper the loaders call through ``globals()[name]`` (asvspoof_2019_augall_3.py:359-374).

    ``online_aug`` true: augment on the fly. Otherwise reuse / create ``<aug_dir>/RawBoost12/<utt>`` as 16-bit PCM;
    that cold branch needs ``librosa`` / ``soundfile`` exactly as the reference does."""
    if getattr(args, "online_aug", True):
        return process_Rawboost_feature(x, sr, args, algo=5)
    cache = os.path.join(args.aug_dir, "RawBoost12", os.path.basename(audio_path))
    if os.path.exists(cache):
        import librosa
        wav, _ = librosa.load(cache, sr=sr, mono=True)
        return wav
    import soundfile as sf
    wav = process_Rawboost_feature(x, sr, args, algo=5)
    sf.write(cache, wav, sr, subtype="PCM_16")
    return wav

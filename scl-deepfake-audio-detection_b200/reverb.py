"""Reverb view on the device (SURVEY.md 8f-4): the arithmetic of ``ReverbAugmentor.transform``
(``/root/reference/datautils/audio_augmentor/reverb.py:33-44``) -- a full convolution of the waveform with a room impulse
response followed by peak normalisation. Two device paths:

* ``reverb_batch`` / ``reverb_convolve`` (host waveforms): the FIR-bank kernel (long filters run as 512-tap segments) and the
  one-kernel ``normWav``;
* ``reverb_device`` / ``Engine.reverb`` (waveforms already on the device, C entry ``rb_reverb``): FFT overlap-save with
  8192-tap partitions, whose cost grows with the number of partitions rather than with every tap (DESIGN.md 4.5).

    reverberate = np.convolve(data, rir_data)            # length len(data) + len(rir) - 1
    reverberate /= np.max(np.abs(reverberate))

What stays with the caller, exactly as in the reference: choosing and loading the RIR file (``random.choice`` over the
corpus, ``librosa.load``) and the 16-bit pydub round trip of the augmentor framework. There is no CPU fallback.
"""
from __future__ import annotations

from typing import Sequence

import numpy as np
import torch

from .engine import Engine, default_engine
from .plans import padded_ld


def reverb_batch(eng: Engine, waves: Sequence[np.ndarray], rirs: Sequence[np.ndarray]):
    """``normWav(np.convolve(wave_u, rir_u), 1)`` for every utterance; returns ([B, ld] float32 device tensor, int32 lengths).

    filterFIR computes y[n] = sum_k b[k] x[n + (K+1)//2 - k] (RawBoost.py:51-56); feeding it the waveform delayed by
    (K+1)//2 samples and zero-extended to len + K - 1 turns that into the full convolution sum_k b[k] x[n - k]."""
    if len(waves) != len(rirs):
        raise ValueError("one impulse response per waveform")
    B = len(waves)
    rirs = [np.asarray(r, dtype=np.float32).reshape(-1) for r in rirs]
    out_len = np.array([w.shape[0] + r.shape[0] - 1 if w.shape[0] and r.shape[0] else 0 for w, r in zip(waves, rirs)], dtype=np.int32)
    shift = [(r.shape[0] + 1) // 2 for r in rirs]
    in_len = np.array([n + s if n else 0 for n, s in zip(out_len, shift)], dtype=np.int32)
    ld = padded_ld(int(in_len.max()) if B else 0)
    host = np.zeros((B, ld), dtype=np.float32)
    for u, (w, s) in enumerate(zip(waves, shift)):
        host[u, s:s + w.shape[0]] = np.asarray(w, dtype=np.float32)
    x = torch.from_numpy(host).to(eng.device)
    taps, off = pack_rirs(eng, rirs)
    # the kernel takes one length per row for both input and output: run over the delayed input's length; the outputs beyond
    # len + K - 1 are exact zeros (no tap reaches a sample there), so they do not disturb the peak
    ln_in = torch.from_numpy(in_len).to(eng.device)
    y = eng.filter_fir(x, ln_in, taps, off)
    return eng.normwav(y, ln_in, True), torch.from_numpy(out_len).to(eng.device)


def pack_rirs(eng: Engine, rirs: Sequence[np.ndarray]):
    """Host impulse responses -> (float32 taps, int32 CSR offsets [B + 1]) on the engine's device."""
    rirs = [np.asarray(r, dtype=np.float32).reshape(-1) for r in rirs]
    taps = np.concatenate(rirs) if rirs else np.zeros(0, np.float32)
    off = np.concatenate([[0], np.cumsum([r.shape[0] for r in rirs])]).astype(np.int32)
    return torch.from_numpy(taps).to(eng.device), torch.from_numpy(off).to(eng.device)


def reverb_device(eng: Engine, x: torch.Tensor, lengths: torch.Tensor, rirs: Sequence[np.ndarray], ld_out=None):
    """Reverb views of waveforms that already live on the device: x [B, ld] float32 and int32 lengths on ``eng.device``, one
    host impulse response per row (as the caller loads them from the RIR corpus). Returns ([B, ld_out] float32 device tensor,
    int32 device lengths len + K - 1). FFT overlap-save on the device (``Engine.reverb``); raises ``ValueError`` if a row could
    not be computed (an empty impulse response, or ``ld_out`` too small for its result)."""
    if len(rirs) != x.shape[0]:
        raise ValueError("one impulse response per waveform")
    taps, off = pack_rirs(eng, rirs)
    y, out_len = eng.reverb(x, lengths, taps, off, ld_out=ld_out, max_taps=max((len(r) for r in rirs), default=1))
    if ld_out is not None:
        bad = np.flatnonzero(out_len.cpu().numpy() < 0)
        if bad.size:
            raise ValueError(f"rows {bad.tolist()[:8]} were not computed: empty impulse response or ld_out={ld_out} too small")
    return y, out_len


def reverb_convolve(data, rir_data) -> np.ndarray:
    """One utterance: float32 array of length ``len(data) + len(rir_data) - 1``, peak-normalised like the reference."""
    data = np.asarray(data).reshape(-1)
    rir_data = np.asarray(rir_data).reshape(-1)
    if data.shape[0] == 0 or rir_data.shape[0] == 0:
        raise ValueError("reverb_convolve needs a non-empty waveform and impulse response (np.convolve raises too)")
    y, ln = reverb_batch(default_engine(), [data], [rir_data])
    return y[0, :int(ln[0])].cpu().numpy()

"""CPU restatement of the time-stretch and pitch-shift attacks (aware_b200.attacks.TimeStretch /
PitchShift).  TEST INFRASTRUCTURE ONLY, like oracle/aware_oracle.py; nothing under aware_b200/
imports it.

Parity status: UNPINNED to the upstream attacks, which call rubberband (scripts/attacks.py:150-252)
and have no arithmetic to follow.  The attacks are defined by this file: the classical phase vocoder
of librosa.effects.time_stretch / pitch_shift in the project's STFT conventions (DESIGN.md section 7).
The STFT and iSTFT are torch's on the CPU, the phase vocoder is numpy float64 (a loop over frames,
vectorised over bins), the resample is scipy.signal.resample_poly.
"""
from __future__ import annotations

import math
from fractions import Fraction

import numpy as np
import torch

N_FFT, HOP, N_BINS = 1024, 256, 513


def stft(x) -> torch.Tensor:
    """complex64 [513, T], T = 1 + N // 256, of a float32 clip as it is (no normalisation)."""
    x = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))
    return torch.stft(x, n_fft=N_FFT, hop_length=HOP, window=torch.hann_window(N_FFT), center=True,
                      pad_mode="reflect", return_complex=True)


def istft(spec, length: int) -> np.ndarray:
    """float32 [length] from a complex64 [513, T] spectrum (torch.istft with `length`)."""
    spec = torch.as_tensor(np.asarray(spec, dtype=np.complex64))
    return torch.istft(spec, n_fft=N_FFT, hop_length=HOP, window=torch.hann_window(N_FFT), center=True,
                       length=int(length)).numpy()


def phase_vocoder(D, rate: float) -> np.ndarray:
    """librosa.phase_vocoder(D, rate, hop_length=256) with every operation in float64:
    complex64 [513, T] -> complex64 [513, len(np.arange(0, T, rate))]."""
    D = np.asarray(D, dtype=np.complex64)
    nb, T = D.shape
    steps = np.arange(0, T, rate, dtype=np.float64)
    Dp = np.concatenate([D, np.zeros((nb, 2), dtype=np.complex64)], axis=1)   # two zero frames
    re, im = Dp.real.astype(np.float64), Dp.imag.astype(np.float64)
    mags, angs = np.hypot(re, im), np.arctan2(im, re)
    phi = (np.pi / 2) * np.arange(nb, dtype=np.float64)                          # hop * 2 pi k / n_fft
    two_pi = 2.0 * np.pi
    acc = angs[:, 0].copy()
    out = np.empty((nb, len(steps)), dtype=np.complex64)
    for t, s in enumerate(steps):
        i = int(s)
        alpha = s - i
        mag = (1.0 - alpha) * mags[:, i] + alpha * mags[:, i + 1]
        out[:, t].real = mag * np.cos(acc)
        out[:, t].imag = mag * np.sin(acc)
        dphi = angs[:, i + 1] - angs[:, i] - phi
        dphi = dphi - two_pi * np.rint(dphi / two_pi)
        acc = acc + (phi + dphi)
    return out


def attack_time_stretch(x, rate: float) -> np.ndarray:
    """TimeStretch(rate) of one clip: istft(phase_vocoder(stft(x), rate), length=round(N / rate))."""
    x = np.asarray(x, dtype=np.float32)
    return istft(phase_vocoder(stft(x).numpy(), rate), int(round(len(x) / rate)))


def pitch_ratio(n_steps, max_cents: float = 0.05) -> Fraction:
    """Smallest-denominator p / q (p = round(q r)) within max_cents of r = 2^(n_steps / 12)."""
    r = 2.0 ** (float(n_steps) / 12.0)
    q = 1
    while True:
        p = max(1, round(r * q))
        if abs(1200.0 * math.log2(p / (q * r))) <= max_cents:
            return Fraction(p, q)
        q += 1


def attack_pitch_shift(x, n_steps, max_cents: float = 0.05) -> np.ndarray:
    """PitchShift(n_steps) of one clip: time-stretch by 2^(-n_steps/12), resample_poly(., q, p) with
    p / q = pitch_ratio(n_steps) (skipped when p = q), truncate / zero-pad to len(x)."""
    from scipy.signal import resample_poly
    x = np.asarray(x, dtype=np.float32)
    y = attack_time_stretch(x, 2.0 ** (-float(n_steps) / 12.0))
    f = pitch_ratio(n_steps, max_cents)
    if f.numerator != f.denominator:
        y = resample_poly(y, f.denominator, f.numerator).astype(np.float32)
    out = np.zeros(len(x), dtype=np.float32)
    out[:min(len(x), len(y))] = y[:len(x)]
    return out

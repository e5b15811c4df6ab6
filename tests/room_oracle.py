"""Float64 restatement of the reverberation and echo attacks (aware_b200.attacks.Reverb / Echo).
TEST INFRASTRUCTURE ONLY, like oracle/aware_oracle.py; nothing under aware_b200/ imports it.

The attacks have no upstream counterpart.  They are defined in DESIGN.md section 7 as the causal
convolution y[n] = sum_{m < M} h[m] x[n - m], x[< 0] = 0, truncated to the input's length.  This file
states that definition directly (np.convolve / scipy.signal.fftconvolve) and once more as the
partitioned overlap-save bookkeeping the CUDA kernels follow, both in float64.
"""
from __future__ import annotations

import numpy as np

P = 512                          # partition length and hop
DECAY_60DB = 6.907755278982137   # ln(1000)


def synth_rir(rt60: float, sr: int, seed: int) -> np.ndarray:
    """The synthetic room impulse response of `Reverb`: float32 [round(rt60 sr)]."""
    M = int(round(rt60 * sr))
    g = np.random.default_rng(seed)
    h = g.standard_normal(M) * np.exp(-DECAY_60DB * np.arange(M) / (rt60 * sr))
    h[0] = 1.0
    h /= np.sqrt(np.sum(h * h))
    return h.astype(np.float32)


def echo_response(delay: float, decay: float, sr: int) -> np.ndarray:
    """The impulse response of `Echo`: float32 [D + 1] = [1, 0, ..., 0, decay], D = round(delay sr)."""
    D = int(round(delay * sr))
    h = np.zeros(D + 1, dtype=np.float32)
    h[0], h[D] = 1.0, decay
    return h


def convolve(x, h) -> np.ndarray:
    """float64 y = np.convolve(x, h)[:len(x)] (fftconvolve for long inputs, which agrees to ~1e-15)."""
    x = np.asarray(x, dtype=np.float64)
    h = np.asarray(h, dtype=np.float64)
    if len(x) * len(h) <= 5e7:
        return np.convolve(x, h)[:len(x)]
    from scipy.signal import fftconvolve
    return fftconvolve(x, h)[:len(x)]


def partitioned_convolve(x, h) -> np.ndarray:
    """float64 uniformly partitioned overlap-save with the kernels' block bookkeeping: input block b is
    x[512 (b-1), 512 (b+1)) (zero outside the clip), partition j is h[512 j, 512 j + 512) zero-padded to 1024,
    Y_b = sum_{j <= min(K-1, b)} X_{b-j} H_j in ascending j, and samples 512 .. 1023 of irfft(Y_b) are
    y[512 b, 512 b + 512)."""
    x = np.asarray(x, dtype=np.float64)
    h = np.asarray(h, dtype=np.float64)
    N, M = len(x), len(h)
    NB, K = -(-N // P), -(-M // P)
    xp = np.zeros(P * (NB + 1))
    xp[P:P + N] = x
    X = np.fft.rfft(np.stack([xp[P * b:P * b + 2 * P] for b in range(NB)]), axis=1)
    hp = np.zeros(P * K)
    hp[:M] = h
    H = np.fft.rfft(hp.reshape(K, P), n=2 * P, axis=1)
    y = np.zeros(P * NB)
    for b in range(NB):
        Y = np.zeros(P + 1, dtype=np.complex128)
        for j in range(min(K - 1, b) + 1):
            Y += X[b - j] * H[j]
        y[P * b:P * b + P] = np.fft.irfft(Y, n=2 * P)[P:]
    return y[:N]

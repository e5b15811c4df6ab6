"""Attack classes with the reference's `.apply(audio, sr)` / `.name` interface
(scripts/attacks.py there), executed by the batched CUDA kernels.

Each class also has `.apply_batch(x, sr, rng)` taking a CUDA float32 tensor
[n_clips, n_samples].  Randomness is explicit: start indices / band edges are drawn
from the numpy Generator passed in (or given directly), never from global state
(the reference draws from unseeded global RNGs, attacks.py:170,340,378).
Filter design (scipy.signal.butter / firwin / lfilter_zi) stays on the host; only
coefficients travel.  Upstream's MP3Compression / TimeStretch / PitchShift shell out to
ffmpeg / rubberband and have no arithmetic to restate.  MP3 is not provided (`CompressionApprox`
is an in-repo stand-in); `TimeStretch` / `PitchShift` are defined here as the classical phase
vocoder (parity unpinned to rubberband), with `desync_attacks()` as the set the evaluation
driver adds on request.  `Reverb` / `Echo` (room reverberation and echo, a partitioned FFT
convolution on the GPU) have no upstream counterpart; `room_attacks()` is the set the driver adds
on request.
"""
from __future__ import annotations

import math
from fractions import Fraction

import numpy as np
import torch

_engine = None


def set_engine(engine):
    """Engine used by `.apply()`; `load()`-ed embedders expose theirs as `embedder.engine`."""
    global _engine
    _engine = engine


def _eng(engine=None):
    if engine is not None:
        return engine
    if _engine is None:
        raise RuntimeError("aware_b200.attacks: call set_engine(embedder.engine) first")
    return _engine


def _warm_samples(b, a, tol: float = 1e-16) -> int:
    """Look-back length W for the chunk-parallel IIR: ignoring every input older than W
    samples changes an output by at most max|x| * sum_{m>W} |h[m]| (h = impulse response), so
    W is the smallest multiple of 256 whose impulse-response tail sum is below `tol`.
    (The pole radius alone under-estimates it: Butterworth band-stops have clustered poles
    whose response decays like n^3 r^n.)"""
    from scipy.signal import lfilter
    n = 1 << 14
    while True:
        imp = np.zeros(n)
        imp[0] = 1.0
        h = np.abs(lfilter(b, a, imp))
        tail = np.cumsum(h[::-1])[::-1]                  # tail[i] = sum_{m>=i} |h[m]|
        if not np.isfinite(tail[0]):
            raise ValueError("unstable filter")
        if tail[n // 2] < tol * 1e-3:                     # the truncated remainder is negligible
            w = int(np.argmax(tail < tol))
            return max(256, -(-w // 256) * 256)
        n *= 2
        if n > (1 << 22):
            raise ValueError("filter memory too long for the chunked scan")


class Attack:
    name = "attack"

    def apply_batch(self, x: torch.Tensor, sr: int, rng=None, engine=None) -> torch.Tensor:
        raise NotImplementedError

    def apply(self, audio, sr):
        """Single clip, numpy in -> numpy float32 out (reference calling convention)."""
        eng = _eng()
        x = torch.from_numpy(np.ascontiguousarray(audio, dtype=np.float32)).reshape(1, -1).to(eng.device)
        return self.apply_batch(x, sr, engine=eng)[0].cpu().numpy()


_side_streams = {}


def run_suite(suite, y, sr, consume, rng=None, engine=None):
    """Apply every attack of `suite` to the batch `y` and hand each result to `consume(index, attacked)`.

    Attacks whose kernel is a bit-exact sequential recurrence (`attack.sequential`: the direct-form IIRs in
    `fast=False` mode -- one 32-thread block per four clips, tens of milliseconds of dependent float64
    operations that occupy well under 1 % of the GPU) are launched first on a side stream and consumed last,
    so the rest of the suite and its detections run underneath them instead of after them."""
    eng = _eng(engine)
    main = torch.cuda.current_stream()
    slow = [i for i, a in enumerate(suite) if getattr(a, "sequential", False)]
    if getattr(eng, "profiling", False):                    # per-launch timeline: one stream, one ordered list
        slow = []
    pending = []
    if slow and len(slow) < len(suite):
        key = eng.device.index
        if key not in _side_streams:
            _side_streams[key] = torch.cuda.Stream(device=eng.device)
        side = _side_streams[key]
        side.wait_stream(main)                              # y is complete before the side stream reads it
        with torch.cuda.stream(side):
            for i in slow:
                pending.append((i, suite[i].apply_batch(y, sr, rng=rng, engine=eng)))
        y.record_stream(side)
    else:
        slow = []
    for i, att in enumerate(suite):
        if i not in slow:
            consume(i, att.apply_batch(y, sr, rng=rng, engine=eng))
    if pending:
        main.wait_stream(side)
        for i, z in pending:
            z.record_stream(main)
            consume(i, z)


class PCMBitDepthConversion(Attack):
    def __init__(self, pcm=16):
        self.pcm = pcm
        self.name = f"pcm_{pcm}"

    def apply_batch(self, x, sr, rng=None, engine=None):
        return _eng(engine).attack_pcm(x, self.pcm)


class DeleteSamples(Attack):
    def __init__(self, percentage, start=None):
        self.percentage, self.start = percentage, start
        self.name = f"delete_{percentage}"

    def apply_batch(self, x, sr, rng=None, engine=None):
        n = x.shape[1]
        n_del = int(self.percentage * n)
        start = self.start
        if start is None:
            rng = rng or np.random.default_rng()
            start = rng.integers(0, n - n_del, size=x.shape[0])
        start = torch.as_tensor(np.broadcast_to(np.asarray(start), (x.shape[0],)).copy(), dtype=torch.int32)
        return _eng(engine).attack_delete(x, start, n_del)


class Cropout(Attack):
    def __init__(self, percentage):
        self.percentage = percentage
        self.name = f"cropout_{percentage}"

    def apply_batch(self, x, sr, rng=None, engine=None):
        return _eng(engine).attack_cropout(x, int(self.percentage * sr))


class SampleSupression(Attack):
    def __init__(self, percentage, start=None):
        self.percentage, self.start = percentage, start
        self.name = f"sample_supression_{percentage}"

    def apply_batch(self, x, sr, rng=None, engine=None):
        n = x.shape[1]
        n_zero = int(self.percentage * sr)
        start = self.start
        if start is None:
            rng = rng or np.random.default_rng()
            start = rng.integers(0, n - n_zero, size=x.shape[0])
        start = torch.as_tensor(np.broadcast_to(np.asarray(start), (x.shape[0],)).copy(), dtype=torch.int32)
        return _eng(engine).attack_suppress(x, start, n_zero)


def polyphase_plan(n_in: int, up: int, down: int, window=("kaiser", 5.0), taps=None):
    """Host half of scipy.signal.resample_poly(x, up, down) for float32 input: the FIR
    (firwin, cast to float32, times `up`), its zero padding, the transposed+flipped tap
    table scipy's upfirdn uses, and the output window.  `taps` = an explicit FIR, as when
    resample_poly is given an array for `window` (pystoi's resample_oct).  Returns
    (h_tf float32[up*taps_per_phase], taps_per_phase, first_out, n_out)."""
    from scipy.signal import firwin
    g = math.gcd(up, down)
    up, down = up // g, down // g
    n_out = n_in * up
    n_out = n_out // down + bool(n_out % down)
    max_rate = max(up, down)
    if taps is not None:
        h = np.asarray(taps, dtype=np.float64).copy()
        half_len = (len(h) - 1) // 2
        h = (h * up).astype(np.float32)
    else:
        half_len = 10 * max_rate
        h = firwin(2 * half_len + 1, 1.0 / max_rate, window=window).astype(np.float32)
        h *= up
    n_pre_pad = down - half_len % down
    n_post_pad = 0
    n_pre_remove = (half_len + n_pre_pad) // down

    def out_len(len_h):
        return (((n_in - 1) * up + len_h) - 1) // down + 1

    while out_len(len(h) + n_pre_pad + n_post_pad) < n_out + n_pre_remove:
        n_post_pad += 1
    h = np.concatenate((np.zeros(n_pre_pad, dtype=h.dtype), h, np.zeros(n_post_pad, dtype=h.dtype)))
    pad = -len(h) % up
    h_full = np.concatenate((h, np.zeros(pad, dtype=h.dtype)))
    h_tf = np.ascontiguousarray(h_full.reshape(-1, up).T[:, ::-1]).ravel()
    return h_tf, len(h_full) // up, n_pre_remove, n_out


class Resample(Attack):
    def __init__(self, target_sr=16000):
        self.target_sr = target_sr
        self.name = f"resample_{target_sr}"
        self._plans = {}

    def _plan(self, eng, n, up, down):
        key = (n, up, down, eng.device.index)
        if key not in self._plans:
            h_tf, tpp, first, n_out = polyphase_plan(n, up, down)
            self._plans[key] = (torch.from_numpy(h_tf).to(eng.device), tpp, first, n_out)
        return self._plans[key]

    def apply_batch(self, x, sr, rng=None, engine=None):
        eng = _eng(engine)
        f = sr // self.target_sr
        if f > 1:                                     # decimate + np.interp back (attacks.py:276-287)
            return eng.attack_decimate_interp(x, f)
        up, down = 441, 160                           # polyphase there and back (attacks.py:289-294)
        h1, t1, k1, n1 = self._plan(eng, x.shape[1], up, down)
        mid = eng.attack_upfirdn(x, h1, t1, up, down, k1, n1)
        h2, t2, k2, n2 = self._plan(eng, n1, down, up)
        return eng.attack_upfirdn(mid, h2, t2, down, up, k2, n2)


class _Butter(Attack):
    """`fast=False` (default): sequential recurrence, one thread per clip -- bit-identical to
    scipy.signal.lfilter.  `fast=True`: chunk-parallel scan with look-back (agrees to ~1 ulp of
    float32 for these well-conditioned designs)."""
    fast = False

    @property
    def sequential(self):
        return not self.fast

    def _design(self, sr):
        raise NotImplementedError

    def apply_batch(self, x, sr, rng=None, engine=None):
        b, a = self._design(sr)
        return _eng(engine).attack_lfilter(x, b, a, _warm_samples(b, a) if self.fast else 0)


class LowPassFilter(_Butter):
    def __init__(self, cut_off=4000.0, order=6, fast=False):
        self.cut_off, self.order, self.name, self.fast = cut_off, order, "low_pass", fast

    def _design(self, sr):
        from scipy.signal import butter
        return butter(self.order, self.cut_off / (0.5 * sr), btype="low", analog=False)


class HighPassFilter(_Butter):
    def __init__(self, cut_off=500.0, order=4, fast=False):
        self.cut_off, self.order, self.name, self.fast = cut_off, order, "high_pass", fast

    def _design(self, sr):
        from scipy.signal import butter
        return butter(self.order, self.cut_off / (0.5 * sr), btype="highpass", analog=False)


class RandomBandstop(Attack):
    """One random 200 Hz stop band per call (as upstream: one draw per apply), zero-phase
    Butterworth via filtfilt.  The reference evaluates the 8th-order design in direct form,
    whose float64 round-off noise reaches 1e-6 (f_low ~ 1.2 kHz) to 6e-4 (f_low ~ 300 Hz) at
    44.1 kHz (vs the SOS form); only the sequential recurrence (`fast=False`, default)
    reproduces that noise bit for bit, the chunk-parallel scan agrees to that noise level."""

    def __init__(self, band_width=200.0, min_freq=300.0, max_freq=4000.0, order=4, f_low=None, fast=False):
        self.fast = fast
        self.band_width, self.min_freq, self.max_freq = float(band_width), float(min_freq), float(max_freq)
        self.order, self.f_low = int(order), f_low
        self.name = f"bandstop_{int(band_width)}Hz"

    @property
    def sequential(self):
        return not self.fast

    def apply_batch(self, x, sr, rng=None, engine=None):
        from scipy.signal import butter, lfilter_zi
        f_low = self.f_low
        if f_low is None:
            rng = rng or np.random.default_rng()
            f_low = float(rng.uniform(self.min_freq, self.max_freq - self.band_width))
        nyq = sr / 2.0
        b, a = butter(self.order, [f_low / nyq, (f_low + self.band_width) / nyq], btype="bandstop")
        return _eng(engine).attack_filtfilt(x, b, a, lfilter_zi(b, a), _warm_samples(b, a) if self.fast else 0)


# ---- extensions named by the build brief that have no reference arithmetic ("parity unpinned")
class AdditiveNoise(Attack):
    """y = x + sigma * buf, buf a host-seeded standard-normal buffer.  `buffer` (float32 [n, >= N], host or
    device) is the caller's own buffer -- a sweep draws it once and keeps it resident in HBM; without it the
    buffer is drawn per call from `seed` on the host and copied over."""

    def __init__(self, sigma=0.01, seed=99, buffer=None):
        self.sigma, self.seed, self.name = sigma, seed, f"noise_{sigma}"
        self.buffer = buffer

    def apply_batch(self, x, sr, rng=None, engine=None):
        if self.buffer is not None:
            buf = torch.as_tensor(self.buffer, dtype=torch.float32).to(x.device)
            if buf.dim() != 2 or buf.shape[0] != x.shape[0] or buf.shape[1] < x.shape[1] or buf.stride(1) != 1:
                raise ValueError("noise buffer must be float32 [n_clips, >= n_samples] with unit sample stride")
        else:
            g = torch.Generator(device="cpu").manual_seed(self.seed)
            buf = torch.randn(x.shape, generator=g, dtype=torch.float32).to(x.device)
        return _eng(engine).attack_affine(x, 1.0, buf, self.sigma)


class Gain(Attack):
    def __init__(self, gain=0.5):
        self.gain, self.name = gain, f"gain_{gain}"

    def apply_batch(self, x, sr, rng=None, engine=None):
        return _eng(engine).attack_affine(x, self.gain)


class FIRFilter(Attack):
    """Windowed-sinc FIR low / high / band-pass (the brief's "lowpass/highpass/bandpass FIR"; the
    reference itself only has Butterworth IIRs).  Defined as `scipy.signal.upfirdn(h, x)[:n]` with
    `h = firwin(numtaps, cutoff, pass_zero=..., fs=sr)` cast to float32 -- a causal FIR, the same
    single-pass polyphase kernel as `Resample` with up = down = 1, so it is bit-exact against
    scipy's float32 upfirdn (parity pinned to scipy, not to the reference)."""

    def __init__(self, kind="lowpass", cutoff=4000.0, numtaps=101):
        if kind not in ("lowpass", "highpass", "bandpass"):
            raise ValueError("kind must be lowpass, highpass or bandpass")
        self.kind, self.cutoff, self.numtaps = kind, cutoff, int(numtaps) | 1
        self.name = f"fir_{kind}"
        self._taps = {}

    def taps(self, sr):
        from scipy.signal import firwin
        pass_zero = {"lowpass": True, "highpass": False, "bandpass": False}[self.kind]
        return firwin(self.numtaps, self.cutoff, pass_zero=pass_zero, fs=sr).astype(np.float32)

    def apply_batch(self, x, sr, rng=None, engine=None):
        eng = _eng(engine)
        key = (sr, eng.device.index)
        if key not in self._taps:
            h = self.taps(sr)
            self._taps[key] = (torch.from_numpy(np.ascontiguousarray(h[::-1])).to(eng.device), len(h))
        h_tf, n_taps = self._taps[key]
        return eng.attack_upfirdn(x, h_tf, n_taps, 1, 1, 0, x.shape[1])


class CompressionApprox(Attack):
    """The brief's "compression approximation" -- PARITY UNPINNED: upstream's MP3Compression shells out to
    ffmpeg (attacks.py:73-148) and has no arithmetic to follow, so the attack is defined here.  It is what a
    transform codec does to the band that carries the watermark, in closed form: STFT (1024 / 256, Hann) of
    the input restricted to the embedding band; per frame, bins more than `floor_db` below the frame's
    strongest band bin are dropped (masking) and the others are rounded to a `step_db` grid in
    log-magnitude (coarse quantisation); phases are kept; the change is resynthesised (overlap-add) and
    added to the input, so content outside the band passes through.  Output length 256 * (N // 256).
    Pinned by its numpy restatement `oracle/aware_oracle.py::attack_compression_approx` in
    tests/test_gpu_parity.py."""

    def __init__(self, step_db=1.5, floor_db=-60.0):
        self.step_db, self.floor_db = float(step_db), float(floor_db)
        self.name = f"compress_{step_db}dB"

    def apply_batch(self, x, sr, rng=None, engine=None):
        eng = _eng(engine)
        L = 256 * (x.shape[1] // 256)
        mag, ph = eng.stft_band(x, sr, normalize=False, phasor=True)
        delta = eng.istft_band(eng.spectral_quantize(mag, self.step_db, self.floor_db), ph, sr)
        return eng.attack_affine(x[:, :L], 1.0, delta, 1.0)


# ---- desynchronisation attacks (upstream: rubberband, scripts/attacks.py:150-252; parity unpinned)
RATE_MIN, RATE_MAX = 0.25, 4.0


def check_rate(rate) -> float:
    """The phase vocoder's rate as a float; ValueError unless it is finite and in [0.25, 4]."""
    r = float(rate)
    if not (math.isfinite(r) and RATE_MIN <= r <= RATE_MAX):
        raise ValueError(f"time-stretch rate must be finite and in [{RATE_MIN:g}, {RATE_MAX:g}] (got {rate!r})")
    return r


def stretch_frames(n_frames: int, rate: float) -> int:
    """Output frames of the phase vocoder: len(np.arange(0, n_frames, rate)) = ceil(n_frames / rate)."""
    return math.ceil(n_frames / rate)


def stretch_length(n_samples: int, rate: float) -> int:
    """Output samples of a time stretch: round(N / rate) (librosa.effects.time_stretch)."""
    return int(round(n_samples / rate))


def pitch_ratio(n_steps, max_cents: float = 0.05) -> Fraction:
    """The resampling ratio of `PitchShift`: the fraction p / q with the smallest q (p = round(q r)) within
    `max_cents` of r = 2^(n_steps / 12).  At 0.05 cents, +-2 semitones give 55/49 and 49/55, and no q
    exceeds 433 for |n_steps| <= 12.  (Fraction(r).limit_denominator(256) misses 0.05 cents at +-5 and
    +-7 semitones, by up to 1.4 cents.)"""
    r = 2.0 ** (float(n_steps) / 12.0)
    if not (math.isfinite(r) and max_cents > 0):
        raise ValueError("pitch_ratio: n_steps must be finite and max_cents > 0")
    q = 1
    while True:
        p = max(1, round(r * q))
        if abs(1200.0 * math.log2(p / (q * r))) <= max_cents:
            return Fraction(p, q)
        q += 1


def _time_stretch(eng, x, rate):
    spec = eng.stft_full(x)
    return eng.istft_full(eng.phase_vocoder(spec, rate), stretch_length(x.shape[1], rate))


class TimeStretch(Attack):
    """Time stretch by `rate` without changing pitch -- PARITY UNPINNED: upstream calls rubberband, whose
    engine (transient detection, phase locking) has no arithmetic to follow, so the attack is defined here
    as the classical phase vocoder of librosa.effects.time_stretch in this project's STFT conventions:

      D     = torch.stft(x, 1024, 256, window=hann_window(1024), center=True)   (reflect pad, all 513
              bins, the float32 input as it is, no peak normalisation), T = 1 + N // 256 frames
      out   = librosa.phase_vocoder(D, rate, hop_length=256) with every operation in float64
              (DESIGN.md section 7 spells it out), rounded to complex64, ceil(T / rate) frames
      y     = torch.istft(out, 1024, 256, window, center=True, length=round(N / rate))

    rate > 1 gives shorter, faster audio (pyrubberband's convention); rate must lie in [0.25, 4].
    Stages: Engine.stft_full / phase_vocoder / istft_full.  Pinned by its numpy restatement
    (tests/desync_oracle.py) in tests/test_desync_attacks.py."""

    def __init__(self, rate):
        self.rate = check_rate(rate)
        self.name = f"time_stretch_{rate}"

    def apply_batch(self, x, sr, rng=None, engine=None):
        eng = _eng(engine)
        return _time_stretch(eng, eng._audio(x), self.rate)


class PitchShift(Attack):
    """Pitch shift by `n_steps` semitones at constant length -- PARITY UNPINNED (upstream: rubberband), defined
    as librosa.effects.pitch_shift's construction on the phase vocoder of `TimeStretch`:

      1. time-stretch by rate 2^(-n_steps / 12) (n_steps > 0: longer audio);
      2. resample by q / p, where p / q = pitch_ratio(n_steps, max_cents) approximates 2^(n_steps / 12):
         scipy.signal.resample_poly(y, q, p), the bit-exact polyphase kernel of `Resample` (skipped when p = q);
      3. truncate or zero-pad to the input length N.

    n_steps > 0 raises the pitch; |n_steps| <= 24 (the stretch rate stays in [0.25, 4])."""

    def __init__(self, n_steps, max_cents=0.05):
        self.n_steps = n_steps
        self.rate = check_rate(2.0 ** (-float(n_steps) / 12.0))
        self.ratio = pitch_ratio(n_steps, max_cents)
        self.name = f"pitch_shift_{n_steps}"
        self._plans = {}

    def apply_batch(self, x, sr, rng=None, engine=None):
        eng = _eng(engine)
        x = eng._audio(x)
        n = x.shape[1]
        y = _time_stretch(eng, x, self.rate)
        p, q = self.ratio.numerator, self.ratio.denominator
        if p != q:
            key = (y.shape[1], eng.device.index)
            if key not in self._plans:
                h_tf, tpp, first, n_res = polyphase_plan(y.shape[1], q, p)
                self._plans[key] = (torch.from_numpy(h_tf).to(eng.device), tpp, first, n_res)
            h, tpp, first, n_res = self._plans[key]
            y = eng.attack_upfirdn(y, h, tpp, q, p, first, n_res)
        if y.shape[1] >= n:
            return y[:, :n]
        return torch.nn.functional.pad(y, (0, n - y.shape[1]))


def desync_attacks():
    """The desynchronisation attacks `evaluate_clips(..., desync=True)` appends.  Upstream's time-stretch
    and pitch-shift parameters are not recorded in this repository; these values are this project's
    choice: +-10 % tempo and +-2 semitones."""
    return [TimeStretch(0.9), TimeStretch(1.1), PitchShift(-2), PitchShift(2)]


# ---- room attacks: reverberation and echo (no upstream counterpart; parity pinned to a float64 convolution)
CONV_PART = 512                   # partition length of the partitioned convolution
CONV_MAX_TAPS = 512 * CONV_PART   # 262 144 taps: 512 partitions
_DECAY_60DB = 6.907755278982137   # ln(1000): amplitude -60 dB


def conv_spectra(h) -> np.ndarray:
    """Partition spectra of impulse responses `h` ([M] or [R, M]) for `Engine.attack_convolve`: complex64
    [R, K, 513], K = ceil(M / 512), the rfft of each 512-tap partition zero-padded to 1024, computed in float64
    and rounded to complex64."""
    h = np.asarray(h, dtype=np.float64)
    if h.ndim == 1:
        h = h[None]
    if h.ndim != 2 or not 1 <= h.shape[1] <= CONV_MAX_TAPS or h.shape[0] < 1:
        raise ValueError(f"impulse responses must be [M] or [R, M] with 1 <= M <= {CONV_MAX_TAPS} (got {h.shape})")
    if not np.isfinite(h).all():
        raise ValueError("impulse responses must be finite")
    R, M = h.shape
    K = -(-M // CONV_PART)
    parts = np.zeros((R, K, CONV_PART), dtype=np.float64)
    parts.reshape(R, K * CONV_PART)[:, :M] = h
    return np.fft.rfft(parts, n=2 * CONV_PART, axis=2).astype(np.complex64)


def synthetic_rir(rt60: float, sr: int, seed: int) -> np.ndarray:
    """Exponentially decaying Gaussian noise of length round(rt60 sr) whose amplitude falls by 60 dB over
    rt60, with h[0] = 1 (direct path), scaled to unit energy; float64 throughout, returned as float32."""
    M = int(round(rt60 * sr))
    if not 1 <= M <= CONV_MAX_TAPS:
        raise ValueError(f"rt60 * sr = {rt60 * sr:g} taps is outside [1, {CONV_MAX_TAPS}]")
    h = np.random.default_rng(seed).standard_normal(M) * np.exp(-_DECAY_60DB * np.arange(M) / (rt60 * sr))
    h[0] = 1.0
    return (h / np.linalg.norm(h)).astype(np.float32)


class _Convolve(Attack):
    """Causal convolution of every clip with an impulse response, truncated to the input's length:
    y[n] = sum_{m < M} h[m] x[n - m], x[< 0] = 0 (scipy.signal.fftconvolve(x, h)[:N] in float64, float32 out).
    The GPU runs it as a uniformly partitioned overlap-save convolution (Engine.attack_convolve)."""

    def responses(self, sr: int) -> np.ndarray:
        """float32 [R, M] impulse responses at sample rate `sr`."""
        raise NotImplementedError

    def _index(self, n_clips, n_resp, rng):
        return None

    def apply_batch(self, x, sr, rng=None, engine=None):
        eng = _eng(engine)
        key = (int(sr), eng.device.index)
        if key not in self._spectra:
            h = self.responses(int(sr))
            self._spectra[key] = torch.from_numpy(conv_spectra(h)).to(eng.device)
        spec = self._spectra[key]
        return eng.attack_convolve(x, spec, self._index(x.shape[0], spec.shape[0], rng))


class Reverb(_Convolve):
    """Room reverberation -- an extension with no upstream counterpart (DESIGN.md section 7).  Each clip is
    convolved (see `_Convolve`) with one of `n_rirs` synthetic room impulse responses r = 0 .. n_rirs-1:
    M = round(rt60 sr) taps of np.random.default_rng(seed + r).standard_normal(M) times
    exp(-6.907755278982137 m / (rt60 sr)) (-60 dB at rt60), then h[0] = 1 (direct path) and h /= ||h||_2,
    all in float64, cast to float32.  `rir` ([M] or [R, M]) replaces them with the caller's own responses,
    e.g. a measured one read with `evaluate.read_wav`; rt60 is then not given.  With R > 1 responses every clip draws its own with
    rng.integers(0, R, n_clips); `index` (one int, or one per clip) fixes the choice instead.  Responses are
    built per sample rate and cached per (sr, device).  1 <= M <= 262 144."""

    def __init__(self, rt60=None, n_rirs=1, seed=0, rir=None, index=None):
        if rir is not None:
            if rt60 is not None:
                raise ValueError("give either rt60 (synthetic responses) or rir (the caller's own), not both")
            h = np.asarray(rir, dtype=np.float32)
            if h.ndim == 1:
                h = h[None]
            if h.ndim != 2 or h.shape[0] < 1 or not 1 <= h.shape[1] <= CONV_MAX_TAPS or not np.isfinite(h).all():
                raise ValueError(f"rir must be finite, [M] or [R, M] with 1 <= M <= {CONV_MAX_TAPS}")
            self.rir, self.n_rirs, self.rt60 = h, h.shape[0], None
            self.name = "reverb_rir"
        else:
            rt60 = float("nan") if rt60 is None else float(rt60)
            if not (math.isfinite(rt60) and rt60 > 0):
                raise ValueError(f"rt60 must be finite and > 0 (got {rt60!r})")
            if int(n_rirs) < 1:
                raise ValueError("n_rirs must be >= 1")
            self.rir, self.n_rirs, self.rt60 = None, int(n_rirs), rt60
            self.name = f"reverb_{rt60:g}"
        self.seed = int(seed)
        if index is not None:
            index = np.asarray(index)
            if (index.dtype.kind not in "iu" or index.ndim > 1 or not index.size
                    or index.min() < 0 or index.max() >= self.n_rirs):
                raise ValueError(f"index must be integers in [0, {self.n_rirs})")
        self.index = index
        self._spectra = {}

    def responses(self, sr: int) -> np.ndarray:
        if self.rir is not None:
            return self.rir
        if not 1 <= round(self.rt60 * sr) <= CONV_MAX_TAPS:
            raise ValueError(f"rt60 = {self.rt60:g} s at {sr} Hz gives {round(self.rt60 * sr)} taps, outside "
                             f"[1, {CONV_MAX_TAPS}]")
        return np.stack([synthetic_rir(self.rt60, sr, self.seed + r) for r in range(self.n_rirs)])

    def _index(self, n_clips, n_resp, rng):
        if self.index is not None:
            try:
                return np.broadcast_to(self.index, (n_clips,)).astype(np.int32)
            except ValueError:
                raise ValueError(f"index holds {self.index.size} entries for {n_clips} clips") from None
        if n_resp == 1:
            return None
        rng = rng or np.random.default_rng()
        return rng.integers(0, n_resp, n_clips).astype(np.int32)


class Echo(_Convolve):
    """A single echo -- an extension with no upstream counterpart (DESIGN.md section 7):
    y[n] = x[n] + decay x[n - D], D = round(delay sr) >= 1, as the convolution of `_Convolve` with
    h = [1, 0, ..., 0, decay] (D + 1 taps, not normalised)."""

    def __init__(self, delay=0.05, decay=0.5):
        self.delay, self.decay = float(delay), float(decay)
        if not (math.isfinite(self.delay) and self.delay > 0 and math.isfinite(self.decay)):
            raise ValueError(f"delay must be finite and > 0 and decay finite (got {delay!r}, {decay!r})")
        self.name = f"echo_{self.delay:g}_{self.decay:g}"
        self._spectra = {}

    def responses(self, sr: int) -> np.ndarray:
        """float32 [1, D + 1]: the one impulse response at sample rate `sr`."""
        D = int(round(self.delay * sr))
        if not 1 <= D < CONV_MAX_TAPS:
            raise ValueError(f"delay = {self.delay:g} s at {sr} Hz gives D = {D}, outside [1, {CONV_MAX_TAPS - 1}]")
        h = np.zeros((1, D + 1), dtype=np.float32)
        h[0, 0], h[0, D] = 1.0, self.decay
        return h


def room_attacks():
    """The room attacks `evaluate_clips(..., room=True)` appends.  There is no upstream counterpart, so these
    parameters are this project's choice: a small and a large room (RT60 0.3 s and 0.7 s, eight synthetic
    responses each, one drawn per clip) and a 50 ms echo at half amplitude."""
    return [Reverb(0.3, n_rirs=8, seed=0), Reverb(0.7, n_rirs=8, seed=100), Echo(0.05, 0.5)]


def reference_suite():
    """The in-scope part of scripts/test.py's attack_list (test.py:15-18)."""
    return [PCMBitDepthConversion(8), PCMBitDepthConversion(12), PCMBitDepthConversion(16),
            PCMBitDepthConversion(24), DeleteSamples(0.1), DeleteSamples(0.15), DeleteSamples(0.2),
            Resample(), RandomBandstop(), SampleSupression(0.1), SampleSupression(0.25),
            LowPassFilter(), HighPassFilter()]

"""Batched device engine: torch tensors for memory / streams, the C ABI for compute.

One Engine per process and device.  Every method takes and returns CUDA tensors
(audio: float32 [n_clips, n_samples]); the reference-shaped numpy API in
aware_b200.service / .embedding / .detection is a thin layer over it.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from . import _lib

N_BITS = 20
HOP = 256
N_BINS_FULL = 513


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class Engine:
    def __init__(self, weights, mel_basis, window, bands=(500.0, 4000.0), tolerance_db=6.0,
                 threshold=0.0, precision="tf32", device=None):
        if not torch.cuda.is_available():
            raise RuntimeError("aware_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = _lib.lib()
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        ws = [np.ascontiguousarray(w, dtype=np.float32) for w in weights]
        mel = np.ascontiguousarray(mel_basis, dtype=np.float32)
        win = np.ascontiguousarray(window, dtype=np.float32)
        assert [w.shape for w in ws] == [(512, 128), (1024, 512), (1024, 1024), (40, 1024)]
        assert mel.shape == (128, 513) and win.shape == (1024,)
        m = _lib.AwModel()
        for i, w in enumerate(ws):
            m.w[i] = w.ctypes.data_as(C.POINTER(C.c_float))
        m.mel_basis = mel.ctypes.data_as(C.POINTER(C.c_float))
        m.window = win.ctypes.data_as(C.POINTER(C.c_float))
        m.band_lo_hz, m.band_hi_hz = float(bands[0]), float(bands[1])
        m.tolerance_db, m.threshold = float(tolerance_db), float(threshold)
        self._ctx = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.aw_ctx_create(C.byref(self._ctx), self.device.index, C.byref(m)))
        self.threshold = float(threshold)
        self.exact_margin = 1e-3
        self.embed_precision = None      # None: same as `precision`; "bf16" speeds up the embed loop
        self.set_precision(precision)

    def __del__(self):
        try:
            if getattr(self, "_ctx", None):
                self.lib.aw_ctx_destroy(self._ctx)
                self._ctx = None
        except Exception:
            pass

    # ------------------------------------------------------------------ misc
    _PREC = {"tf32": _lib.PREC_TF32, "fp32": _lib.PREC_FP32, "bf16": _lib.PREC_BF16, "fp16": _lib.PREC_FP16}

    def set_precision(self, precision: str):
        """GEMM arithmetic of the detector stack: "tf32" (tcgen05, TF32 operands), "fp32" (CUDA
        cores, validation) or "bf16" (tcgen05, bf16 operands and bf16 activation storage)."""
        _lib.check(self.lib.aw_ctx_set_precision(self._ctx, self._PREC[precision]))
        self.precision = precision

    def _with_precision(self, precision):
        class _Ctx:
            def __enter__(c):
                c.prev = self.precision
                if precision and precision != c.prev:
                    self.set_precision(precision)

            def __exit__(c, *a):
                if self.precision != c.prev:
                    self.set_precision(c.prev)
        return _Ctx()

    def launch_count(self) -> int:
        return int(self.lib.aw_launch_count(self._ctx))

    def set_threshold(self, threshold: float):
        """Decision threshold used by `decide` and by detect's low-margin test (detector.threshold)."""
        if float(threshold) != self.threshold:
            _lib.check(self.lib.aw_ctx_set_option(self._ctx, _lib.OPT_THRESHOLD, float(threshold)))
            self.threshold = float(threshold)

    def set_exact_margin(self, margin: float):
        """Clips whose min |v - threshold| is below `margin` are re-evaluated by `detect` through the
        exact fp32 GEMMs (bit decisions equal to the reference's arithmetic).  0 disables it."""
        _lib.check(self.lib.aw_ctx_set_option(self._ctx, _lib.OPT_EXACT_MARGIN, float(margin)))
        self.exact_margin = float(margin)

    def set_tc_spectral(self, on: bool, min_frames: int | None = None):
        """fp16 embed loop at 44.1 / 48 kHz: band-limited STFT / iSTFT as tcgen05 GEMMs (default for batches
        of at least `min_frames` = n_clips * frames, 24 576 unless given) or the fp32 FFT kernels."""
        v = 0.0 if not on else (float(min_frames) if min_frames and min_frames > 1 else 1.0)
        _lib.check(self.lib.aw_ctx_set_option(self._ctx, _lib.OPT_TC_SPECTRAL, v))

    def set_two_pass(self, on: bool):
        _lib.check(self.lib.aw_ctx_set_option(self._ctx, _lib.OPT_TWO_PASS, 1.0 if on else 0.0))

    def set_pair_gemm(self, on: bool):
        """K >= 512 layers on CTA pairs (cta_group::2); off = the one-CTA kernel (bit-identical results)."""
        _lib.check(self.lib.aw_ctx_set_option(self._ctx, _lib.OPT_PAIR_GEMM, 1.0 if on else 0.0))

    def set_bwd64_stream(self, on: bool):
        """16-bit loops: backward K = 64 layer on the TMA-streaming kernel (gemm64.cuh); off = generic GEMM epilogues."""
        _lib.check(self.lib.aw_ctx_set_option(self._ctx, _lib.OPT_BWD64_STREAM, 1.0 if on else 0.0))

    def detect_stats(self):
        """(clips seen by detect, clips re-evaluated exactly) since the engine was created."""
        out = []
        for which in (_lib.STAT_DETECT_CLIPS, _lib.STAT_REEVAL_CLIPS):
            v = C.c_int64()
            _lib.check(self.lib.aw_ctx_get_stat(self._ctx, which, C.byref(v)))
            out.append(int(v.value))
        return tuple(out)

    def profile(self, on: bool):
        _lib.check(self.lib.aw_profile_enable(self._ctx, int(on)))
        self.profiling = bool(on)      # the per-launch timeline is one ordered list: attacks.run_suite stays on one stream

    def profile_read(self):
        """[(n, k, epilogue, launches, total_ms)] of the tensor-core GEMMs since the last read."""
        mx = 32
        nc = C.c_int()
        n, k, e = (C.c_int * mx)(), (C.c_int * mx)(), (C.c_int * mx)()
        cnt, ms = (C.c_int64 * mx)(), (C.c_double * mx)()
        _lib.check(self.lib.aw_profile_read(self._ctx, mx, C.byref(nc), n, k, e, cnt, ms))
        return [(n[i], k[i], e[i], int(cnt[i]), float(ms[i])) for i in range(nc.value)]

    def profile_read_named(self):
        """{kernel class: (launches, total_ms)} of EVERY kernel launched since the last read."""
        mx = 64
        nc = C.c_int()
        names = C.create_string_buffer(32 * mx)
        cnt, ms = (C.c_int64 * mx)(), (C.c_double * mx)()
        _lib.check(self.lib.aw_profile_read_named(self._ctx, mx, C.byref(nc), names, cnt, ms))
        raw = names.raw
        return {raw[32 * i:32 * i + 32].split(b"\0", 1)[0].decode(): (int(cnt[i]), float(ms[i]))
                for i in range(nc.value)}

    def band_bins(self, sample_rate: int):
        b0, nb = C.c_int(), C.c_int()
        _lib.check(self.lib.aw_band_bins(self._ctx, int(sample_rate), C.byref(b0), C.byref(nb)))
        return b0.value, nb.value

    def _audio(self, x):
        if not (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float32 and x.dim() == 2
                and x.stride(1) == 1):
            raise ValueError("expected a CUDA float32 tensor [n_clips, n_samples] with unit inner stride")
        return x

    # ------------------------------------------------------------- hot path
    def detect(self, audio: torch.Tensor, sample_rate: int) -> torch.Tensor:
        """[n, N] -> [n, 20] tanh outputs (AWAREDetector.detect for a batch)."""
        x = self._audio(audio)
        n, N = x.shape
        out = torch.empty((n, N_BITS), dtype=torch.float32, device=x.device)
        _lib.check(self.lib.aw_detect_batch(self._ctx, _ptr(x), n, N, x.stride(0), int(sample_rate),
                                            _ptr(out), _stream()))
        return out

    def embed(self, audio: torch.Tensor, sample_rate: int, pattern: torch.Tensor, iters: int = 400,
              scale: torch.Tensor | str | None = None, wave_clips: int = 0, return_losses: bool = False,
              precision: str | None = None):
        """[n, N] + [n, 20] int32 (+-1) -> [n, 256*(N//256)] watermarked, peak-normalised
        (AWAREEmbedder.embed for a batch); optionally multiplied per clip by `scale` (a tensor, or
        "signed_max": each clip's signed max computed on the device, service/embed.py:69,73)."""
        x = self._audio(audio)
        n, N = x.shape
        L = HOP * (N // HOP)
        pat = pattern.to(device=x.device, dtype=torch.int32).contiguous()
        if pat.shape != (n, N_BITS):
            raise ValueError("Invalid watermark length.")
        out = torch.empty((n, L), dtype=torch.float32, device=x.device)
        best = torch.empty((n,), dtype=torch.float32, device=x.device)
        losses = torch.zeros((max(iters, 1), n), dtype=torch.float32, device=x.device) if return_losses else None
        mode = _lib.SCALE_NONE
        if isinstance(scale, str):
            if scale != "signed_max":
                raise ValueError("scale must be a tensor, None or 'signed_max'")
            mode, sc = _lib.SCALE_SIGNED_MAX, None
        else:
            sc = scale.to(device=x.device, dtype=torch.float32).contiguous() if scale is not None else None
        with self._with_precision(precision or self.embed_precision):
            _lib.check(self.lib.aw_embed_batch(self._ctx, _ptr(x), n, N, x.stride(0), int(sample_rate),
                                               _ptr(pat), int(iters), _ptr(sc), mode, _ptr(out), out.stride(0),
                                               _ptr(best), _ptr(losses), int(wave_clips), _stream()))
        self._last_embed_n = n
        if return_losses:
            return out, best, losses
        return out

    def embed_status(self) -> torch.Tensor:
        """int32 [n] flags of the last `embed`: 1 = the clip met a non-finite gradient in the loop
        (its update was skipped; only possible with 16-bit loop GEMMs)."""
        n = getattr(self, "_last_embed_n", 0)
        flags = torch.empty((n,), dtype=torch.int32, device=self.device)
        _lib.check(self.lib.aw_embed_status(self._ctx, _ptr(flags), n, _stream()))
        return flags

    def embed_state(self, which: str, n: int, n_frames: int, sample_rate: int) -> torch.Tensor:
        """Optimisation state of the last embed wave, [n, T, nbins] (parity hooks)."""
        sel = {"c": 0, "best": 1, "c0": 2, "m": 3, "v": 4}[which]
        _, nb = self.band_bins(sample_rate)
        dst = torch.empty((n, n_frames, nb), dtype=torch.float32, device=self.device)
        _lib.check(self.lib.aw_embed_state(self._ctx, sel, _ptr(dst), dst.numel(), _stream()))
        return dst

    def debug_buffer(self, which: int, words: int) -> torch.Tensor:
        """Raw float32 view of an intermediate of the last embed iteration (development aid):
        10 y, 11 dpad, 12 packed peak, 13 dA, 14 |S~|, 15 y_oob."""
        dst = torch.empty((words,), dtype=torch.float32, device=self.device)
        _lib.check(self.lib.aw_embed_state(self._ctx, int(which), _ptr(dst), dst.numel(), _stream()))
        return dst

    def decide(self, values: torch.Tensor, ref_bits: torch.Tensor | None = None,
               counters: torch.Tensor | None = None, threshold: float | None = None):
        """values [n,20] -> bits int32 [n,20] (strict '>' threshold); with ref_bits also
        per-clip error counts, and `counters` (int64[3]: errors, bits, clips) is incremented.
        `threshold` (the detector's) overrides the engine's current one."""
        if threshold is not None:
            self.set_threshold(threshold)
        n = values.shape[0]
        bits = torch.empty((n, N_BITS), dtype=torch.int32, device=values.device)
        errs = torch.zeros((n,), dtype=torch.int32, device=values.device) if ref_bits is not None else None
        ref = ref_bits.to(device=values.device, dtype=torch.int32).contiguous() if ref_bits is not None else None
        _lib.check(self.lib.aw_decide_and_count(self._ctx, _ptr(values.contiguous()), _ptr(ref), n,
                                                _ptr(bits), _ptr(errs), _ptr(counters), _stream()))
        return (bits, errs) if ref_bits is not None else bits

    def snr(self, out: torch.Tensor, target: torch.Tensor, snr_sum: torch.Tensor | None = None):
        n = out.shape[0]
        m = min(out.shape[1], target.shape[1])
        res = torch.empty((n,), dtype=torch.float64, device=out.device)
        _lib.check(self.lib.aw_snr_batch(self._ctx, _ptr(out), out.stride(0), _ptr(target), target.stride(0),
                                         n, m, _ptr(res), _ptr(snr_sum), _stream()))
        return res

    def stoi(self, clean: torch.Tensor, processed: torch.Tensor, sample_rate: int,
             stoi_sum: torch.Tensor | None = None, keep_above: float = 0.1):
        """STOI per clip (float64 [n]) of processed against clean, both [n, N] float32 on the device at
        `sample_rate` (metrics/audio.py:43-64 -> pystoi.stoi(clean, processed, sr)): resample to pystoi's
        10 kHz with its Octave-style window through the polyphase kernel, then aw_stoi_batch.
        stoi_sum: float64[2] += {sum of scores > keep_above, count} (scripts/test.py:86-88)."""
        from . import metrics
        x, y = self._audio(clean), self._audio(processed)
        m = min(x.shape[1], y.shape[1])
        x, y = x[:, :m], y[:, :m]
        if int(sample_rate) != metrics.audio.STOI_FS:
            x, y = (metrics.audio.resample_oct_batch(t, metrics.audio.STOI_FS, int(sample_rate), self) for t in (x, y))
        n = x.shape[0]
        res = torch.empty((n,), dtype=torch.float64, device=x.device)
        _lib.check(self.lib.aw_stoi_batch(self._ctx, _ptr(x), x.stride(0), _ptr(y), y.stride(0), n, x.shape[1],
                                          _ptr(res), _ptr(stoi_sum), float(keep_above), _stream()))
        return res

    # ---------------------------------------------------------- stage hooks
    def stft_band(self, audio, sample_rate, normalize=True, phasor=False):
        x = self._audio(audio)
        n, N = x.shape
        T = 1 + N // HOP
        _, nb = self.band_bins(sample_rate)
        mag = torch.empty((n, T, nb), dtype=torch.float32, device=x.device)
        ph = torch.empty((n, T, nb, 2), dtype=torch.float32, device=x.device) if phasor else None
        _lib.check(self.lib.aw_stft_band(self._ctx, _ptr(x), n, N, x.stride(0), int(sample_rate),
                                         int(bool(normalize)), _ptr(mag), _ptr(ph), _stream()))
        return (mag, ph) if phasor else mag

    def istft_band(self, mag, phasor, sample_rate):
        n, T, nb = mag.shape
        wave = torch.empty((n, HOP * (T - 1)), dtype=torch.float32, device=mag.device)
        _lib.check(self.lib.aw_istft_band(self._ctx, _ptr(mag.contiguous()), _ptr(phasor.contiguous()), n, T,
                                          int(sample_rate), _ptr(wave), _stream()))
        return wave

    @staticmethod
    def _spectrum(spec):
        if not (isinstance(spec, torch.Tensor) and spec.is_cuda and spec.dtype == torch.complex64 and spec.dim() == 3
                and spec.shape[2] == N_BINS_FULL):
            raise ValueError("expected a CUDA complex64 spectrum [n_clips, n_frames, 513]")
        return torch.view_as_real(spec.contiguous())

    def stft_full(self, audio):
        """[n, N] -> complex64 [n, T, 513], T = 1 + N // 256: torch.stft(x, 1024, 256, hann_window(1024),
        center=True) of every clip, all bins, the input as it is (no peak normalisation).  Frame-major: clip
        i's torch.stft result is out[i].T."""
        x = self._audio(audio)
        n, N = x.shape
        spec = torch.empty((n, 1 + N // HOP, N_BINS_FULL, 2), dtype=torch.float32, device=x.device)
        _lib.check(self.lib.aw_stft_full(self._ctx, _ptr(x), n, N, x.stride(0), _ptr(spec), _stream()))
        return torch.view_as_complex(spec)

    def phase_vocoder(self, spec, rate):
        """complex64 [n, T, 513] -> [n, ceil(T / rate), 513]: librosa.phase_vocoder(D, rate, hop_length=256)
        in float64 (aw_phase_vocoder); rate finite and in [0.25, 4]."""
        s = self._spectrum(spec)
        n, T = s.shape[:2]
        rate = float(rate)
        T_out = math.ceil(T / rate) if math.isfinite(rate) and rate > 0 else 0
        out = torch.empty((n, max(T_out, 1), N_BINS_FULL, 2), dtype=torch.float32, device=s.device)
        _lib.check(self.lib.aw_phase_vocoder(self._ctx, _ptr(s), n, T, rate, T_out, _ptr(out), _stream()))
        return torch.view_as_complex(out)

    def istft_full(self, spec, n_out):
        """complex64 [n, T, 513] -> float32 [n, n_out]: torch.istft(D, 1024, 256, hann_window(1024),
        center=True, length=n_out) of every clip (imaginary parts of bins 0 and 512 ignored)."""
        s = self._spectrum(spec)
        n, T = s.shape[:2]
        if int(n_out) < 1:
            raise ValueError("n_out must be >= 1")
        wave = torch.empty((n, int(n_out)), dtype=torch.float32, device=s.device)
        _lib.check(self.lib.aw_istft_full(self._ctx, _ptr(s), n, T, int(n_out), _ptr(wave), wave.stride(0),
                                          _stream()))
        return wave

    def gemm(self, a, b, precision=None):
        rows, k = a.shape
        n = b.shape[0]
        out = torch.empty((rows, n), dtype=torch.float32, device=a.device)
        prec = self._PREC[precision or self.precision]
        _lib.check(self.lib.aw_gemm(self._ctx, _ptr(a.contiguous()), _ptr(b.contiguous()), _ptr(out),
                                    rows, n, k, prec, _stream()))
        return out

    # -------------------------------------------------------------- attacks
    def _out_like(self, x, n_out=None):
        return torch.empty((x.shape[0], x.shape[1] if n_out is None else n_out), dtype=torch.float32,
                           device=x.device)

    def attack_pcm(self, x, bits):
        x = self._audio(x); out = self._out_like(x)
        _lib.check(self.lib.aw_attack_pcm(self._ctx, _ptr(x), x.shape[0], x.shape[1], x.stride(0), int(bits),
                                          _ptr(out), out.stride(0), _stream()))
        return out

    def attack_decimate_interp(self, x, factor):
        x = self._audio(x); out = self._out_like(x)
        _lib.check(self.lib.aw_attack_decimate_interp(self._ctx, _ptr(x), x.shape[0], x.shape[1], x.stride(0),
                                                      int(factor), _ptr(out), out.stride(0), _stream()))
        return out

    def attack_upfirdn(self, x, h_tf, taps_per_phase, up, down, first_out, n_out):
        x = self._audio(x); out = self._out_like(x, n_out)
        _lib.check(self.lib.aw_attack_upfirdn(self._ctx, _ptr(x), x.shape[0], x.shape[1], x.stride(0),
                                              _ptr(h_tf), int(taps_per_phase), int(up), int(down),
                                              int(first_out), int(n_out), _ptr(out), out.stride(0), _stream()))
        return out

    @staticmethod
    def _dbl(v):
        a = np.ascontiguousarray(v, dtype=np.float64)
        return a, a.ctypes.data_as(C.POINTER(C.c_double))

    def attack_lfilter(self, x, b, a, warm):
        x = self._audio(x); out = self._out_like(x)
        bb, bp = self._dbl(b); aa, ap = self._dbl(a)
        _lib.check(self.lib.aw_attack_lfilter(self._ctx, _ptr(x), x.shape[0], x.shape[1], x.stride(0), bp, ap,
                                              len(bb) - 1, int(warm), _ptr(out), out.stride(0), _stream()))
        return out

    def attack_filtfilt(self, x, b, a, zi, warm):
        x = self._audio(x); out = self._out_like(x)
        bb, bp = self._dbl(b); aa, ap = self._dbl(a); zz, zp = self._dbl(zi)
        _lib.check(self.lib.aw_attack_filtfilt(self._ctx, _ptr(x), x.shape[0], x.shape[1], x.stride(0), bp, ap,
                                               zp, len(bb) - 1, int(warm), _ptr(out), out.stride(0), _stream()))
        return out

    def attack_delete(self, x, start, n_delete):
        x = self._audio(x); out = self._out_like(x, x.shape[1] - n_delete)
        st = start.to(device=x.device, dtype=torch.int32).contiguous()
        _lib.check(self.lib.aw_attack_delete(self._ctx, _ptr(x), x.shape[0], x.shape[1], x.stride(0), _ptr(st),
                                             int(n_delete), _ptr(out), out.stride(0), _stream()))
        return out

    def attack_suppress(self, x, start, n_zero):
        x = self._audio(x); out = self._out_like(x)
        st = start.to(device=x.device, dtype=torch.int32).contiguous()
        _lib.check(self.lib.aw_attack_suppress(self._ctx, _ptr(x), x.shape[0], x.shape[1], x.stride(0), _ptr(st),
                                               int(n_zero), _ptr(out), out.stride(0), _stream()))
        return out

    def attack_cropout(self, x, n_drop):
        x = self._audio(x); out = self._out_like(x, x.shape[1] - n_drop)
        _lib.check(self.lib.aw_attack_cropout(self._ctx, _ptr(x), x.shape[0], x.shape[1], x.stride(0),
                                              int(n_drop), _ptr(out), out.stride(0), _stream()))
        return out

    def attack_affine(self, x, gain=1.0, noise=None, sigma=0.0):
        x = self._audio(x); out = self._out_like(x)
        ns = noise.stride(0) if noise is not None else 0
        _lib.check(self.lib.aw_attack_affine(self._ctx, _ptr(x), x.shape[0], x.shape[1], x.stride(0), float(gain),
                                             _ptr(noise), ns, float(sigma), _ptr(out), out.stride(0), _stream()))
        return out

    def attack_convolve(self, x, spec, filter_of_clip=None):
        """[n, N] -> [n, N]: every clip convolved with its filter, causal and truncated to N samples
        (scipy.signal.fftconvolve(x, h)[:N]; aw_attack_convolve).  `spec`: complex64 [R, K, 513] on x's device, the
        partition spectra of `attacks.conv_spectra`; `filter_of_clip`: int [n] in [0, R), or None (filter 0)."""
        x = self._audio(x)
        if not (isinstance(spec, torch.Tensor) and spec.device == x.device and spec.dtype == torch.complex64
                and spec.dim() == 3 and spec.shape[2] == N_BINS_FULL):
            raise ValueError("expected complex64 partition spectra [n_filters, n_parts, 513] on the device of x")
        s = torch.view_as_real(spec.contiguous())
        idx = None
        if filter_of_clip is not None:
            idx = np.ascontiguousarray(filter_of_clip, dtype=np.int32)
            if idx.shape != (x.shape[0],):
                raise ValueError("filter_of_clip must hold one index per clip")
        out = self._out_like(x)
        _lib.check(self.lib.aw_attack_convolve(self._ctx, _ptr(x), x.shape[0], x.shape[1], x.stride(0), _ptr(s),
                                               s.shape[0], s.shape[1],
                                               idx.ctypes.data_as(C.c_void_p) if idx is not None else None,
                                               _ptr(out), out.stride(0), _stream()))
        return out

    def spectral_quantize(self, mag, step_db, floor_db):
        """[n, T, nb] band magnitudes -> (quantised - original) magnitudes (CompressionApprox attack)."""
        n, T, nb = mag.shape
        out = torch.empty_like(mag)
        _lib.check(self.lib.aw_attack_spectral_quantize(self._ctx, _ptr(mag.contiguous()), n, T, nb, float(step_db),
                                                        float(floor_db), _ptr(out), _stream()))
        return out

"""Time-stretch and pitch-shift attacks (aware_b200.attacks.TimeStretch / PitchShift).

Parity is UNPINNED to upstream (rubberband); the attacks are defined by the phase-vocoder restatement
in tests/desync_oracle.py (DESIGN.md section 7).  The CPU tests pin properties of that restatement and
of the host-side helpers; the GPU tests pin each CUDA stage and the composed attacks to it."""
import math

import numpy as np
import pytest
import torch

import aware_oracle as O
import desync_oracle as D
from aware_b200 import attacks as A

RATES = [0.5, 0.8, 0.9, 1.0, 1.1, 1.25, 2.0]
SIZES = [(16000, 1.3), (44100, 1.0)]          # 20 800 and 44 100 samples: neither a multiple of 256


def _tone(f, n, sr):
    return (0.5 * np.sin(2 * np.pi * f * np.arange(n) / sr)).astype(np.float32)


def _dominant_bin(x):
    mag = D.stft(x).abs().numpy()
    return int(np.argmax(mag[:, 4:-4].mean(axis=1)))   # frames clear of the reflect-padded edges


def _snr(a, b):
    return 10 * np.log10(np.sum(b.astype(np.float64) ** 2) / max(np.sum((a.astype(np.float64) - b) ** 2), 1e-300))


# ---------------------------------------------------------------- CPU: the restatement and host helpers
def test_time_stretch_at_rate_one_is_stft_then_istft():
    x = O.synth_clip(0, 1.3, 16000)
    y = D.attack_time_stretch(x, 1.0)
    ref = D.istft(D.stft(x), len(x))
    assert y.shape == ref.shape == x.shape
    assert np.abs(y - ref).max() <= 1e-6 * np.abs(ref).max()


@pytest.mark.parametrize("rate", [0.8, 1.25])
def test_time_stretch_keeps_the_pitch_of_a_tone(rate):
    sr, n = 16000, 16000 + 77
    x = _tone(1000.0, n, sr)
    y = D.attack_time_stretch(x, rate)
    assert len(y) == round(n / rate) == A.stretch_length(n, rate)
    assert _dominant_bin(y) == _dominant_bin(x)


@pytest.mark.parametrize("n_steps", [-12, 12])
def test_pitch_shift_by_an_octave_moves_a_tone_by_an_octave(n_steps):
    sr, n = 16000, 16000 + 77
    x = _tone(1000.0, n, sr)
    y = D.attack_pitch_shift(x, n_steps)
    assert y.shape == x.shape
    want = 2.0 ** (n_steps / 12) * _dominant_bin(x)
    assert abs(_dominant_bin(y) - want) <= 1


def test_pitch_shift_by_zero_is_the_rate_one_stretch():
    x = O.synth_clip(1, 1.0, 16000)
    np.testing.assert_array_equal(D.attack_pitch_shift(x, 0), D.attack_time_stretch(x, 1.0))


def test_output_frame_count_equals_np_arange_length():
    rates = [0.25, 0.3, 0.5, 0.7, 0.8, 0.9, 1.0, 1.1, 1.25, 1.5, 2.0, 3.3, 4.0]
    for T in (2, 5, 63, 82, 173, 1723, 4000):
        near = []
        for m in range(max(1, T // 4), 4 * T + 1, max(1, T // 40)):
            r = T / m                                       # T / r within rounding of the integer m
            for q in (r, np.nextafter(r, 0.0), np.nextafter(r, 1e9), r * (1 + 1e-12), r * (1 - 1e-12)):
                if 0.25 <= q <= 4.0:
                    near.append(float(q))
        for r in rates + near:
            assert A.stretch_frames(T, r) == len(np.arange(0, T, r)), (T, r)
    assert D.phase_vocoder(np.ones((513, 10), np.complex64), 0.3).shape == (513, A.stretch_frames(10, 0.3))


def test_pitch_ratio_table_is_within_five_hundredths_of_a_cent():
    for n in range(-12, 13):
        f = A.pitch_ratio(n)
        assert f == D.pitch_ratio(n)
        assert abs(1200 * math.log2(f.numerator / f.denominator / 2 ** (n / 12))) <= 0.05, (n, f)
    assert (A.pitch_ratio(2).numerator, A.pitch_ratio(2).denominator) == (55, 49)
    assert (A.pitch_ratio(-2).numerator, A.pitch_ratio(-2).denominator) == (49, 55)
    assert A.pitch_ratio(0) == 1 and A.pitch_ratio(12) == 2


@pytest.mark.parametrize("bad", [0.0, 0.2, 4.5, -1.0, float("nan"), float("inf")])
def test_out_of_range_rates_raise_before_any_library_call(bad):
    with pytest.raises(ValueError):
        A.TimeStretch(bad)


def test_pitch_shift_beyond_two_octaves_raises():
    for n in (25, -25, float("nan")):
        with pytest.raises(ValueError):
            A.PitchShift(n)
    assert [a.name for a in A.desync_attacks()] == ["time_stretch_0.9", "time_stretch_1.1", "pitch_shift_-2",
                                                    "pitch_shift_2"]


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def model():
    from aware_b200.utils.models import load
    emb, det = load()
    emb.verbose = False
    A.set_engine(emb.engine)
    return emb, det


@pytest.mark.gpu
@pytest.mark.parametrize("sr,secs", SIZES)
def test_stft_full_matches_torch_stft(model, sr, secs):
    eng = model[0].engine
    x = np.stack([O.synth_clip(i, secs, sr) * s for i, s in ((0, 1.0), (1, 3.0), (2, 0.01))])
    got = eng.stft_full(torch.from_numpy(x).cuda()).cpu().numpy()
    assert got.shape == (3, 1 + x.shape[1] // 256, 513) and got.dtype == np.complex64
    for i in range(3):
        want = D.stft(x[i]).numpy().T
        assert np.abs(got[i] - want).max() <= 1e-5 * np.abs(want).max()


@pytest.mark.gpu
@pytest.mark.parametrize("sr,secs", SIZES)
def test_istft_full_matches_torch_istft_with_length(model, sr, secs):
    eng = model[0].engine
    T = 1 + int(round(secs * sr)) // 256
    L = 256 * (T - 1)
    g = np.random.default_rng(5)
    spec = (g.standard_normal((2, T, 513)) + 1j * g.standard_normal((2, T, 513))).astype(np.complex64)
    assert (spec[:, :, 0].imag != 0).all() and (spec[:, :, 512].imag != 0).all()
    sd = torch.from_numpy(spec).cuda()
    for n_out in (L - 100, L, L + 13, L + 300, L + 600):
        got = eng.istft_full(sd, n_out).cpu().numpy()
        assert got.shape == (2, n_out)
        for i in range(2):
            want = D.istft(spec[i].T, n_out)
            assert np.abs(got[i] - want).max() <= 1e-4 * np.abs(want).max(), n_out
            m = min(n_out, L)
            assert np.abs(got[i, :m] - want[:m]).max() <= 1e-4 * np.abs(want[:m]).max(), n_out
            assert (got[i, L + 512:] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("sr,secs", SIZES)
def test_phase_vocoder_matches_the_float64_restatement(model, sr, secs):
    eng = model[0].engine
    x = np.stack([O.synth_clip(i, secs, sr) for i in (3, 4)])
    spec = eng.stft_full(torch.from_numpy(x).cuda())
    s_np = spec.cpu().numpy()
    for rate in RATES:
        got = eng.phase_vocoder(spec, rate).cpu().numpy()
        assert got.shape == (2, A.stretch_frames(s_np.shape[1], rate), 513)
        for i in range(2):
            want = D.phase_vocoder(s_np[i].T, rate).T
            assert np.abs(got[i] - want).max() <= 1e-6 * np.abs(s_np[i]).max(), rate


@pytest.mark.gpu
def test_stage_arguments_are_validated(model):
    from aware_b200 import _lib
    eng = model[0].engine
    spec = eng.stft_full(torch.zeros((1, 4000), device="cuda"))
    for bad in (0.2, 4.5, float("nan")):
        with pytest.raises(ValueError):
            eng.phase_vocoder(spec, bad)
    out = torch.empty((1, 40, 513, 2), device="cuda")
    rc = eng.lib.aw_phase_vocoder(eng._ctx, spec.data_ptr(), 1, spec.shape[1], 0.5, spec.shape[1] * 2 + 1,
                                  out.data_ptr(), None)
    assert rc != 0 and b"n_frames_out" in eng.lib.aw_last_error()
    with pytest.raises(ValueError):
        _lib.check(eng.lib.aw_istft_full(eng._ctx, spec.data_ptr(), 1, spec.shape[1], 0, out.data_ptr(), 1, None))
    with pytest.raises(ValueError):
        eng.stft_full(torch.zeros((1, 1024), device="cuda"))


@pytest.mark.gpu
@pytest.mark.parametrize("sr,secs", SIZES)
def test_attacks_end_to_end_match_the_restatement(model, sr, secs):
    """Bounds are estimates: float32 FFT round-off (~1e-7) perturbs the angle differences, and for
    rate != 1 the accumulated phase random-walks with it.  Measured values are printed."""
    x = np.stack([O.synth_clip(i, secs, sr) for i in (5, 6)])
    xd = torch.from_numpy(x).cuda()
    for att in (A.TimeStretch(0.8), A.TimeStretch(1.25), A.PitchShift(-2), A.PitchShift(2)):
        got = att.apply_batch(xd, sr).cpu().numpy()
        for i in range(2):
            if isinstance(att, A.TimeStretch):
                want = D.attack_time_stretch(x[i], att.rate)
            else:
                want = D.attack_pitch_shift(x[i], att.n_steps)
            assert got[i].shape == want.shape
            mg, mw = D.stft(got[i]).abs().numpy(), D.stft(want).abs().numpy()
            d_mag = np.abs(mg - mw).max() / mw.max()
            snr = _snr(got[i], want)
            print("%s @ %d Hz clip %d: max |STFT| diff %.2e of max, SNR %.1f dB" % (att.name, sr, i, d_mag, snr))
            assert d_mag <= 1e-3 and snr >= 40.0


@pytest.mark.gpu
def test_a_clip_in_a_batch_equals_the_clip_alone_and_silence_stays_zero(model):
    sr = 16000
    x = np.stack([O.synth_clip(i, 1.3, sr) for i in range(8)])
    x[5] = 0.0
    xd = torch.from_numpy(x).cuda()
    for att in (A.TimeStretch(0.9), A.TimeStretch(1.1), A.PitchShift(-2), A.PitchShift(2)):
        batch = att.apply_batch(xd, sr).cpu().numpy()
        alone = att.apply_batch(xd[3:4].contiguous(), sr).cpu().numpy()
        np.testing.assert_array_equal(batch[3], alone[0])
        assert np.isfinite(batch).all() and (batch[5] == 0).all()


@pytest.mark.gpu
def test_desync_robustness_is_reported_and_detector_bits_match_the_oracle(model):
    """Robustness is reported, not gated.  On the same GPU-attacked audio the CUDA detector's bits equal
    the CPU oracle's wherever the oracle's margin is at least 1e-3."""
    from aware_b200.service import detect_watermark_batch, embed_watermark_batch
    emb, det = model
    sr = 44100
    x = np.stack([O.synth_clip(i, 1.5, sr) for i in (1, 2)])
    bits = O.synth_bits(2)
    emb.num_iterations, prev = 150, emb.num_iterations
    emb.enforce_16k = det.enforce_16k = False
    try:
        y = embed_watermark_batch(x, sr, bits, emb)
        for att in A.desync_attacks():
            z = att.apply_batch(y, sr)
            dec = detect_watermark_batch(z, sr, det).cpu().numpy()
            print("%s: BER %.1f %%" % (att.name, 100 * (dec != bits).mean()))
            zc = z.cpu().numpy()
            for i in range(2):
                v = O.detect(zc[i], sr)
                sure = np.abs(v) >= 1e-3
                np.testing.assert_array_equal(dec[i][sure], O.decode_values(v)[sure])
    finally:
        emb.num_iterations = prev
        emb.enforce_16k = det.enforce_16k = True


@pytest.mark.gpu
def test_evaluation_driver_appends_the_desync_attacks_on_request(model):
    from aware_b200.evaluate import default_attacks, evaluate_clips
    emb, det = model
    clips = [O.synth_clip(0, 2.0, 16000), O.synth_clip(1, 1.5, 16000), O.synth_clip(2, 1.2, 44100)]
    rates = [16000, 16000, 44100]
    defaults = ["orig"] + [a.name for a in default_attacks(np.random.default_rng(0))]
    prev = emb.num_iterations
    emb.num_iterations = 20
    try:
        plain = evaluate_clips(clips, rates, emb, det, seed=3)
        extra = evaluate_clips(clips, rates, emb, det, seed=3, desync=True)
    finally:
        emb.num_iterations = prev
    assert list(plain["ber_percent"]) == defaults
    assert list(extra["ber_percent"]) == defaults + [a.name for a in A.desync_attacks()]
    assert all(0.0 <= v <= 100.0 for v in extra["ber_percent"].values())
    print({k: round(v, 1) for k, v in extra["ber_percent"].items() if k not in defaults})

"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle and the
committed reference outputs (tests/golden).  Run with `pytest -m gpu` on the B200 box.

Tolerances (BASELINE.json north_star): decoded bits / BER counts bit-exact; integer- and
copy-type attacks bit-exact; floating-point tensors max-abs <= 1e-4 (relative to peak) and
SNR >= 80 dB; detector outputs <= 1e-5 (fp32 GEMMs) / <= 1e-3 (TF32 tensor-core GEMMs).
The iterative embed is chaotic (SURVEY F7): it is gated per step and functionally."""
import os
import random

import numpy as np
import pytest
import torch

import aware_oracle as O

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def model():
    from aware_b200 import attacks as A
    from aware_b200.utils.models import load
    emb, det = load()
    emb.verbose = False
    A.set_engine(emb.engine)
    return emb, det


@pytest.fixture(scope="module")
def eng(model):
    return model[0].engine


def _clips(idx, secs, sr):
    return np.stack([O.synth_clip(i, secs, sr) for i in idx])


def _snr(a, b):
    return 10 * np.log10(np.sum(b.astype(np.float64) ** 2) / max(np.sum((a.astype(np.float64) - b) ** 2), 1e-300))


# ------------------------------------------------------------------ STFT / iSTFT
@pytest.mark.parametrize("sr,secs", [(16000, 1.3), (44100, 1.0), (44100, 2.7)])
def test_stft_band_matches_torch_stft(eng, sr, secs):
    x = _clips([0, 1, 2], secs, sr)
    mag, ph = eng.stft_band(torch.from_numpy(x).cuda(), sr, phasor=True)
    mag, ph = mag.cpu().numpy(), ph.cpu().numpy()
    fi, _ = O.band_indices(sr)
    assert eng.band_bins(sr) == (int(fi[0]), len(fi))
    for i in range(len(x)):
        s = O.stft(O.normalize_waveform(torch.from_numpy(x[i]))).numpy()[fi].T
        assert mag[i].shape == s.shape
        peak = np.abs(s).max()
        assert np.abs(mag[i] - np.abs(s)).max() <= 1e-5 * peak
        spec = (ph[i][..., 0] + 1j * ph[i][..., 1]) * mag[i]
        assert np.abs(spec - s).max() <= 1e-5 * peak
        assert _snr(np.ascontiguousarray(spec.astype(np.complex64)).view(np.float32),
                    np.ascontiguousarray(s.astype(np.complex64)).view(np.float32)) >= 80


@pytest.mark.parametrize("sr,secs", [(16000, 1.3), (44100, 1.0)])
def test_istft_band_matches_torch_istft(eng, sr, secs):
    x = _clips([3, 4], secs, sr)
    mag, ph = eng.stft_band(torch.from_numpy(x).cuda(), sr, phasor=True)
    y = eng.istft_band(mag, ph, sr).cpu().numpy()
    _, nfi = O.band_indices(sr)
    for i in range(len(x)):
        s = O.stft(O.normalize_waveform(torch.from_numpy(x[i])))
        s[torch.from_numpy(nfi)] = 0
        yr = O.istft(s).numpy()
        assert y[i].shape == yr.shape == (256 * (x.shape[1] // 256),)
        assert np.abs(y[i] - yr).max() <= 1e-5
        assert _snr(y[i], yr) >= 80


# ------------------------------------------------------------------ GEMM
@pytest.mark.parametrize("rows,n,k", [(128, 64, 64), (256, 128, 512), (384, 512, 128), (256, 1024, 1024),
                                      (1280, 1024, 512), (256, 64, 1024), (256, 1024, 64)])
def test_gemm_tensor_core_and_exact(eng, rows, n, k):
    torch.manual_seed(rows + n + k)
    a = torch.randn(rows, k, device="cuda")
    b = torch.randn(n, k, device="cuda") / k ** 0.5
    want = a.double() @ b.double().T
    scale = want.abs().max().item()
    assert (eng.gemm(a, b, "fp32").double() - want).abs().max().item() <= 1e-5 * scale
    # TF32 operands (10-bit mantissa), fp32 accumulate
    assert (eng.gemm(a, b, "tf32").double() - want).abs().max().item() <= 4e-3 * scale


# ------------------------------------------------------------------ detect
@pytest.mark.parametrize("precision,tol", [("fp32", 1e-5), ("tf32", 1e-3), ("fp16", 1e-3)])
def test_detect_matches_oracle(eng, precision, tol):
    """Raw tensor-core outputs (exact re-evaluation switched off) against the oracle, with the flip
    rate below the 1e-3 margin reported (SURVEY 8c(2))."""
    eng.set_precision(precision)
    eng.set_exact_margin(0.0)
    n_low = n_flip = 0
    try:
        for sr, secs in ((16000, 2.0), (44100, 1.5), (44100, 3.1)):
            x = _clips([0, 1, 2, 3, 4], secs, sr)
            v = eng.detect(torch.from_numpy(x).cuda(), sr).cpu().numpy()
            ref = np.stack([O.detect(x[i], sr) for i in range(len(x))])
            assert np.abs(v - ref).max() <= tol
            safe = np.abs(ref) > tol                       # un-watermarked clips have ~0 margins
            assert np.array_equal((v > 0)[safe], (ref > 0)[safe])
            n_low += int((~safe).sum())
            n_flip += int(((v > 0) != (ref > 0))[~safe].sum())
    finally:
        eng.set_precision("tf32")
        eng.set_exact_margin(1e-3)
    print("%s: %d values below the %g margin, %d of them decoded differently" % (precision, n_low, tol, n_flip))


def test_detect_bits_exact_through_low_margin_reevaluation(eng):
    """Default detect path (TF32 tensor cores + exact re-evaluation of clips whose margin is below
    1e-3): decoded bits equal the oracle's on UN-watermarked clips, whose outputs sit near 0 --
    everywhere except where the reference's own fp32 value is within 1e-5 of the threshold (there
    fp32 summation order decides, reference vs reference)."""
    before = eng.detect_stats()
    n_low = 0
    for sr, secs, idx in ((16000, 2.0, range(0, 12)), (44100, 1.5, range(12, 20))):
        x = _clips(list(idx), secs, sr)
        v = eng.detect(torch.from_numpy(x).cuda(), sr).cpu().numpy()
        ref = np.stack([O.detect(x[i], sr) for i in range(len(x))])
        low = np.abs(ref).min(axis=1) < 1e-3
        n_low += int(low.sum())
        decidable = np.abs(ref) >= 1e-5
        assert np.array_equal((v > 0)[decidable], (ref > 0)[decidable])
        assert np.abs(v - ref)[low].max(initial=0.0) <= 2e-6          # re-evaluated clips: fp32-exact values
        bits = eng.decide(torch.from_numpy(v).cuda()).cpu().numpy()
        want = np.stack([O.decode_values(r) for r in ref])
        assert np.array_equal(bits[decidable], want[decidable])
    after = eng.detect_stats()
    assert after[0] - before[0] == 20
    assert after[1] - before[1] >= n_low                               # every low-margin clip was re-evaluated
    print("low-margin clips: %d of 20, re-evaluated %d" % (n_low, after[1] - before[1]))


def test_detect_matches_reference_golden(eng):
    g = np.load(os.path.join(GOLDEN, "detect.npz"))
    eng.set_precision("fp32")
    try:
        for key in g.files:
            _, sr, clip, secs = key.split("_")
            sr, clip, secs = int(sr[2:]), int(clip[4:]), float(secs[1:])
            x = O.synth_clip(clip, secs, sr)[None]
            v = eng.detect(torch.from_numpy(x).cuda(), sr).cpu().numpy()[0]
            np.testing.assert_allclose(v, g[key], atol=1e-5, rtol=0, err_msg=key)
    finally:
        eng.set_precision("tf32")


def test_detect_on_reference_watermarked_audio_bits_exact(model):
    """Cross-detection: audio watermarked by the UNMODIFIED reference (golden), decoded by the
    CUDA detector through the service API: bits and BER identical to the reference's."""
    from aware_b200.metrics.audio import BER
    from aware_b200.service import detect_watermark
    emb, det = model
    g = np.load(os.path.join(GOLDEN, "embed_full.npz"))
    got = detect_watermark(g["wave"], 16000, det)
    np.testing.assert_array_equal(got, g["decoded"])
    assert BER()(g["bits"], got) == float(g["ber"]) == 0.0
    np.testing.assert_allclose(det.detect(g["wave"], 16000), g["values"], atol=1e-3)
    det.enforce_16k = False
    try:
        np.testing.assert_array_equal(detect_watermark(g["wave44"], 44100, det), g["decoded44"])
    finally:
        det.enforce_16k = True


def test_decide_and_count_matches_numpy(eng):
    rng = np.random.default_rng(0)
    v = rng.uniform(-1, 1, (37, 20)).astype(np.float32)
    v[0, :3] = [0.0, 1e-12, -1e-12]                        # strict '>' at the threshold
    ref = rng.integers(0, 2, (37, 20), dtype=np.int32)
    counters = torch.zeros(3, dtype=torch.int64, device="cuda")
    bits, errs = eng.decide(torch.from_numpy(v).cuda(), torch.from_numpy(ref), counters)
    want = np.stack([O.decode_values(r) for r in v])
    np.testing.assert_array_equal(bits.cpu().numpy(), want)
    np.testing.assert_array_equal(errs.cpu().numpy(), (want != ref).sum(1))
    assert counters.tolist() == [int((want != ref).sum()), 37 * 20, 37]
    assert O.ber_percent(want, ref) == pytest.approx(100.0 * counters[0].item() / counters[1].item())


def test_snr_kernel_matches_metric(eng):
    from aware_b200.metrics.audio import SNR
    x = _clips([0, 1], 0.5, 16000)
    y = x + 0.01 * np.random.default_rng(1).standard_normal(x.shape).astype(np.float32)
    s = eng.snr(torch.from_numpy(y).cuda(), torch.from_numpy(x).cuda()).cpu().numpy()
    for i in range(2):
        assert s[i] == pytest.approx(SNR()(y[i], x[i]), abs=1e-3)


# ------------------------------------------------------------------ attacks
@pytest.mark.parametrize("sr", [16000, 44100])
def test_attacks_match_oracle(model, sr):
    from aware_b200 import attacks as A
    x = _clips([3, 5], 0.8, sr)
    xd = torch.from_numpy(x).cuda()
    n = x.shape[1]

    def check(att, want_fn, exact=True, tol=0.0):
        got = att.apply_batch(xd, sr).cpu().numpy()
        for i in range(len(x)):
            want = np.asarray(want_fn(x[i], i), dtype=np.float32)
            assert got[i].shape == want.shape, att.name
            if exact:
                np.testing.assert_array_equal(got[i], want, err_msg=att.name)
            else:
                assert np.abs(got[i] - want).max() <= tol, att.name

    for pcm in (8, 12, 16, 24):
        check(A.PCMBitDepthConversion(pcm), lambda a, i: O.attack_pcm(a, pcm))
    st = np.array([100, n // 2])
    check(A.DeleteSamples(0.15, start=st), lambda a, i: O.attack_delete(a, 0.15, int(st[i])))
    check(A.SampleSupression(0.25, start=st), lambda a, i: O.attack_suppress(a, 0.25, sr, int(st[i])))
    check(A.Cropout(0.1), lambda a, i: O.attack_cropout(a, 0.1, sr))
    check(A.Resample(), lambda a, i: O.attack_resample(a, sr))
    # IIR attacks: the default sequential scan reproduces scipy's float64 recurrence bit for bit
    check(A.LowPassFilter(), lambda a, i: O.attack_lowpass(a, sr))
    check(A.HighPassFilter(), lambda a, i: O.attack_highpass(a, sr))
    random.seed(5)
    f_low = random.uniform(300.0, 3800.0)
    check(A.RandomBandstop(f_low=f_low), lambda a, i: O.attack_bandstop(a, sr, f_low))
    # chunk-parallel variants: to float32 resolution for the well-conditioned designs
    check(A.LowPassFilter(fast=True), lambda a, i: O.attack_lowpass(a, sr), exact=False, tol=1e-6)
    check(A.HighPassFilter(fast=True), lambda a, i: O.attack_highpass(a, sr), exact=False, tol=1e-6)


def test_attacks_match_reference_golden(model):
    from aware_b200 import attacks as A
    for sr in (16000, 44100):
        g = np.load(os.path.join(GOLDEN, "attacks_sr%d.npz" % sr))
        x = O.synth_clip(3, 0.4, sr)
        n = len(x)
        for pcm in (8, 12, 16, 24):
            np.testing.assert_array_equal(A.PCMBitDepthConversion(pcm).apply(x, sr), g["pcm%d_sr%d" % (pcm, sr)])
        for p in (0.1, 0.15, 0.2):
            np.random.seed(11)
            st = np.random.randint(0, n - int(p * n))
            np.testing.assert_array_equal(A.DeleteSamples(p, start=st).apply(x, sr), g["delete%g_sr%d" % (p, sr)])
        for p in (0.1, 0.25):
            np.random.seed(12)
            st = np.random.randint(0, n - int(p * sr))
            np.testing.assert_array_equal(A.SampleSupression(p, start=st).apply(x, sr), g["suppress%g_sr%d" % (p, sr)])
        np.testing.assert_array_equal(A.Cropout(0.1).apply(x, sr), g["cropout0.1_sr%d" % sr])
        np.testing.assert_array_equal(A.Resample().apply(x, sr), g["resample_sr%d" % sr].astype(np.float32))
        random.seed(13)
        f_low = random.uniform(300.0, 3800.0)
        np.testing.assert_array_equal(A.RandomBandstop(f_low=f_low).apply(x, sr), g["bandstop_sr%d" % sr])
        np.testing.assert_array_equal(A.LowPassFilter().apply(x, sr), g["lowpass_sr%d" % sr].astype(np.float32))
        np.testing.assert_array_equal(A.HighPassFilter().apply(x, sr), g["highpass_sr%d" % sr].astype(np.float32))


def test_long_clip_iir_scans(model):
    """5 s clip: sequential scan bit-exact; chunk-parallel scan (many chunks, look-back warm-up)
    to float32 resolution for low/high-pass and to the direct form's own round-off noise
    (distance to the SOS evaluation) for the ill-conditioned band-stop."""
    from scipy.signal import butter, sosfiltfilt
    from aware_b200 import attacks as A
    sr = 44100
    x = _clips([6], 5.0, sr)
    xd = torch.from_numpy(x).cuda()
    lp, hp = O.attack_lowpass(x[0], sr).astype(np.float32), O.attack_highpass(x[0], sr).astype(np.float32)
    np.testing.assert_array_equal(A.LowPassFilter().apply_batch(xd, sr).cpu().numpy()[0], lp)
    np.testing.assert_array_equal(A.HighPassFilter().apply_batch(xd, sr).cpu().numpy()[0], hp)
    assert np.abs(A.LowPassFilter(fast=True).apply_batch(xd, sr).cpu().numpy()[0] - lp).max() <= 1e-6
    assert np.abs(A.HighPassFilter(fast=True).apply_batch(xd, sr).cpu().numpy()[0] - hp).max() <= 1e-6
    for f_low in (3700.0, 1206.5):
        ref = O.attack_bandstop(x[0], sr, f_low)
        np.testing.assert_array_equal(A.RandomBandstop(f_low=f_low).apply_batch(xd, sr).cpu().numpy()[0], ref)
        sos = butter(4, [f_low / (sr / 2), (f_low + 200.0) / (sr / 2)], btype="bandstop", output="sos")
        noise = np.abs(sosfiltfilt(sos, x[0].astype(np.float64), padlen=27) - ref).max()
        fast = A.RandomBandstop(f_low=f_low, fast=True).apply_batch(xd, sr).cpu().numpy()[0]
        assert np.abs(fast - ref).max() <= 10 * noise + 1e-6, (f_low, noise)


# ------------------------------------------------------------------ embed
def _gate_waveform_1e4(got, ref, frac=0.995):
    """north_star tolerance for one optimisation step: max-abs <= 1e-4 and SNR >= 80 dB.  A NAdam
    first step is lr * sign(g) for |g| >> 1e-8, so the few coefficients whose gradient is within
    fp32 noise of 0 move by 2 * lr = 0.2 in the other direction; each one perturbs the 4 frames
    (1024 samples) it overlaps.  The gate therefore holds the STATED tolerance on at least `frac` of
    the samples, reports the distribution of the rest, and bounds the rest loosely."""
    d = np.abs(got.astype(np.float64) - ref)
    ok = d <= 1e-4
    share = ok.mean()
    print("one-step waveform: %.4f %% of samples within 1e-4, max %.2e, p99.9 %.2e, SNR(all) %.1f dB, "
          "SNR(within) %.1f dB" % (100 * share, d.max(), np.quantile(d, 0.999), _snr(got, ref),
                                    _snr(got[ok], ref[ok])))
    assert share >= frac, share
    assert _snr(got[ok], ref[ok]) >= 80.0
    assert d.max() <= 3e-3 and _snr(got, ref) >= 70.0


def _embed_state(eng, x, sr, pat, iters, precision):
    eng.set_precision(precision)
    try:
        out, best, losses = eng.embed(torch.from_numpy(x).cuda(), sr, torch.from_numpy(pat), iters=iters,
                                      return_losses=True)
        T = 1 + x.shape[1] // 256
        st = {k: eng.embed_state(k, len(x), T, sr).cpu().numpy() for k in ("c", "c0", "m")}
    finally:
        eng.set_precision("tf32")
    return out.cpu().numpy(), losses.cpu().numpy(), st


@pytest.mark.parametrize("sr,secs", [(16000, 1.0), (44100, 0.8)])
def test_embed_one_iteration_matches_oracle(eng, sr, secs):
    """One optimisation step from identical state (fp32 GEMMs): initial coefficients, loss,
    gradient and updated coefficients against the oracle.  A NAdam first step is
    lr * g / (|g| + 1e-8), i.e. discontinuous at g = 0, and the reference's own fp32
    gradient is only accurate to ~2e-3 of its median magnitude (fp32 vs fp64, measured),
    so a handful of near-zero-gradient coefficients legitimately land on the other side:
    the gate is >= 99.5 % of coefficients within 1e-4 and the gradient within fp32 noise."""
    from kernel_model import Model
    x = _clips([0], secs, sr)
    pat = np.stack([O.encode_bits(O.synth_bits(8)[0])])
    out, losses, st = _embed_state(eng, x, sr, pat, 1, "fp32")
    keep = {}
    y = O.embed(x[0], sr, pat[0], num_iters=1, keep=keep)
    T = 1 + x.shape[1] // 256
    B = st["c"].shape[2]
    c0_ref = keep["c0"].numpy().reshape(B, T).T
    c_ref = keep["coeffs_after"][1].numpy().reshape(B, T).T
    g_ref = keep["grads"][0].numpy().reshape(B, T).T
    assert np.abs(st["c0"][0] - c0_ref).max() <= 1e-5 * np.abs(c0_ref).max()
    assert abs(losses[0, 0] - keep["losses"][0]) <= 1e-5
    g_gpu = st["m"][0] / 0.1                               # m_1 = (1 - beta1) * g
    fi, _ = O.band_indices(sr)
    mdl = Model(O.make_weights(), O.mel_basis(), fi)
    mdl.forward(mdl.init(x[0]), pat[0].astype(np.float64))
    g64 = mdl.backward(pat[0].astype(np.float64))
    rms = lambda a: float(np.sqrt(np.mean(a ** 2)))        # noqa: E731
    # LeakyReLU is not differentiable at 0: a pre-activation within fp32 rounding of the kink
    # (|IN output| ~ 1e-6) takes slope 1 in one fp32 evaluation order and 0.2 in another, and
    # that one pooled row's gradient then differs by O(1 %) in either implementation.  Rows
    # whose float64 pre-activation is that close to 0 reach frames 2j-3 .. 2j+4 through the
    # STFT/iSTFT adjoints (7-frame support): those frames are compared separately.
    kink = np.zeros(T, dtype=bool)
    for P in mdl.s["P"][1:]:
        hh = np.abs(np.where(P > 0, P, P / 0.2))
        for j in np.nonzero((hh < 2e-5).any(axis=1))[0]:
            kink[max(0, 2 * j - 4):2 * j + 6] = True
    assert kink.mean() < 0.5
    ok = ~kink
    err_gpu, err_ref = rms((g_gpu - g64)[ok]), rms((g_ref - g64)[ok])
    assert err_gpu <= 5 * err_ref + 1e-12, (err_gpu, err_ref)   # as close to the truth as torch-fp32 is
    assert rms((g_gpu - g_ref)[ok]) <= 1e-3 * rms(g_ref[ok])
    assert rms(g_gpu - g_ref) <= 5e-2 * rms(g_ref)              # kink frames: bounded, not equal
    d = np.abs(st["c"][0] - c_ref)
    assert (d <= 1e-4 * np.maximum(1.0, np.abs(c_ref))).mean() >= 0.995
    _gate_waveform_1e4(out[0], y)


def test_embed_one_iteration_matches_reference_golden(eng):
    g = np.load(os.path.join(GOLDEN, "embed_short.npz"))
    pat = np.stack([O.encode_bits(O.synth_bits(8)[0])])
    for sr in (16000, 44100):
        x = _clips([0], 1.0, sr)
        out, _, _ = _embed_state(eng, x, sr, pat, 1, "fp32")
        ref = g["wave_sr%d_it1" % sr]
        assert out[0].shape == ref.shape
        _gate_waveform_1e4(out[0], ref)


def test_embed_three_iterations_losses_track_oracle(eng):
    x = _clips([1], 1.0, 16000)
    pat = np.stack([O.encode_bits(O.synth_bits(8)[1])])
    keep = {}
    O.embed(x[0], 16000, pat[0], num_iters=3, keep=keep)
    for precision, tol in (("fp32", 2e-3), ("tf32", 1e-2), ("fp16", 1e-2)):
        _, losses, _ = _embed_state(eng, x, 16000, pat, 3, precision)
        assert np.abs(losses[:3, 0] - np.array(keep["losses"])).max() <= tol, precision


@pytest.mark.parametrize("precision", ["tf32", "fp32", "fp16"])
def test_embed_full_functional_parity(model, precision):
    """400 iterations through the service API: bits recovered by the CUDA detector AND by the
    CPU oracle (cross-detection), SNR within 1 dB of the reference's golden run."""
    from aware_b200.service import detect_watermark, embed_watermark
    emb, det = model
    g = np.load(os.path.join(GOLDEN, "embed_full.npz"))
    x = O.synth_clip(1, 2.0, 16000)
    emb.engine.set_precision(precision)
    prev = emb.embed_precision
    emb.embed_precision = precision
    emb.num_iterations = 400
    try:
        y = embed_watermark(x, 16000, g["bits"], emb)
        got = detect_watermark(y, 16000, det)
    finally:
        emb.engine.set_precision("tf32")
        emb.embed_precision = prev
    assert y.shape == g["wave"].shape and y.dtype == np.float32
    np.testing.assert_array_equal(got, g["bits"])                       # BER 0, as the reference
    np.testing.assert_array_equal(O.detect_watermark(y, 16000), g["bits"])
    assert abs(O.snr_db(y, x) - float(g["snr"])) <= 1.0                 # BASELINE.md section 3: +-1 dB
    assert np.abs(det.detect(y, 16000)).min() > 0.05                    # comfortable margins


def test_batched_pipeline_ber_bit_exact_vs_oracle(model):
    """embed -> attack -> detect -> BER on a small batch: per-clip decoded bits and error
    counts from the CUDA path equal the oracle's on the same (GPU-embedded) audio."""
    from aware_b200 import attacks as A
    from aware_b200.service import detect_watermark_batch, embed_watermark_batch
    emb, det = model
    emb.num_iterations = 120
    emb.enforce_16k = det.enforce_16k = False
    sr = 44100
    try:
        x = _clips([0, 1, 2, 3], 2.0, sr)
        bits = O.synth_bits(4)
        y = embed_watermark_batch(x, sr, bits, emb)
        counters = torch.zeros(3, dtype=torch.int64, device="cuda")
        dec, errs = detect_watermark_batch(y, sr, det, bits, counters)
        yh = y.cpu().numpy()
        want = np.stack([O.detect_watermark(yh[i], sr) for i in range(4)])
        np.testing.assert_array_equal(dec.cpu().numpy(), want)
        assert counters.tolist() == [int((want != bits).sum()), 80, 4]
        for att, fn in ((A.PCMBitDepthConversion(8), lambda a: O.attack_pcm(a, 8)),
                        (A.Resample(), lambda a: O.attack_resample(a, sr)),
                        (A.LowPassFilter(), lambda a: O.attack_lowpass(a, sr))):
            z = att.apply_batch(y, sr)
            dec = detect_watermark_batch(z, sr, det).cpu().numpy()
            ref_vals = np.stack([O.detect(np.asarray(fn(yh[i]), dtype=np.float32), sr) for i in range(4)])
            safe = np.abs(ref_vals) > 1e-3
            assert np.array_equal(dec[safe], (ref_vals > 0)[safe].astype(np.int32)), att.name
    finally:
        emb.num_iterations = 400
        emb.enforce_16k = det.enforce_16k = True


def test_full_size_batch_properties(model):
    """BASELINE-size clips (10 s @ 44.1 kHz, a slice of the 256-clip batch): size-independent
    properties -- output length 256*(N//256), |y| <= 1 with the peak at exactly 1/(1+1e-8),
    a clip's result does not depend on its neighbours in the batch, and wave-splitting the
    batch gives bit-identical audio."""
    from aware_b200.synth import synth_batch, synth_bits
    emb, _ = model
    eng = emb.engine
    sr = 44100
    x = torch.from_numpy(synth_batch(6, 10.0, sr)).cuda()
    pat = torch.from_numpy(2 * synth_bits(6) - 1)
    y_all = eng.embed(x, sr, pat, iters=8)
    assert y_all.shape == (6, 256 * (x.shape[1] // 256))
    peak = y_all.abs().max(dim=1).values.cpu().numpy()
    assert np.all(peak <= 1.0) and np.all(peak > 0.999999)
    y_sub = eng.embed(x[2:4], sr, pat[2:4], iters=8)
    assert torch.equal(y_sub, y_all[2:4])
    y_wave = eng.embed(x, sr, pat, iters=8, wave_clips=4)
    assert torch.equal(y_wave, y_all)
    v = eng.detect(y_all, sr)
    assert v.shape == (6, 20) and torch.isfinite(v).all()


def test_long_clips_config4_and_config5_shapes(eng):
    """BASELINE configs[3] clip length (30 s) and a long-form clip (5 min, the configs[4] code path
    with T = 51 681 frames on one GPU): detector outputs against the oracle, a one-iteration embed
    against the oracle at 30 s, and finite / deterministic long-form embedding."""
    sr = 44100
    x30 = _clips([5], 30.0, sr)
    v = eng.detect(torch.from_numpy(x30).cuda(), sr).cpu().numpy()[0]
    assert np.abs(v - O.detect(x30[0], sr)).max() <= 1e-3
    pat = np.stack([O.encode_bits(O.synth_bits(8)[5])])
    out, _, _ = _embed_state(eng, x30, sr, pat, 1, "fp32")
    y = O.embed(x30[0], sr, pat[0], num_iters=1)
    assert out.shape == (1, 256 * (x30.shape[1] // 256))
    # 418 k coefficients: a handful of sign flips of the NAdam first step (|g| ~ 0) are expected
    assert _snr(out[0], y) >= 75 and np.abs(out[0] - y).max() <= 3e-3
    x300 = np.tile(_clips([6], 30.0, sr), (1, 10))                  # 5 min
    xd = torch.from_numpy(x300).cuda()
    v = eng.detect(xd, sr).cpu().numpy()[0]
    assert np.abs(v - O.detect(x300[0], sr)).max() <= 1e-3
    ya = eng.embed(xd, sr, torch.from_numpy(pat), iters=3)
    yb = eng.embed(xd, sr, torch.from_numpy(pat), iters=3)
    assert ya.shape == (1, 256 * (x300.shape[1] // 256)) and torch.isfinite(ya).all()
    assert torch.equal(ya, yb)
    # the fp16 loop's gradient loss scale grows with the clip length (gradients shrink like 1/T'):
    # its loss trajectory stays on the TF32 loop's
    traj = {}
    for prec in ("tf32", "fp16"):
        _, _, losses = eng.embed(xd, sr, torch.from_numpy(pat), iters=12, return_losses=True, precision=prec)
        traj[prec] = losses[:12, 0].cpu().numpy()
    assert traj["tf32"][-1] < traj["tf32"][0] - 0.05                 # the optimiser makes progress
    assert np.abs(traj["fp16"] - traj["tf32"]).max() <= 2e-2, traj


@pytest.mark.parametrize("n_samples", [1100, 2048, 2303, 58 * 256 + 7, 59 * 256 + 1, 65 * 256, 115 * 256 + 13,
                                       116 * 256 + 3, 117 * 256 + 250, 123 * 256])
def test_embed_tile_edges_match_oracle(eng, n_samples):
    """Clip lengths that put the fused spectral kernel's tile seams everywhere: fewer frames than
    one tile (T = 5..9), exactly one / two / three tiles, and a last tile shorter than the
    8-frame reflect seam (T = 60, 117, 118): two optimisation steps against the oracle."""
    sr = 44100
    x = O.synth_clip(3, 1.0 + n_samples / sr, sr)[None, :n_samples].copy()
    pat = np.stack([O.encode_bits(O.synth_bits(8)[3])])
    out, losses, st = _embed_state(eng, x, sr, pat, 2, "fp32")
    keep = {}
    y = O.embed(x[0], sr, pat[0], num_iters=2, keep=keep)
    T = 1 + n_samples // 256
    B = st["c"].shape[2]
    assert out.shape == (1, 256 * (T - 1))
    c0_ref = keep["c0"].numpy().reshape(B, T).T
    assert np.abs(st["c0"][0] - c0_ref).max() <= 1e-5 * np.abs(c0_ref).max()
    # T = 5 pools to T' = 2 frames: InstanceNorm over two samples divides by sqrt(var + 1e-5) with
    # var ~ 1e-5 for many channels, which amplifies fp32 rounding ~100x (the detect-only path shows
    # the same 7e-5 there against 2e-6 from T = 7 on): a conditioning limit of the degenerate clip
    assert abs(losses[0, 0] - keep["losses"][0]) <= (3e-3 if T <= 6 else 2e-5)
    g_ref = keep["grads"][0].numpy().reshape(B, T).T
    c1_ref = keep["coeffs_after"][1].numpy().reshape(B, T).T
    # the first NAdam step is sign-like: compare where the reference gradient is not ~0
    big = np.abs(g_ref) > 1e-2 * np.median(np.abs(g_ref))
    # c after step 1 is not kept by the kernel; the loss of step 2 depends on all of it
    if T > 6:
        assert abs(losses[1, 0] - keep["losses"][1]) <= 5e-3, (losses[:2, 0], keep["losses"])
    assert big.mean() > 0.5 and np.isfinite(out).all()
    assert _snr(out[0], y) >= (25 if T <= 6 else 55)
    assert c1_ref.shape == st["c"][0].shape


@pytest.mark.gpu
def test_evaluation_driver_ragged_clips(model):
    """aware_b200.evaluate (batched scripts/test.py): clips of different lengths and rates are
    resampled to 16 kHz on the GPU bit-exactly like scipy.signal.resample_poly, bucketed by
    length, embedded, attacked and detected; the decoded bits equal the CPU oracle's on the same
    watermarked audio and the clean BER is 0."""
    from scipy.signal import resample_poly
    from aware_b200.evaluate import evaluate_clips, resample_poly_batch
    emb, det = model
    eng = emb.engine
    clips = [O.synth_clip(0, 2.0, 16000), O.synth_clip(1, 2.0, 16000), O.synth_clip(2, 1.5, 44100),
             O.synth_clip(3, 1.25, 32000), O.synth_clip(4, 1.5, 44100)]
    rates = [16000, 16000, 44100, 32000, 44100]
    for x, sr in ((clips[2], 44100), (clips[3], 32000)):
        want = resample_poly(x, 16000, sr)
        got = resample_poly_batch(torch.from_numpy(x[None]).cuda(), 16000, sr, eng).cpu().numpy()[0]
        np.testing.assert_array_equal(got, want.astype(np.float32))
    prev = emb.num_iterations
    emb.num_iterations = 200
    try:
        res = evaluate_clips(clips, rates, emb, det, seed=3, keep_audio=True)
    finally:
        emb.num_iterations = prev
    assert res["n_clips"] == 5 and set(res["decoded"]) == set(range(5))
    assert res["ber_percent"]["orig"] == 0.0
    assert {"pcm_8", "delete_0.1", "resample_16000", "low_pass", "high_pass"} <= set(res["ber_percent"])
    assert all(0.0 <= v <= 60.0 for v in res["ber_percent"].values())
    assert 15.0 < res["snr_db_mean"] < 45.0
    # quality aggregates (scripts/test.py:76-88): GPU STOI of watermarked vs original audio, equal to the numpy
    # restatement clip by clip; PESQ only where the third-party package exists
    import stoi_oracle as S
    from scipy.signal import resample_poly
    st = []
    for i in range(5):
        x16 = clips[i] if rates[i] == 16000 else resample_poly(clips[i], 16000, rates[i])
        w = res["audio"][i]
        st.append(S.stoi(np.asarray(x16[:len(w)], dtype=np.float64), w.astype(np.float64), 16000))
    st = np.array(st)
    assert abs(res["stoi_mean"] - st[st > 0.1].mean()) <= 1e-4, (res["stoi_mean"], st)
    assert np.isnan(res["pesq_mean"]) or 1.0 <= res["pesq_mean"] <= 4.7
    for i in range(5):
        np.testing.assert_array_equal(res["decoded"][i], res["bits"][i])
        np.testing.assert_array_equal(O.detect_watermark(res["audio"][i], 16000), res["bits"][i])


@pytest.mark.parametrize("sr", [22050, 32000, 48000])
def test_other_sample_rates_use_generic_band_kernels(eng, sr):
    """Rates whose 500-4000 Hz band does not fall in the two specialised 32-bin group ranges
    (22.05 kHz: bins 24..185, 32 kHz: 16..128) run the generic <0,15> kernel instantiations;
    48 kHz (bins 11..85) shares the 44.1 kHz one.  Detector and one optimisation step vs the oracle."""
    x = _clips([2], 1.2, sr)
    eng.set_precision("fp32")
    try:
        v = eng.detect(torch.from_numpy(x).cuda(), sr).cpu().numpy()[0]
    finally:
        eng.set_precision("tf32")
    assert np.abs(v - O.detect(x[0], sr)).max() <= 1e-5
    pat = np.stack([O.encode_bits(O.synth_bits(8)[2])])
    out, losses, st = _embed_state(eng, x, sr, pat, 2, "fp32")
    keep = {}
    y = O.embed(x[0], sr, pat[0], num_iters=2, keep=keep)
    T = 1 + x.shape[1] // 256
    B = st["c"].shape[2]
    fi, _ = O.band_indices(sr)
    assert B == len(fi)
    c0_ref = keep["c0"].numpy().reshape(B, T).T
    assert np.abs(st["c0"][0] - c0_ref).max() <= 1e-5 * np.abs(c0_ref).max()
    assert abs(losses[0, 0] - keep["losses"][0]) <= 2e-5
    assert abs(losses[1, 0] - keep["losses"][1]) <= 5e-3
    assert _snr(out[0], y) >= 55


@pytest.mark.parametrize("kind,cutoff", [("lowpass", 4000.0), ("highpass", 500.0), ("bandpass", [500.0, 4000.0])])
def test_fir_attack_matches_scipy_upfirdn(model, kind, cutoff):
    """FIR extension (no reference counterpart): bit-exact against scipy's float32 upfirdn."""
    from scipy.signal import upfirdn
    from aware_b200 import attacks as A
    emb, _ = model
    A.set_engine(emb.engine)
    sr = 44100
    x = _clips([0, 1], 1.0, sr)
    att = A.FIRFilter(kind, cutoff, numtaps=129)
    got = att.apply_batch(torch.from_numpy(x).cuda(), sr).cpu().numpy()
    h = att.taps(sr)
    for i in range(len(x)):
        want = upfirdn(h, x[i], 1, 1)[:x.shape[1]]
        assert want.dtype == np.float32
        np.testing.assert_array_equal(got[i], want)


@pytest.mark.parametrize("numtaps", [1, 5, 8, 64, 101, 1023, 1024, 1500])
def test_register_tiled_fir_equals_scipy_for_every_tap_count_and_window(eng, numtaps):
    """k_fir_tiled (up = down = 1, <= 1024 taps; 1500 takes the generic polyphase kernel): tap counts below,
    at and off the unroll width, clip lengths off the 2048-sample tile, output windows that start inside the
    clip and run past its end (the convolution tail) -- bit-exact against scipy's float32 upfirdn."""
    from scipy.signal import upfirdn
    rng = np.random.default_rng(numtaps)
    h = (rng.standard_normal(numtaps) / np.sqrt(numtaps)).astype(np.float32)
    h_tf = torch.from_numpy(h[::-1].copy()).cuda()
    for n in (1, 7, 2047, 2048, 6151):
        x = rng.standard_normal((3, n)).astype(np.float32)
        xd = torch.from_numpy(x).cuda()
        full = np.stack([upfirdn(h, x[i], 1, 1) for i in range(3)])        # n + numtaps - 1 samples
        assert full.dtype == np.float32
        for first, n_out in ((0, n), (0, n + numtaps - 1), (min(3, n - 1), n + numtaps - 1 - min(3, n - 1)),
                             (n // 2, n - n // 2)):
            got = eng.attack_upfirdn(xd, h_tf, numtaps, 1, 1, first, n_out).cpu().numpy()
            np.testing.assert_array_equal(got, full[:, first:first + n_out], err_msg=str((n, first, n_out)))


def test_service_stereo_equals_two_mono_calls(model):
    """service/embed.py:37-59 and detect.py:23-43 semantics: a stereo clip is two independent mono
    embeds (each rescaled by its own signed max) and the decoder takes, per bit, the channel with
    the larger |v|."""
    from aware_b200.service import detect_watermark, embed_watermark
    emb, det = model
    prev = emb.num_iterations
    emb.num_iterations = 80
    try:
        left, right = O.synth_clip(7, 1.5, 16000), 0.6 * O.synth_clip(8, 1.5, 16000)
        bits = O.synth_bits(8)[7]
        st = embed_watermark(np.column_stack((left, right)), 16000, bits, emb)
        ml, mr = embed_watermark(left, 16000, bits, emb), embed_watermark(right, 16000, bits, emb)
    finally:
        emb.num_iterations = prev
    assert st.shape == (len(ml), 2)
    np.testing.assert_array_equal(st[:, 0], ml)
    np.testing.assert_array_equal(st[:, 1], mr)
    got = detect_watermark(st, 16000, det)
    vl, vr = det.detect(st[:, 0], 16000), det.detect(st[:, 1], 16000)
    want = (np.where(np.abs(vl) > np.abs(vr), vl, vr) > 0).astype(np.int32)
    np.testing.assert_array_equal(got, want)
    np.testing.assert_array_equal(got, bits)
    with pytest.raises(ValueError):
        detect_watermark(st[:, :1], 16000, det)              # (N, 1) is rejected by detect (detect.py:44,55)


def test_degenerate_inputs_stay_finite(eng):
    """All-zero clips, a clip that is silent for most of its length, and a full-scale square wave
    (many samples tie at the peak): detect and embed stay finite, a silent clip stays silent and
    the oracle agrees on the detector outputs."""
    sr = 16000
    n = 2 * sr
    sq = np.sign(np.sin(2 * np.pi * 440.0 * np.arange(n) / sr)).astype(np.float32)
    half = O.synth_clip(9, 2.0, sr).copy()
    half[: n * 3 // 4] = 0.0
    x = np.stack([np.zeros(n, np.float32), half, sq])
    xd = torch.from_numpy(x).cuda()
    eng.set_precision("fp32")
    try:
        v = eng.detect(xd, sr).cpu().numpy()
    finally:
        eng.set_precision("tf32")
    assert np.isfinite(v).all() and np.all(v[0] == 0.0)
    for i in (1, 2):
        assert np.abs(v[i] - O.detect(x[i], sr)).max() <= 2e-5
    pat = torch.from_numpy(np.stack([O.encode_bits(b) for b in O.synth_bits(3)]))
    for prec in ("fp16", "tf32"):
        y = eng.embed(xd, sr, pat, iters=12, precision=prec).cpu().numpy()
        assert np.isfinite(y).all() and np.all(y[0] == 0.0), prec
        assert np.abs(y[1:]).max() <= 1.0


# ------------------------------------------------------------------ round-2 additions
def test_noise_and_gain_attacks_match_their_definition(model):
    """X1 (no reference counterpart, SURVEY 8a): y = fl(gain * x) + fl(sigma * buf) in float32, buf a
    host-seeded standard-normal buffer -- bit-exact against numpy; the detector is scale-invariant
    (WaveformNormalizer), so a pure gain must not change a decoded bit."""
    from aware_b200 import attacks as A
    emb, det = model
    eng = emb.engine
    sr = 44100
    x = _clips([0, 1, 2], 1.0, sr)
    xd = torch.from_numpy(x).cuda()
    for gain in (0.5, 1.7, -1.0):
        got = A.Gain(gain).apply_batch(xd, sr).cpu().numpy()
        np.testing.assert_array_equal(got, np.float32(gain) * x)
    eng.set_precision("fp32")
    try:                                                              # exact GEMMs: only the 1e-8 in x/(max|x|+1e-8) moves
        v0 = eng.detect(xd, sr).cpu().numpy()
        v1 = eng.detect(A.Gain(0.25).apply_batch(xd, sr), sr).cpu().numpy()
    finally:
        eng.set_precision("tf32")
    assert np.abs(v0 - v1).max() <= 1e-5
    for sigma, seed in ((0.01, 99), (0.1, 5)):
        att = A.AdditiveNoise(sigma, seed=seed)
        got = att.apply_batch(xd, sr).cpu().numpy()
        g = torch.Generator(device="cpu").manual_seed(seed)
        buf = torch.randn(xd.shape, generator=g, dtype=torch.float32).numpy()
        np.testing.assert_array_equal(got, np.float32(1.0) * x + np.float32(sigma) * buf)
        assert got.dtype == np.float32 and got.shape == x.shape
        # the caller's own buffer, already resident in HBM (wider than the clips: row stride != n)
        wide = torch.zeros((x.shape[0], x.shape[1] + 7), dtype=torch.float32)
        wide[:, :x.shape[1]] = torch.from_numpy(buf)
        got2 = A.AdditiveNoise(sigma, buffer=wide.cuda()).apply_batch(xd, sr).cpu().numpy()
        np.testing.assert_array_equal(got2, got)
    with pytest.raises(ValueError):
        A.AdditiveNoise(0.01, buffer=torch.zeros((1, 8))).apply_batch(xd, sr)
    one = A.AdditiveNoise(0.01).apply(x[0], sr)                       # reference calling convention
    assert one.shape == x[0].shape and one.dtype == np.float32


def test_signed_max_scale_on_device_equals_host_scale(eng):
    """service/embed.py:69,73 rescales by the SIGNED np.max(audio); scale='signed_max' takes it on the
    device in the pass that finds the peak.  Bit-identical to passing the host-computed scale, also for
    a clip whose largest |x| is negative and for an all-negative clip."""
    sr = 16000
    x = _clips([0, 1, 2], 1.0, sr)
    x[1] = -np.abs(x[1]) - 0.01                                       # all negative: max < 0
    x[2][100] = -0.95                                                 # peak |x| is a negative sample
    xd = torch.from_numpy(x).cuda()
    pat = torch.from_numpy(np.stack([O.encode_bits(b) for b in O.synth_bits(3)]))
    a = eng.embed(xd, sr, pat, iters=4, scale=xd.max(dim=1).values)
    b = eng.embed(xd, sr, pat, iters=4, scale="signed_max")
    assert torch.equal(a, b)
    assert (b[1].abs().max() > 0) and float(b[1][b[1].abs().argmax()]) * float(xd[1].max()) != 0.0
    assert int(eng.embed_status().sum()) == 0                          # no non-finite gradient was skipped


def test_embed_one_iteration_on_a_clipped_clip_with_tied_peaks(eng):
    """Peak ties (SURVEY A.7): a hard-clipped clip has hundreds of samples at exactly +-peak.  torch.max
    splits the normaliser's sub-gradient evenly across exact ties; after the STFT -> iSTFT round trip
    the re-synthesised y only has near-ties (rounding noise ~1e-7), so reference and kernel each pick
    ONE arg-max sample -- possibly different ones.  One step against the oracle shows that the rank-one
    term this moves is far below the gate: coefficients and waveform agree as on ordinary clips."""
    sr = 16000
    x = np.clip(1.6 * _clips([4], 1.0, sr), -0.8, 0.8).astype(np.float32)
    assert (np.abs(x[0]) == 0.8).sum() > 50
    pat = np.stack([O.encode_bits(O.synth_bits(8)[4])])
    out, losses, st = _embed_state(eng, x, sr, pat, 1, "fp32")
    keep = {}
    y = O.embed(x[0], sr, pat[0], num_iters=1, keep=keep)
    T = 1 + x.shape[1] // 256
    B = st["c"].shape[2]
    c_ref = keep["coeffs_after"][1].numpy().reshape(B, T).T
    g_ref = keep["grads"][0].numpy().reshape(B, T).T
    assert abs(losses[0, 0] - keep["losses"][0]) <= 1e-5
    g_gpu = st["m"][0] / 0.1
    rms = lambda a: float(np.sqrt(np.mean(a ** 2)))                   # noqa: E731
    print("tied-peak clip: gradient rel. RMS diff %.2e" % (rms(g_gpu - g_ref) / rms(g_ref)))
    assert rms(g_gpu - g_ref) <= 2e-3 * rms(g_ref)                    # as on ordinary clips (1e-3 outside kink frames)
    d = np.abs(st["c"][0] - c_ref)
    assert (d <= 1e-4 * np.maximum(1.0, np.abs(c_ref))).mean() >= 0.99
    # Waveform: the ~1 % of coefficients whose gradient is within rounding of 0 step the other way
    # (2 lr = 0.2 each, 4e-4 over the 1024 samples they overlap); a clipped clip has a broad spread of
    # gradient magnitudes, so more of them than an ordinary clip.  The output is also y / max|y| with the
    # maximum taken over hundreds of near-tied samples, which moves ONE global scalar (reported, removed).
    alpha = float(np.dot(out[0].astype(np.float64), y) / np.dot(y.astype(np.float64), y))
    print("tied-peak clip: peak-normaliser scalar differs by %.2e" % (alpha - 1.0))
    assert abs(alpha - 1.0) <= 3e-4
    d = np.abs(out[0] / alpha - y)
    print("tied-peak clip: %.2f %% of samples within 1e-4, max %.2e, SNR %.1f dB" % (
        100 * (d <= 1e-4).mean(), d.max(), _snr(out[0] / alpha, y)))
    assert (d <= 1e-4).mean() >= 0.90 and d.max() <= 2e-3 and _snr(out[0] / alpha, y) >= 70


def test_detector_threshold_reaches_the_batch_decision(model):
    """The engine is shared by embedder and detector; the detector's own threshold must be the one the
    batched bit decision uses (it used to be captured once at engine creation)."""
    from aware_b200.service import detect_watermark, detect_watermark_batch
    emb, det = model
    sr = 16000
    x = _clips([0, 1], 1.0, sr)
    prev = det.threshold
    try:
        for thr in (0.0, 0.02, -0.03):
            det.threshold = thr
            got = detect_watermark_batch(x, sr, det).cpu().numpy()
            want = np.stack([detect_watermark(x[i], sr, det) for i in range(2)])
            np.testing.assert_array_equal(got, want)
            v = det.detect_batch(x, sr).cpu().numpy()
            np.testing.assert_array_equal(got, (v > thr).astype(np.int32))
    finally:
        det.threshold = prev
        emb.engine.set_threshold(prev)


def test_compression_approx_matches_its_numpy_definition(model):
    """X3 (parity unpinned to the reference -- upstream's MP3 attack is an ffmpeg call; pinned to the
    definition restated in numpy, oracle/aware_oracle.py::attack_compression_approx).  The quantised
    magnitudes agree except where log2 lands within rounding of a grid midpoint (device log2f vs numpy),
    the waveform to 1e-4 / 80 dB, and a watermark survives the attack."""
    from aware_b200 import attacks as A
    emb, det = model
    eng = emb.engine
    sr = 44100
    x = _clips([1, 2], 1.5, sr)
    xd = torch.from_numpy(x).cuda()
    att = A.CompressionApprox(step_db=1.5, floor_db=-30.0)
    got = att.apply_batch(xd, sr).cpu().numpy()
    mag = eng.stft_band(xd, sr, normalize=False).cpu().numpy()
    dq = eng.spectral_quantize(torch.from_numpy(mag).cuda(), 1.5, -30.0).cpu().numpy()
    for i in range(2):
        want, mag_ref, q_ref = O.attack_compression_approx(x[i], sr, 1.5, -30.0)
        assert got[i].shape == want.shape == (256 * (x.shape[1] // 256),)
        assert np.abs(mag[i] - mag_ref).max() <= 1e-5 * mag_ref.max()
        q = dq[i] + mag[i]
        same = np.abs(q - q_ref) <= 1e-4 * np.maximum(q_ref, 1e-3)
        assert same.mean() >= 0.999, same.mean()               # grid-midpoint / masking-floor ties only
        assert (q[q_ref == 0][same[q_ref == 0]] == 0).all()
        d = np.abs(got[i] - want)
        assert (d <= 1e-4).mean() >= 0.995 and _snr(got[i], want) >= 60
        assert _snr(got[i], x[i][:len(want)]) < 60                 # it does change the audio
    # robustness is not a parity matter: BER after the default and a harsher setting is reported only
    from aware_b200.service import detect_watermark_batch, embed_watermark_batch
    emb.num_iterations, prev = 150, emb.num_iterations
    emb.enforce_16k = det.enforce_16k = False
    try:
        bits = O.synth_bits(2)
        y = embed_watermark_batch(x, sr, bits, emb)
        for a_ in (A.CompressionApprox(), att):
            dec = detect_watermark_batch(a_.apply_batch(y, sr), sr, det).cpu().numpy()
            print("%s (floor %g dB): BER %.1f %%" % (a_.name, a_.floor_db, 100 * (dec != bits).mean()))
            assert dec.shape == bits.shape
    finally:
        emb.num_iterations = prev
        emb.enforce_16k = det.enforce_16k = True


@pytest.mark.parametrize("precision", ["tf32", "fp16"])
def test_two_pass_small_k_layers_match_the_one_pass_form(eng, precision):
    """The K <= 128 layers run as a statistics pass + an apply pass (the raw H1 / dHhat3 never reach HBM).
    Same GEMM, same column sums; the apply pass normalises the fp32 accumulator instead of the stored
    (fp16 / TF32-rounded) value, so it can only be closer to the oracle: detector outputs and the first
    losses agree with the one-pass form at storage-rounding level, and with the oracle as before."""
    sr = 44100
    x = _clips([0, 1, 2], 1.5, sr)
    xd = torch.from_numpy(x).cuda()
    pat = torch.from_numpy(np.stack([O.encode_bits(b) for b in O.synth_bits(3)]))
    eng.set_precision(precision)
    eng.set_exact_margin(0.0)
    try:
        out = {}
        for two in (False, True):
            eng.set_two_pass(two)
            v = eng.detect(xd, sr).cpu().numpy()
            _, _, losses = eng.embed(xd, sr, pat, iters=3, return_losses=True, precision=precision)
            out[two] = (v, losses[:3].cpu().numpy())
    finally:
        eng.set_two_pass(True)
        eng.set_precision("tf32")
        eng.set_exact_margin(1e-3)
    ref = np.stack([O.detect(x[i], sr) for i in range(3)])
    tol = 1e-3
    assert np.abs(out[True][0] - out[False][0]).max() <= tol
    assert np.abs(out[True][0] - ref).max() <= tol
    assert np.abs(out[True][1] - out[False][1]).max() <= 5e-3


@pytest.mark.parametrize("precision", ["tf32", "fp16", "bf16"])
def test_cta_pair_gemm_is_bit_identical_to_the_one_cta_kernel(eng, precision):
    """The K >= 512 layers on CTA pairs (tcgen05 cta_group::2, M = 256, each CTA staging half of the weight
    tile): the same products accumulated in the same k order per output element, so detector values, the
    watermarked clips of a short embed and its losses are IDENTICAL to the one-CTA kernel's; with an odd number
    of 128-row tiles the library falls back to the one-CTA kernel by itself."""
    sr = 44100
    x = _clips([0, 1, 2, 3], 1.5, sr)
    xd = torch.from_numpy(x).cuda()
    pat = torch.from_numpy(np.stack([O.encode_bits(b) for b in O.synth_bits(4)]))
    eng.set_precision(precision)
    eng.set_exact_margin(0.0)
    try:
        out = {}
        for pair in (False, True):
            eng.set_pair_gemm(pair)
            n0 = eng.launch_count()
            v = eng.detect(xd, sr).cpu().numpy()
            y, _, losses = eng.embed(xd, sr, pat, iters=3, return_losses=True, precision=precision)
            v3 = eng.detect(xd[:3], sr).cpu().numpy()       # 21 row tiles: odd -> one-CTA kernel either way
            out[pair] = (v, y.cpu().numpy(), losses[:3].cpu().numpy(), v3, eng.launch_count() - n0)
    finally:
        eng.set_pair_gemm(True)
        eng.set_precision("tf32")
        eng.set_exact_margin(1e-3)
    for a, b in zip(out[True][:4], out[False][:4]):
        assert np.array_equal(a, b)
    assert out[True][4] == out[False][4]
    ref = np.stack([O.detect(x[i], sr) for i in range(4)])
    assert np.abs(out[True][0] - ref).max() <= (1e-3 if precision == "tf32" else 3e-2)


def test_run_suite_side_stream_equals_one_stream(model):
    """attacks.run_suite launches the sequential (bit-exact) IIR attacks on a side stream and consumes them
    last; every attacked batch must equal the one-stream result bit for bit, in the suite's own index order,
    also when the next call reuses the scratch the filtfilt parks in the gradient buffers."""
    from aware_b200 import attacks as A
    emb, det = model
    eng = emb.engine
    sr = 16000
    y = torch.from_numpy(_clips([0, 1, 2, 3, 4], 1.5, sr)).cuda()
    suite = [A.PCMBitDepthConversion(16), A.RandomBandstop(f_low=1000.0, fast=False), A.SampleSupression(0.1, start=100),
             A.LowPassFilter(fast=False), A.HighPassFilter(fast=True), A.RandomBandstop(f_low=333.0, fast=False)]
    assert [getattr(a, "sequential", False) for a in suite] == [False, True, False, True, False, True]
    want = [a.apply_batch(y, sr, engine=eng).clone() for a in suite]
    for _ in range(2):
        got, vals = {}, {}

        def consume(i, z):
            got[i] = z.clone()
            vals[i] = eng.detect(z, sr)
        A.run_suite(suite, y, sr, consume, engine=eng)
        torch.cuda.synchronize()
        assert sorted(got) == list(range(len(suite)))
        for i in range(len(suite)):
            assert torch.equal(got[i], want[i]), suite[i].name
            assert torch.equal(vals[i], eng.detect(want[i], sr)), suite[i].name
    eng.profile(True)                                      # profiling keeps everything on one stream
    try:
        order = []
        A.run_suite(suite, y, sr, lambda i, z: order.append(i), engine=eng)
    finally:
        eng.profile(False)
        eng.profile_read()
        eng.profile_read_named()
    assert order == list(range(len(suite)))


def test_stoi_kernels_match_the_numpy_restatement(model):
    """f4 (SURVEY 8f-4): GPU STOI (aw_stoi_batch) against oracle/stoi_oracle.py -- pystoi's algorithm restated
    (the package is absent: parity unpinned to pystoi itself).  Tolerance 1e-4 absolute on the score (float32
    resampling / DFT on the device, float64 in the restatement); covers a silence gap (frames removed by the
    40 dB gate), noise levels from inaudible to destructive, the 10 kHz no-resample path, a clip that is too
    short (1e-5 as pystoi answers), the reference metric's call signature, and the > 0.1 running sums of
    scripts/test.py:86-88."""
    import stoi_oracle as S
    from aware_b200.metrics import STOI
    emb, det = model
    eng = emb.engine
    sr = 16000
    x = _clips([0, 1, 2, 3], 3.0, sr)
    x[1, 8000:20000] *= 1e-4                                           # a gap the silence gate removes
    rng = np.random.default_rng(5)
    noise = rng.standard_normal(x.shape).astype(np.float32)
    y = x + np.array([1e-3, 1e-2, 5e-2, 0.5], dtype=np.float32)[:, None] * noise
    want = np.array([S.stoi(x[i].astype(np.float64), y[i].astype(np.float64), sr) for i in range(4)])
    sums = torch.zeros(2, dtype=torch.float64, device="cuda")
    got = eng.stoi(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), sr, stoi_sum=sums).cpu().numpy()
    print("STOI gpu", got, "oracle", want)
    assert np.abs(got - want).max() <= 1e-4
    keep = want > 0.1
    s = sums.cpu().numpy()
    assert s[1] == keep.sum() and abs(s[0] - got[got > 0.1].sum()) < 1e-9
    assert abs(eng.stoi(torch.from_numpy(x).cuda(), torch.from_numpy(x).cuda(), sr).cpu().numpy() - 1.0).max() < 1e-5
    # already at pystoi's 10 kHz: no resampling
    x10 = _clips([4, 5], 2.0, 10000)
    y10 = x10 + 0.02 * rng.standard_normal(x10.shape).astype(np.float32)
    w10 = np.array([S.stoi(x10[i].astype(np.float64), y10[i].astype(np.float64), 10000) for i in range(2)])
    g10 = eng.stoi(torch.from_numpy(x10).cuda(), torch.from_numpy(y10).cuda(), 10000).cpu().numpy()
    assert np.abs(g10 - w10).max() <= 1e-4
    # too short for 30 frames
    short = eng.stoi(torch.from_numpy(x[:, :4000].copy()).cuda(), torch.from_numpy(y[:, :4000].copy()).cuda(), sr)
    assert np.all(short.cpu().numpy() == 1e-5)
    # reference call signature: STOI()(output, target, sampling_rate) -> float, truncation to the shorter input
    m = STOI(eng)
    one = m(y[2], x[2][:-100], sr)
    assert abs(one - S.stoi(x[2][:-100].astype(np.float64), y[2][:-100].astype(np.float64), sr)) <= 1e-4


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
def test_streaming_k64_backward_kernel_matches_the_generic_epilogues(eng, precision):
    """csrc/gemm64.cuh: the backward K = 64 layer with its activation tiles streamed through a TMA ring and the
    output written by a TMA bulk store, against the generic GEMM's statistics / apply epilogues: the same
    products, statistics and adjoint formula -- only the order in which the 128 rows of a tile are summed into
    the column sums differs (float32 rounding).  Compared on the first-moment estimate after ONE step (m = 0.1 g:
    the gradient itself, before NAdam's sign-like normalisation amplifies rounding), on clips whose pooled length
    is not a multiple of 128 (pad rows must come out zero), and on the losses of three iterations."""
    sr = 44100
    for secs in (1.5, 3.1):
        x = _clips([0, 1, 2], secs, sr)
        xd = torch.from_numpy(x).cuda()
        pat = torch.from_numpy(np.stack([O.encode_bits(b) for b in O.synth_bits(3)]))
        T = 1 + x.shape[1] // 256
        out = {}
        try:
            for on in (False, True):
                eng.set_bwd64_stream(on)
                eng.embed(xd, sr, pat, iters=1, precision=precision)
                m = eng.embed_state("m", 3, T, sr).cpu().numpy()
                _, _, losses = eng.embed(xd, sr, pat, iters=3, return_losses=True, precision=precision)
                out[on] = (m, losses[:3].cpu().numpy())
        finally:
            eng.set_bwd64_stream(True)
        m0, m1 = out[False][0], out[True][0]
        assert np.isfinite(m1).all() and np.abs(m1).max() > 0
        scale = np.abs(m0).max(axis=(1, 2), keepdims=True)
        err = np.abs(m1 - m0) / scale
        print("k64 streaming vs generic (%s, %.1f s): max rel err %.2e, rms %.2e" %
              (precision, secs, err.max(), np.sqrt((err ** 2).mean())))
        assert err.max() <= (2e-3 if precision == "fp16" else 2e-2)
        assert np.sqrt((err ** 2).mean()) <= (1e-4 if precision == "fp16" else 1e-3)
        assert np.abs(out[True][1] - out[False][1]).max() <= 5e-3

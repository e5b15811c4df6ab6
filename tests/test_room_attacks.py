"""Reverberation and echo attacks (aware_b200.attacks.Reverb / Echo) and the partitioned convolution behind
them (Engine.attack_convolve, aw_attack_convolve).

The attacks have no upstream counterpart; they are defined as a causal convolution truncated to the input's
length (DESIGN.md section 7) and pinned to the float64 restatement in tests/room_oracle.py.  The CPU tests
pin the restatement's block bookkeeping and the host-side helpers; the GPU tests pin the CUDA path to the
float64 convolution and to the existing float32 direct-form FIR kernel."""
import ctypes

import numpy as np
import pytest
import torch

import aware_oracle as O
import room_oracle as RO
from aware_b200 import attacks as A

TAPS = [1, 511, 512, 513, 4800, 30870]
SIZES = [(16000, 36800), (44100, 74970)]       # 2.3 s and 1.7 s: neither a multiple of 512
GPU_TAPS = [1, 512, 513, 4800, 30870]


def _taps(M, seed):
    g = np.random.default_rng(seed)
    h = g.standard_normal(M) * np.exp(-3.0 * np.arange(M) / max(M, 1))
    return (h / np.linalg.norm(h)).astype(np.float32)


def _err(got, ref):
    """(max |got - ref| / max |ref|, SNR in dB) in float64."""
    d = got.astype(np.float64) - ref
    rel = np.abs(d).max() / np.abs(ref).max()
    snr = 10 * np.log10(np.sum(ref ** 2) / max(np.sum(d ** 2), 1e-300))
    return rel, snr


# ---------------------------------------------------------------- CPU: the restatement and host helpers
@pytest.mark.parametrize("M", TAPS)
@pytest.mark.parametrize("N", [300, 5000, 20000])
def test_partitioned_restatement_equals_direct_convolution(N, M):
    g = np.random.default_rng(N + M)
    x = g.standard_normal(N)
    h = _taps(M, M)
    ref = np.convolve(x.astype(np.float64), h.astype(np.float64))[:N]
    got = RO.partitioned_convolve(x, h)
    assert got.shape == (N,)
    assert np.abs(got - ref).max() <= 1e-12 * np.abs(ref).max()


@pytest.mark.parametrize("M", TAPS)
def test_conv_spectra_are_the_partition_rffts(M):
    h = np.stack([_taps(M, 1), _taps(M, 2)])
    spec = A.conv_spectra(h)
    K = -(-M // 512)
    assert spec.shape == (2, K, 513) and spec.dtype == np.complex64
    for r in range(2):
        for j in range(K):
            part = np.zeros(1024)
            seg = h[r, 512 * j:512 * j + 512].astype(np.float64)
            part[:len(seg)] = seg
            np.testing.assert_array_equal(spec[r, j], np.fft.rfft(part).astype(np.complex64))
    np.testing.assert_array_equal(A.conv_spectra(h[0]), spec[:1])


@pytest.mark.parametrize("sr", [16000, 44100])
@pytest.mark.parametrize("rt60", [0.3, 0.7, 1.2])
def test_synthetic_rir_length_energy_determinism_and_decay(sr, rt60):
    h = A.synthetic_rir(rt60, sr, 5)
    assert h.dtype == np.float32 and h.shape == (round(rt60 * sr),)
    np.testing.assert_array_equal(h, RO.synth_rir(rt60, sr, 5))
    np.testing.assert_array_equal(h, A.synthetic_rir(rt60, sr, 5))
    assert not np.array_equal(h, A.synthetic_rir(rt60, sr, 6))
    assert abs(np.sum(h.astype(np.float64) ** 2) - 1.0) <= 1e-6
    assert h[0] > 0                                       # the direct path, 1 before normalisation
    # energy per 10 ms window (the direct path's window excluded), in dB, fitted by a line over the first
    # 80 % of the response: -60 dB per rt60 within 2 dB
    w = int(0.01 * sr)
    n_win = int(0.8 * len(h)) // w
    e = (h[:n_win * w].astype(np.float64) ** 2).reshape(n_win, w).sum(axis=1)[1:]
    t = (np.arange(1, n_win) + 0.5) * w / sr
    slope = np.polyfit(t, 10 * np.log10(e), 1)[0]
    assert abs(slope * rt60 + 60.0) <= 2.0, slope * rt60


def test_reverb_responses_and_room_attack_names():
    r = A.Reverb(0.3, n_rirs=3, seed=4)
    resp = r.responses(16000)
    assert resp.shape == (3, 4800) and resp.dtype == np.float32
    for k in range(3):
        np.testing.assert_array_equal(resp[k], RO.synth_rir(0.3, 16000, 4 + k))
    own = np.stack([_taps(700, 1), _taps(700, 2)])
    np.testing.assert_array_equal(A.Reverb(rir=own).responses(44100), own)
    np.testing.assert_array_equal(A.Reverb(rir=own[0]).responses(16000), own[:1])
    assert [a.name for a in A.room_attacks()] == ["reverb_0.3", "reverb_0.7", "echo_0.05_0.5"]
    assert not any(getattr(a, "sequential", False) for a in A.room_attacks())


def test_echo_response_layout():
    h = A.Echo(0.05, 0.5).responses(16000)
    assert h.shape == (1, 801) and h.dtype == np.float32
    assert h[0, 0] == 1.0 and h[0, 800] == 0.5 and not h[0, 1:800].any()
    np.testing.assert_array_equal(h[0], RO.echo_response(0.05, 0.5, 16000))
    assert A.Echo(0.05, -0.3).responses(44100).shape == (1, 2206)


class _NoEngine:
    """Stands in for the engine: any library call fails the test."""
    device = torch.device("cpu")

    def attack_convolve(self, *a, **k):
        raise AssertionError("the library was called")


@pytest.mark.parametrize("make", [
    lambda: A.Reverb(0.0), lambda: A.Reverb(-0.5), lambda: A.Reverb(float("nan")), lambda: A.Reverb(float("inf")),
    lambda: A.Reverb(0.3, n_rirs=0),
    lambda: A.Reverb(rir=np.zeros((1, 1, 4))), lambda: A.Reverb(rir=np.zeros((1, 0))),
    lambda: A.Reverb(rir=np.zeros(262145)), lambda: A.Reverb(rir=np.array([1.0, np.nan])),
    lambda: A.Reverb(0.3, n_rirs=3, index=3), lambda: A.Reverb(0.3, n_rirs=3, index=[0, -1]),
    lambda: A.Reverb(0.3, n_rirs=3, index=[0.5]), lambda: A.Reverb(0.3, n_rirs=3, index=[]),
    lambda: A.Echo(0.0, 0.5), lambda: A.Echo(float("nan"), 0.5), lambda: A.Echo(0.05, float("inf")),
    lambda: A.Reverb(0.3, rir=np.ones(10)), lambda: A.Reverb(),
])
def test_bad_parameters_raise_at_construction(make):
    with pytest.raises(ValueError):
        make()


@pytest.mark.parametrize("att,sr,n_clips", [
    (A.Reverb(6.0), 44100, 1),                            # 264 600 taps
    (A.Reverb(1e-5), 16000, 1),                           # 0 taps
    (A.Echo(6.0, 0.5), 44100, 1),                         # D + 1 > 262 144
    (A.Echo(1e-5, 0.5), 16000, 1),                        # D = 0
    (A.Reverb(0.1, n_rirs=3, index=[0, 1]), 16000, 3),    # one index per clip, or one for all
])
def test_bad_sizes_raise_before_any_library_call(att, sr, n_clips):
    with pytest.raises(ValueError):
        att.apply_batch(torch.zeros((n_clips, 1000)), sr, engine=_NoEngine())


def test_convolve_symbol_is_exported():
    from aware_b200 import _lib
    assert "aw_attack_convolve" in _lib.SIGNATURES
    assert getattr(_lib.lib(), "aw_attack_convolve") is not None


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def model():
    from aware_b200.utils.models import load
    emb, det = load()
    emb.verbose = False
    A.set_engine(emb.engine)
    return emb, det


def _clips(n_clips, N, seed):
    g = np.random.default_rng(seed)
    x = g.standard_normal((n_clips, N)).astype(np.float32) * 0.3
    x[:, :N // 3] *= 0.01                                  # a quiet stretch: the error bound is relative to max|y|
    return x


def _convolve(eng, x, h):
    spec = torch.from_numpy(A.conv_spectra(h)).cuda()
    return eng.attack_convolve(torch.from_numpy(x).cuda(), spec).cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("sr,N", SIZES)
def test_convolve_matches_the_float64_convolution(model, sr, N):
    """Measured on a B200: at most 3.6e-7 of max|y| and at least 129.7 dB (printed); the bounds leave about
    3x room over the error and 5 dB over the SNR."""
    eng = model[0].engine
    x = _clips(2, N, sr)
    cases = [("taps_%d" % M, _taps(M, M)) for M in GPU_TAPS]
    cases += [(a.name, a.responses(sr)[0]) for a in (A.Reverb(0.3, seed=1), A.Reverb(0.7, seed=2), A.Echo(0.05, 0.5))]
    for name, h in cases:
        got = _convolve(eng, x, h)
        assert got.shape == x.shape and got.dtype == np.float32
        for i in range(2):
            rel, snr = _err(got[i], RO.convolve(x[i], h))
            print("%s @ %d Hz (N %d, M %d) clip %d: max err %.2e of max|y|, SNR %.1f dB" % (name, sr, N, len(h), i,
                                                                                         rel, snr))
            assert rel <= 1e-6 and snr >= 125.0, (name, rel, snr)


@pytest.mark.gpu
@pytest.mark.parametrize("sr,N", SIZES)
def test_convolve_agrees_with_the_direct_form_fir(model, sr, N):
    eng = model[0].engine
    x = _clips(3, N, sr + 1)
    xd = torch.from_numpy(x).cuda()
    for M in [m for m in GPU_TAPS if m <= 4800]:
        h = _taps(M, M + 7) if M != 4800 else A.synthetic_rir(0.3, 16000, 3)
        got = _convolve(eng, x, h)
        direct = eng.attack_upfirdn(xd, torch.from_numpy(h[::-1].copy()).cuda(), M, 1, 1, 0, N).cpu().numpy()
        for i in range(3):
            rel, snr = _err(got[i], direct[i].astype(np.float64))
            print("M %d @ %d Hz clip %d: convolution vs direct form %.2e of max|y|, SNR %.1f dB" % (M, sr, i, rel, snr))
            assert rel <= 5e-6 and snr >= 115.0, (M, rel, snr)


@pytest.mark.gpu
def test_each_clip_is_convolved_with_its_own_response(model):
    eng = model[0].engine
    sr, N = 16000, 36800
    x = _clips(5, N, 11)
    att = A.Reverb(0.3, n_rirs=3, seed=20, index=[2, 0, 1, 2, 0])
    got = att.apply_batch(torch.from_numpy(x).cuda(), sr).cpu().numpy()
    resp = att.responses(sr)
    spec = att._spectra[(sr, eng.device.index)]
    for i, k in enumerate([2, 0, 1, 2, 0]):
        rel, snr = _err(got[i], RO.convolve(x[i], resp[k]))
        assert rel <= 1e-6 and snr >= 125.0
        alone = eng.attack_convolve(torch.from_numpy(x[i:i + 1]).cuda(), spec, [k]).cpu().numpy()
        np.testing.assert_array_equal(got[i], alone[0])
    # drawn indices follow rng.integers(0, R, n_clips)
    drawn = A.Reverb(0.3, n_rirs=3, seed=20).apply_batch(torch.from_numpy(x).cuda(), sr,
                                                          rng=np.random.default_rng(9)).cpu().numpy()
    idx = np.random.default_rng(9).integers(0, 3, 5)
    fixed = A.Reverb(0.3, n_rirs=3, seed=20, index=idx).apply_batch(torch.from_numpy(x).cuda(), sr).cpu().numpy()
    np.testing.assert_array_equal(drawn, fixed)


@pytest.mark.gpu
def test_bit_identity_strides_and_silence(model):
    eng = model[0].engine
    sr, N = 44100, 74970
    x = _clips(6, N, 3)
    x[4] = 0.0
    wide = torch.zeros((6, N + 77), device="cuda")
    wide[:, 13:13 + N] = torch.from_numpy(x).cuda()
    xs = wide[:, 13:13 + N]                                   # row stride N + 77, unaligned rows
    for att in A.room_attacks():
        batch = att.apply_batch(xs, sr, rng=np.random.default_rng(1)).cpu().numpy()
        again = att.apply_batch(xs, sr, rng=np.random.default_rng(1)).cpu().numpy()
        np.testing.assert_array_equal(batch, again)
        idx = np.random.default_rng(1).integers(0, 8, 6) if isinstance(att, A.Reverb) else [0] * 6
        spec = att._spectra[(sr, eng.device.index)]
        alone = eng.attack_convolve(torch.from_numpy(x[2:3]).cuda(), spec, [int(idx[2])]).cpu().numpy()
        np.testing.assert_array_equal(batch[2], alone[0])
        assert np.isfinite(batch).all() and (batch[4] == 0).all()
    # strided output rows, written in place through the C entry
    spec = torch.view_as_real(torch.from_numpy(A.conv_spectra(_taps(4800, 1))).cuda())
    out = torch.full((6, N + 50), 7.0, device="cuda")
    from aware_b200 import _lib
    _lib.check(eng.lib.aw_attack_convolve(eng._ctx, xs.data_ptr(), 6, N, xs.stride(0), spec.data_ptr(), 1,
                                          spec.shape[1], None, out.data_ptr(), out.stride(0), None))
    torch.cuda.synchronize()
    ref = eng.attack_convolve(xs, torch.view_as_complex(spec))
    np.testing.assert_array_equal(out[:, :N].cpu().numpy(), ref.cpu().numpy())
    assert (out[:, N:] == 7.0).all()


@pytest.mark.gpu
def test_c_entry_validates_its_arguments(model):
    eng = model[0].engine
    x = torch.zeros((2, 4000), device="cuda")
    spec = torch.view_as_real(torch.from_numpy(A.conv_spectra(np.stack([_taps(600, 1), _taps(600, 2)]))).cuda())
    out = torch.empty((2, 4000), device="cuda")

    def call(n=4000, in_stride=4000, n_filters=2, n_parts=2, idx=None, out_stride=4000):
        p = None if idx is None else (ctypes.c_int32 * len(idx))(*idx)
        return eng.lib.aw_attack_convolve(eng._ctx, x.data_ptr(), 2, n, in_stride, spec.data_ptr(), n_filters,
                                          n_parts, p, out.data_ptr(), out_stride, None)

    assert call(idx=[0, 1]) == 0
    for kw, msg in ((dict(idx=[0, 2]), b"filter_of_clip"), (dict(idx=[-1, 0]), b"filter_of_clip"),
                    (dict(n_parts=0), b"n_parts"), (dict(n_parts=513), b"n_parts"),
                    (dict(in_stride=3999), b"stride"), (dict(out_stride=100), b"stride"), (dict(n=0), b"n must"),
                    (dict(n_filters=0), b"n_filters"),
                    (dict(n=2 ** 31 - 2047, in_stride=2 ** 31, out_stride=2 ** 31), b"n must")):
        assert call(**kw) != 0, kw
        assert msg in eng.lib.aw_last_error(), (kw, eng.lib.aw_last_error())
    with pytest.raises(ValueError):
        eng.attack_convolve(x, torch.view_as_complex(spec), [0, 5])
    with pytest.raises(ValueError):
        eng.attack_convolve(x, torch.view_as_complex(spec)[:, :, :512])
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_room_robustness_is_reported(model):
    """BER after embedding at 16 kHz with the default iteration count under each room attack: reported, not
    gated."""
    from aware_b200.service import detect_watermark_batch, embed_watermark_batch
    emb, det = model
    sr = 16000
    x = np.stack([O.synth_clip(i, 2.0, sr) for i in (1, 2)])
    bits = O.synth_bits(2)
    y = embed_watermark_batch(x, sr, bits, emb)
    for att in A.room_attacks():
        z = att.apply_batch(y, sr, rng=np.random.default_rng(0))
        dec = detect_watermark_batch(z, sr, det).cpu().numpy()
        print("%s (%d iterations): BER %.1f %%" % (att.name, emb.num_iterations, 100 * (dec != bits).mean()))


@pytest.mark.gpu
def test_evaluation_driver_appends_the_room_attacks_on_request(model):
    from aware_b200.evaluate import default_attacks, evaluate_clips
    emb, det = model
    clips = [O.synth_clip(0, 2.0, 16000), O.synth_clip(1, 1.5, 16000), O.synth_clip(2, 1.2, 44100)]
    rates = [16000, 16000, 44100]
    defaults = ["orig"] + [a.name for a in default_attacks(np.random.default_rng(0))]
    prev = emb.num_iterations
    emb.num_iterations = 20
    try:
        plain = evaluate_clips(clips, rates, emb, det, seed=3)
        extra = evaluate_clips(clips, rates, emb, det, seed=3, room=True)
    finally:
        emb.num_iterations = prev
    assert list(plain["ber_percent"]) == defaults
    assert list(extra["ber_percent"]) == defaults + [a.name for a in A.room_attacks()]
    # the room attacks draw from their own generator: every default attack's result is unchanged, over
    # three length buckets whose random parameters come from the one shared generator
    assert {k: extra["ber_percent"][k] for k in defaults} == plain["ber_percent"]
    assert extra["snr_db_mean"] == pytest.approx(plain["snr_db_mean"], rel=1e-12)
    assert all(0.0 <= v <= 100.0 for v in extra["ber_percent"].values())
    print({k: round(v, 1) for k, v in extra["ber_percent"].items() if k not in defaults})

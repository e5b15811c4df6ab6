"""Host-side logic of aware_b200 that needs no GPU: the reference-shaped API
objects, codec/metrics, attack planning, and that the C-ABI library loads and
exports every declared symbol."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

import aware_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from aware_b200 import _lib
    header = open(os.path.join(ROOT, "include", "aware_b200.h")).read()
    declared = set(re.findall(r"\b(aw_[a-z0-9_]+)\s*\(", header))
    declared -= {"aw_ctx", "aw_model"}
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    handle = _lib.lib()                      # raises AttributeError on a missing export
    for name in declared:
        assert getattr(handle, name) is not None
    assert b"sm_100a" in handle.aw_version()


def test_python_constants_equal_the_header_enums():
    """Every AW_PREC_* / AW_OPT_* / AW_STAT_* / AW_COMM_* enumerator of include/aware_b200.h has the same value
    on the ctypes side (aware_b200/_lib.py) -- a knob added to one and not the other would silently set another."""
    from aware_b200 import _lib
    header = open(os.path.join(ROOT, "include", "aware_b200.h")).read()
    enums = {m.group(1): int(m.group(2)) for m in re.finditer(r"\bAW_((?:PREC|OPT|STAT|COMM)_[A-Z0-9_]+)\s*=\s*(\d+)", header)}
    assert len(enums) >= 16 and "OPT_BWD64_STREAM" in enums
    for name, value in enums.items():
        assert getattr(_lib, name) == value, name
    # multiply-shift division used by the frame-row kernels (csrc/spectc.cuh: e / nb == (e * magic) >> 32)
    for nb in (1, 2, 40, 81, 96, 225, 256):
        magic = 0xFFFFFFFF // nb + 1
        e = np.arange(0, 1 << 16, dtype=np.uint64)
        assert np.array_equal((e * np.uint64(magic)) >> np.uint64(32), e // np.uint64(nb))


def test_context_creation_fails_loudly_without_gpu():
    if torch.cuda.is_available():
        # CUDA is initialised in this process: rerun the test in a child that sees no device
        out = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider",
                              __file__ + "::test_context_creation_fails_loudly_without_gpu"],
                             env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), cwd=ROOT,
                             capture_output=True, text=True, timeout=600)
        assert out.returncode == 0 and "1 passed" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]
        return
    from aware_b200.engine import Engine
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        Engine(O.make_weights(), O.mel_basis(), O.hann().numpy())
    # and at the C level
    from aware_b200 import _lib
    ctx = ctypes.c_void_p()
    m = _lib.AwModel()
    assert _lib.lib().aw_ctx_create(ctypes.byref(ctx), 0, ctypes.byref(m)) != 0
    assert b"no CUDA device" in _lib.lib().aw_last_error()


def test_load_builds_reference_shaped_objects():
    from aware_b200.utils.models import load
    state = torch.random.get_rng_state()
    emb, det = load()
    torch.random.set_rng_state(state)
    assert det.detection_net is emb.detection_net            # shared net (load_model.py:56 upstream)
    assert emb.pattern_mode == det.pattern_mode == "bits2bipolar"
    assert emb.detection_net.output_length == 20 and det.threshold == 0.0
    assert (emb.tolerance_db, emb.num_iterations, emb.embedding_bands) == (6.0, 400, (500, 4000))
    assert emb.optimizer_name == "nadam" and emb.scheduler_name == "reduce_lr_on_plateau"
    assert emb.detection_net.get_model_info()["total_parameters"] == 1681960
    for w, wo in zip(emb.detection_net.weights, O.make_weights()):
        np.testing.assert_array_equal(w, wo.numpy())
    np.testing.assert_array_equal(emb.detection_net.mel_filter_bank, O.mel_basis())


def test_service_validation_matches_reference():
    from aware_b200.service import detect_watermark, embed_watermark
    from aware_b200.utils.models import load
    emb, det = load()
    x = np.zeros(16000, dtype=np.float32)
    bits = np.zeros(20, dtype=np.int32)
    with pytest.raises(ValueError, match="Invalid sample rate"):
        embed_watermark(x, 44100, bits, emb)
    with pytest.raises(ValueError, match="Invalid sample rate"):
        detect_watermark(x, 22050, det)
    with pytest.raises(ValueError, match="Invalid watermark length"):
        embed_watermark(x, 16000, np.zeros(19, dtype=np.int32), emb)
    with pytest.raises(ValueError, match="Invalid audio shape"):
        embed_watermark(np.zeros((10, 3), dtype=np.float32), 16000, bits, emb)
    with pytest.raises(ValueError, match="Invalid audio shape"):
        detect_watermark(np.zeros((10, 1), dtype=np.float32), 16000, det)   # Q22: (N,1) rejected


def test_codec_matches_oracle():
    from aware_b200.utils.watermark import PatternDecoder, PatternEncoder
    bits = O.synth_bits(3)[1]
    np.testing.assert_array_equal(PatternEncoder("bits2bipolar")(bits), O.encode_bits(bits))
    v = np.array([0.0, 1e-9, -0.3, 0.7, -1e-9], dtype=np.float32)
    np.testing.assert_array_equal(PatternDecoder(0.0, "bits2bipolar")(v), O.decode_values(v))
    assert PatternEncoder("bytes2bits")(b"\xa5").tolist() == [1, 0, 1, 0, 0, 1, 0, 1]
    assert PatternDecoder(0.5, "bytes2bits")(np.array([0.9, 0.1, 0.6])) == bytes([1, 0, 1])


def test_metrics_match_oracle():
    from aware_b200.metrics.audio import BER, SNR
    rng = np.random.default_rng(0)
    a, b = rng.integers(0, 2, 20), rng.integers(0, 2, 20)
    assert BER()(a, b) == O.ber_percent(a, b)
    x = rng.standard_normal(1000).astype(np.float32)
    y = x + 0.01 * rng.standard_normal(1000).astype(np.float32)
    assert SNR()(y, x[:900]) == pytest.approx(O.snr_db(y, x[:900]), rel=1e-12)
    assert SNR()(x, x) == float("inf")


def test_synth_matches_oracle_generator():
    from aware_b200 import synth
    np.testing.assert_array_equal(synth.synth_clip(4, 0.3, 44100), O.synth_clip(4, 0.3, 44100))
    np.testing.assert_array_equal(synth.synth_bits(5), O.synth_bits(5))
    b = synth.synth_batch(40, 0.1, 16000, unique=16)
    assert b.shape == (40, 1600) and len({bytes(r) for r in b}) == 40


def _upfirdn_model(x, h_tf, hpp, up, down, k_off, n_out):
    """numpy transcription of csrc/attacks.cuh:k_upfirdn (float32, oldest sample first)."""
    out = np.zeros(n_out, dtype=np.float32)
    n_in = len(x)
    for k in range(n_out):
        t = (k + k_off) * down
        phase, xi = t % up, t // up
        x0, hidx = xi - hpp + 1, phase * hpp
        if x0 < 0:
            hidx -= x0
            x0 = 0
        acc = np.float32(0)
        for j in range(x0, min(xi, n_in - 1) + 1):
            acc = np.float32(acc + np.float32(x[j] * h_tf[hidx]))
            hidx += 1
        out[k] = acc
    return out


def test_polyphase_plan_reproduces_scipy_resample_poly():
    from scipy.signal import resample_poly
    from aware_b200.attacks import polyphase_plan
    x = O.synth_clip(9, 0.02, 16000)                 # 320 samples
    for up, down in ((441, 160), (160, 441)):
        h_tf, hpp, k_off, n_out = polyphase_plan(len(x), up, down)
        got = _upfirdn_model(x, h_tf, hpp, up, down, k_off, n_out)
        want = resample_poly(x, up, down)
        assert got.shape == want.shape and want.dtype == np.float32
        np.testing.assert_array_equal(got, want)


def test_warm_up_length_bounds_filter_memory():
    """After `warm` samples from a zero state the chunk-parallel IIR scan must agree with the
    sequential recurrence down to the recurrence's own float64 round-off noise (measured as the
    distance between the direct form the reference uses and the well-conditioned SOS form;
    for the 8th-order band-stop that noise is far above 1e-16, see attacks.RandomBandstop)."""
    from scipy.signal import butter, lfilter, sosfilt
    from aware_b200.attacks import _warm_samples
    rng = np.random.default_rng(0)
    designs = (("low", 6, 4000.0), ("highpass", 4, 500.0), ("bandstop", 4, [3800.0, 4000.0]),
               ("bandstop", 4, [1206.5, 1406.5]))
    for sr in (44100, 16000):
        for btype, order, edge in designs:
            wn = np.asarray(edge) / (0.5 * sr)
            b, a = butter(order, wn, btype=btype)
            sos = butter(order, wn, btype=btype, output="sos")
            w = _warm_samples(b, a)
            assert 256 <= w < 40000
            x = rng.standard_normal(w + 4000) + 1.0          # includes a DC component
            full = lfilter(b, a, x)
            noise = np.abs(full - sosfilt(sos, x)).max()
            late = lfilter(b, a, x[2000:])                    # zero state, starts 2000 samples later
            assert np.abs(full[2000 + w:] - late[w:]).max() <= 10 * noise + 1e-12, (btype, sr, w, noise)


def test_wav_io_and_length_buckets(tmp_path):
    """aware_b200.evaluate: PCM WAV reader (16/24-bit, stereo mix-down like librosa mono=True) and
    the length bucketing that turns a ragged set of clips into equal-length launches."""
    import wave
    from aware_b200.evaluate import bucket_by_length, read_wav, write_wav
    rng = np.random.default_rng(5)
    x = (0.8 * rng.uniform(-1, 1, 4000)).astype(np.float32)
    p16 = str(tmp_path / "a.wav")
    write_wav(p16, x, 16000)
    y, sr = read_wav(p16)
    assert sr == 16000 and y.dtype == np.float32 and np.abs(y - x).max() <= 2.0 / 32768   # write x32767, read /32768
    # 24-bit stereo written by hand
    l = np.round(x * 8388607).astype(np.int32)
    r = np.round(-0.5 * x * 8388607).astype(np.int32)
    inter = np.stack([l, r], axis=1).reshape(-1)
    raw = bytearray()
    for v in inter:
        raw += int(v & 0xFFFFFF).to_bytes(3, "little")
    p24 = str(tmp_path / "b.wav")
    with wave.open(p24, "wb") as w:
        w.setnchannels(2); w.setsampwidth(3); w.setframerate(44100); w.writeframes(bytes(raw))
    y, sr = read_wav(p24)
    assert sr == 44100 and y.shape == (4000,)
    assert np.abs(y - 0.25 * x).max() <= 2e-7                       # mean of x and -x/2
    assert bucket_by_length([5, 7, 5, 9, 7, 5]) == {5: [0, 2, 5], 7: [1, 4], 9: [3]}
    assert bucket_by_length([]) == {}


def test_vad_gate_is_explicit_never_silent():
    """ADVICE r1: without webrtcvad the gate must not quietly answer "not silent".  The shipped card opts
    out explicitly (vad_gate: false); switching it on without the package raises ImportError."""
    from aware_b200.service import embed_watermark
    from aware_b200.utils.audio import SilenceChecker, silent_mask
    from aware_b200.utils.models import load
    emb, _ = load()
    assert emb.vad_gate is False
    x = np.zeros(16000, dtype=np.float32)
    assert not silent_mask([x], 16000, emb).any()                 # gate off: nothing is rejected
    try:
        import webrtcvad  # noqa: F401
        pytest.skip("webrtcvad installed")
    except ImportError:
        pass
    with pytest.raises(ImportError, match="webrtcvad"):
        SilenceChecker()(x)
    emb.vad_gate = True
    with pytest.raises(ImportError, match="webrtcvad"):
        embed_watermark(x, 16000, np.zeros(20, dtype=np.int32), emb)


def test_bench_suite_is_identical_for_both_arms():
    """bench.py draws the attack parameters once; the oracle restatement list (reference arm, parity
    gates) and the CUDA attack list are built from the same draw, in the same order."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    from aware_b200 import attacks as A
    p = bench.suite_params(4096, 16000, np.random.default_rng(99), 3)
    both = bench.build_suite(A, 16000, p)
    only_oracle = bench.build_suite(None, 16000, p)
    assert len(both) == len(only_oracle) == 13 and all(a is None for a, _ in only_oracle)
    names = [a.name for a, _ in both]
    assert names[:4] == ["pcm_8", "pcm_12", "pcm_16", "pcm_24"] and names[-2:] == ["low_pass", "high_pass"]
    x = O.synth_clip(0, 4096 / 16000, 16000)
    for (a, f), (_, g) in zip(both, only_oracle):
        np.testing.assert_array_equal(np.asarray(f(O, x, 1)), np.asarray(g(O, x, 1)))
    bs = [a for a, _ in both if a.name.startswith("bandstop")][0]
    assert bs.fast is False and bs.f_low == p["f_low"]           # the bit-exact sequential mode is benched

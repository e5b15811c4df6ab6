"""Batched equivalent of the reference's evaluation driver (scripts/test.py:13-117 upstream):

    for every file: load mono -> resample to 16 kHz -> embed 20 random bits -> detect -> BER,
    then every attack -> detect -> BER; finally the per-attack mean BER.

Upstream does this one clip at a time on the CPU.  Here clips are grouped by length
(length-bucketed launches: every kernel wants equal-length rows), each bucket goes through
`embed_watermark_batch` / `Attack.apply_batch` / `detect_watermark_batch` on the GPU, the
resample-to-16 kHz step (`scipy.signal.resample_poly(audio, 16000, sr)`, test.py:60-65) runs
on the GPU through the same bit-exact polyphase kernel the `Resample` attack uses, and with
`torch.distributed` initialised the per-attack error counters are all-reduced once at the end
(`parallel.allreduce_counters`).  Upstream's MP3 attack calls ffmpeg and is not run.  Its
time-stretch and pitch-shift attacks call rubberband; `desync=True` (`--desync`) appends this
project's phase-vocoder definitions of them (`attacks.desync_attacks()`: time stretch 0.9 / 1.1,
pitch shift -2 / +2 semitones).  `room=True` (`--room`) appends the reverberation and echo
attacks (`attacks.room_attacks()`), which have no upstream counterpart.  STOI runs on the GPU;
PESQ is a third-party package, scored when installed and skipped otherwise, like the optional
`webrtcvad` gate.

    python -m aware_b200.evaluate <folder with .wav files> [--iters 400] [--seed 0] [--desync] [--room]
"""
from __future__ import annotations

import argparse
import math
import os
import wave
from collections import defaultdict

import numpy as np
import torch

from . import attacks as A
from .parallel import allreduce_counters, shard_range
from .utils.logger import logger

TARGET_SR = 16000


# ------------------------------------------------------------------------------ WAV I/O
def read_wav(path: str):
    """(float32 mono in [-1, 1), sample_rate) from a PCM WAV file (8/16/24/32-bit), channels
    averaged like `librosa.load(..., mono=True)` (test.py:53)."""
    with wave.open(path, "rb") as w:
        nch, width, sr, n = w.getnchannels(), w.getsampwidth(), w.getframerate(), w.getnframes()
        raw = w.readframes(n)
    if width == 1:
        x = (np.frombuffer(raw, dtype=np.uint8).astype(np.float32) - 128.0) / 128.0
    elif width == 2:
        x = np.frombuffer(raw, dtype="<i2").astype(np.float32) / 32768.0
    elif width == 3:
        b = np.frombuffer(raw, dtype=np.uint8).reshape(-1, 3).astype(np.int32)
        v = b[:, 0] | (b[:, 1] << 8) | (b[:, 2] << 16)
        x = (v - ((v & 0x800000) << 1)).astype(np.float32) / 8388608.0
    elif width == 4:
        x = np.frombuffer(raw, dtype="<i4").astype(np.float32) / 2147483648.0
    else:
        raise ValueError(f"unsupported PCM sample width {width}")
    if nch > 1:
        x = x.reshape(-1, nch).mean(axis=1).astype(np.float32)
    return x, sr


def write_wav(path: str, audio: np.ndarray, sr: int):
    """16-bit PCM mono."""
    pcm = np.clip(np.round(np.asarray(audio, dtype=np.float64) * 32767.0), -32768, 32767).astype("<i2")
    with wave.open(path, "wb") as w:
        w.setnchannels(1)
        w.setsampwidth(2)
        w.setframerate(int(sr))
        w.writeframes(pcm.tobytes())


# --------------------------------------------------------------------- resample on the GPU
_PLANS = {}


def resample_poly_batch(x: torch.Tensor, up: int, down: int, engine) -> torch.Tensor:
    """scipy.signal.resample_poly(x, up, down) for a float32 batch [n, N] on the device (same
    Kaiser(5.0) FIR, tap order and edge handling: bit-exact, see tests/test_host_logic.py
    `test_polyphase_plan_reproduces_scipy_resample_poly` and the `Resample` attack)."""
    g = math.gcd(int(up), int(down))
    up, down = int(up) // g, int(down) // g
    if up == down:
        return x
    key = (x.shape[1], up, down, engine.device.index)
    if key not in _PLANS:
        h_tf, tpp, first, n_out = A.polyphase_plan(x.shape[1], up, down)
        _PLANS[key] = (torch.from_numpy(h_tf).to(engine.device), tpp, first, n_out)
    h, tpp, first, n_out = _PLANS[key]
    return engine.attack_upfirdn(x, h, tpp, up, down, first, n_out)


# ------------------------------------------------------------------------------- buckets
def bucket_by_length(lengths):
    """{length: [clip indices]} in first-seen order: one launch sequence per distinct length."""
    groups = defaultdict(list)
    for i, n in enumerate(lengths):
        groups[int(n)].append(i)
    return dict(groups)


def default_attacks(rng: np.random.Generator):
    """The in-scope subset of test.py:15-18's list (MP3 / TimeStretch / PitchShift call external
    binaries upstream; the latter two are available as `attacks.desync_attacks()`).  Random parameters
    are drawn per batch from `rng` (upstream draws them unseeded)."""
    return [A.PCMBitDepthConversion(8), A.PCMBitDepthConversion(12), A.PCMBitDepthConversion(16),
            A.PCMBitDepthConversion(24), A.DeleteSamples(0.1), A.DeleteSamples(0.15), A.DeleteSamples(0.2),
            A.Resample(), A.RandomBandstop(), A.SampleSupression(0.1), A.SampleSupression(0.25),
            A.LowPassFilter(), A.HighPassFilter()]       # IIRs: sequential scan = scipy bit for bit


# ------------------------------------------------------------------------------ the driver
def evaluate_clips(clips, rates, embedder, detector, attack_list=None, seed: int = 0, keep_audio: bool = False,
                   desync: bool = False, room: bool = False):
    """clips: list of 1-D float arrays, rates: their sample rates.  Returns a dict with per-attack
    mean BER in percent ('orig' = no attack, as upstream's `rec`), mean SNR, the decoded bits and
    (optionally) the watermarked audio, all for THIS rank's shard when torch.distributed is
    initialised -- the means are over all ranks (counter all-reduce).  `desync` appends
    `attacks.desync_attacks()` (time stretch / pitch shift) to the attack list, `room` appends
    `attacks.room_attacks()` (reverberation / echo) after them.  The appended attacks draw their random
    parameters from their own generator, np.random.default_rng((seed, 2)), so they leave the results of
    the attack list unchanged."""
    from .service import detect_watermark_batch, embed_watermark_batch
    eng = embedder.engine
    A.set_engine(eng)
    rng = np.random.default_rng(seed)
    attack_list = default_attacks(rng) if attack_list is None else list(attack_list)
    # the optional attacks draw from a generator of their own (Reverb picks a response per clip), so the
    # draws of the attack list, and with them its results, are the same with or without them
    extra = (A.desync_attacks() if desync else []) + (A.room_attacks() if room else [])
    extra_rng = np.random.default_rng((seed, 2))
    names = ["orig"] + [a.name for a in attack_list + extra]
    world = torch.distributed.get_world_size() if torch.distributed.is_initialized() else 1
    rank = torch.distributed.get_rank() if torch.distributed.is_initialized() else 0
    bits_all = np.random.default_rng(seed + 1).integers(0, 2, size=(len(clips), 20), dtype=np.int32)
    lo, hi = shard_range(len(clips), rank, world)
    mine = list(range(lo, hi))
    # speech / silence gate per clip (scripts/test.py:68-72 skips a file whose embed raises ValueError):
    # rejected clips are dropped here and never reach the counters
    from .utils.audio import silent_mask
    n_silent = 0
    if getattr(embedder, "vad_gate", False):
        keep = []
        for i in mine:
            if silent_mask([np.asarray(clips[i], dtype=np.float32)], int(rates[i]), embedder)[0]:
                logger.warning(f"clip {i}: no speech detected, skipped")
                n_silent += 1
            else:
                keep.append(i)
        mine = keep

    # resample to 16 kHz on the device, one launch per (length, rate) group
    at16 = {}
    groups = defaultdict(list)
    for i in mine:
        groups[(len(clips[i]), int(rates[i]))].append(i)
    for (n, sr), idx in groups.items():
        x = torch.from_numpy(np.stack([np.asarray(clips[i], dtype=np.float32) for i in idx])).to(eng.device)
        y = resample_poly_batch(x, TARGET_SR, sr, eng) if sr != TARGET_SR else x
        for k, i in enumerate(idx):
            at16[i] = y[k]

    counters = torch.zeros((len(names), 3), dtype=torch.int64, device=eng.device)
    # quality aggregates, all-reduced with the counters: [sum of SNR, clips with finite SNR,
    # sum of STOI > 0.1, their count (scripts/test.py:86-88), sum of PESQ, clips PESQ could score (:79-84)]
    sums = torch.zeros(6, dtype=torch.float64, device=eng.device)
    try:
        import pesq as _pesq_pkg  # noqa: F401
        from .metrics.audio import PESQ
        pesq_metric = PESQ()
    except ImportError:
        pesq_metric = None                                               # third-party host package, optional
    decoded, audio_out = {}, {}
    for n, idx_local in bucket_by_length([at16[i].shape[0] for i in mine]).items():
        idx = [mine[k] for k in idx_local]
        x = torch.stack([at16[i] for i in idx])
        bits = torch.from_numpy(bits_all[idx]).to(eng.device)
        y = embed_watermark_batch(x, TARGET_SR, bits_all[idx], embedder)
        got, _ = detect_watermark_batch(y, TARGET_SR, detector, bits, counters[0])
        snr = eng.snr(y, x)
        ok = torch.isfinite(snr)
        sums[:2] += torch.stack([snr[ok].sum(), ok.sum().double()])
        eng.stoi(x[:, :y.shape[1]], y, TARGET_SR, stoi_sum=sums[2:4])       # GPU STOI, scores > 0.1 accumulate
        if pesq_metric is not None:
            ps = np.asarray(pesq_metric.batch(list(y.cpu().numpy()), list(x.cpu().numpy()), TARGET_SR))
            good = np.isfinite(ps)
            sums[4:6] += torch.tensor([ps[good].sum(), good.sum()], dtype=torch.float64, device=eng.device)
        for k, i in enumerate(idx):
            decoded[i] = got[k].cpu().numpy()
            if keep_audio:
                audio_out[i] = y[k].cpu().numpy()
        A.run_suite(attack_list, y, TARGET_SR,
                    lambda a_i, z: detect_watermark_batch(z, TARGET_SR, detector, bits, counters[a_i + 1]),
                    rng=rng, engine=eng)
        if extra:
            first = 1 + len(attack_list)
            A.run_suite(extra, y, TARGET_SR,
                        lambda a_i, z: detect_watermark_batch(z, TARGET_SR, detector, bits, counters[first + a_i]),
                        rng=extra_rng, engine=eng)
    allreduce_counters(counters, sums)
    c = counters.cpu().numpy()
    ber = {nm: (100.0 * c[k, 0] / c[k, 1] if c[k, 1] else float("nan")) for k, nm in enumerate(names)}
    s = sums.cpu().numpy()
    return {"ber_percent": ber, "snr_db_mean": float(s[0] / s[1]) if s[1] else float("nan"),
            "stoi_mean": float(s[2] / s[3]) if s[3] else float("nan"),
            "pesq_mean": float(s[4] / s[5]) if s[5] else float("nan"),
            "n_clips": int(c[0, 2]), "n_silent_skipped": n_silent, "bits": bits_all, "decoded": decoded,
            "audio": audio_out}


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("folder")
    ap.add_argument("--iters", type=int, default=400)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--desync", action="store_true",
                    help="also run the time-stretch (0.9, 1.1) and pitch-shift (-2, +2 semitones) attacks")
    ap.add_argument("--room", action="store_true",
                    help="also run the reverberation (RT60 0.3 s, 0.7 s) and echo (50 ms, 0.5) attacks")
    args = ap.parse_args(argv)
    from .utils.models import load
    paths = sorted(os.path.join(args.folder, f) for f in os.listdir(args.folder) if f.lower().endswith(".wav"))
    if not paths:
        logger.error(f"Audio file path not found or empty: {args.folder}")
        return 1
    clips, rates = zip(*(read_wav(p) for p in paths))
    embedder, detector = load()
    embedder.num_iterations = args.iters
    embedder.verbose = False
    res = evaluate_clips(list(clips), list(rates), embedder, detector, seed=args.seed, desync=args.desync,
                         room=args.room)
    for name, v in res["ber_percent"].items():
        logger.info(f"{name}: mean: {v:.4f}")
    logger.info(f"snr: mean: {res['snr_db_mean']:.2f} dB over {res['n_clips']} clips")
    logger.info(f"stoi: mean: {res['stoi_mean']:.4f}")
    logger.info(f"pesq: mean: {res['pesq_mean']:.4f}")
    return 0


if __name__ == "__main__":
    raise SystemExit(main())

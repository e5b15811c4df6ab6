"""Throughput of the time-stretch / pitch-shift attacks and of their CUDA stages on one GPU.

    python tests/profile_desync.py [--clips 256 1024] [--iters 20] [--out profiles/desync.jsonl]

For 10 s clips at 44.1 kHz (synthetic, aware_b200.synth) and each batch size, it warms every shape up, then
times with CUDA events, over `--iters` back-to-back launches each:
  * every stage: stft_full, phase_vocoder (per attack rate), istft_full, and the polyphase resample of the
    pitch shifts;
  * every attack of attacks.desync_attacks() end to end, reported as attacked audio-seconds per second;
  * for comparison, the existing band kernels that use the same FFT (analysis_mag, synthesis_wave), read
    through the engine's per-kernel timeline.
Per-frame times are given per (clip, frame).  The phase vocoder is compared with its bytes: the input
spectrum read once (a frame's |D| and angle are carried while the step stays or advances by one) and the
output spectrum written.  Every working set exceeds the 126 MB L2 (about 7 MB of spectrum per clip).  The
card's name and power limit are read in the same run.  One JSON line is appended to --out."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
from aware_b200 import attacks as A                       # noqa: E402
from aware_b200.synth import synth_batch                   # noqa: E402
from aware_b200.utils.models import load                  # noqa: E402

SR, SECONDS = 44100, 10.0


def card():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        name, power, clock = [s.strip() for s in q.stdout.strip().splitlines()[0].split(",")]
        out.update(smi_name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # noqa: BLE001
        out["smi_error"] = repr(e)
    return out


def timed(fn, iters):
    """Mean ms per call over `iters` back-to-back calls, after two warm-up calls."""
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def profile_size(eng, n, iters):
    x = torch.from_numpy(synth_batch(n, SECONDS, SR)).to(eng.device)
    N = x.shape[1]
    T = 1 + N // 256
    spec_bytes = lambda frames: n * frames * 513 * 8      # noqa: E731
    res = {"n_clips": n, "n_samples": N, "frames": T, "stages": {}, "attacks": {}}
    st = res["stages"]

    spec = eng.stft_full(x)
    ms = timed(lambda: eng.stft_full(x), iters)
    st["stft_full"] = {"ms": ms, "ns_per_frame": 1e6 * ms / (n * T), "GB_written": spec_bytes(T) / 1e9}
    for att in A.desync_attacks():
        rate = att.rate
        T_out = A.stretch_frames(T, rate)
        n_out = A.stretch_length(N, rate)
        out = eng.phase_vocoder(spec, rate)
        assert torch.isfinite(torch.view_as_real(out[:4])).all()
        ms = timed(lambda: eng.phase_vocoder(spec, rate), iters)
        moved = spec_bytes(T) + spec_bytes(T_out)
        st["phase_vocoder_%g" % rate] = {"ms": ms, "frames_out": T_out, "GB_moved": moved / 1e9,
                                         "GB_per_s": moved / ms / 1e6, "ns_per_frame": 1e6 * ms / (n * T_out)}
        ms = timed(lambda: eng.istft_full(out, n_out), iters)
        st["istft_full_%g" % rate] = {"ms": ms, "ns_per_frame": 1e6 * ms / (n * T_out)}
        if isinstance(att, A.PitchShift):
            y = eng.istft_full(out, n_out)
            p, q = att.ratio.numerator, att.ratio.denominator
            h, tpp, first, n_res = A.polyphase_plan(y.shape[1], q, p)
            h = torch.from_numpy(h).to(eng.device)
            ms = timed(lambda: eng.attack_upfirdn(y, h, tpp, q, p, first, n_res), iters)
            st["resample_%d_%d" % (q, p)] = {"ms": ms, "taps_per_phase": tpp}
            del y
        del out
        ms = timed(lambda: att.apply_batch(x, SR, engine=eng), iters)
        res["attacks"][att.name] = {"ms": ms, "audio_s_per_s": n * SECONDS / (ms / 1e3)}
        torch.cuda.empty_cache()
    del spec
    torch.cuda.empty_cache()

    # the band kernels that use the same 1024-point warp FFT, as the engine's timeline sees them
    mag, ph = eng.stft_band(x, SR, normalize=False, phasor=True)
    eng.stft_band(x, SR)
    eng.istft_band(mag, ph, SR)
    torch.cuda.synchronize()
    eng.profile(True)
    eng.profile_read_named()
    for _ in range(iters):
        eng.stft_band(x, SR)
    for _ in range(iters):
        eng.istft_band(mag, ph, SR)
    eng.stft_band(x, SR)                                  # closes the last synthesis interval
    named = eng.profile_read_named()
    eng.profile(False)
    _, nb = eng.band_bins(SR)
    for k in ("analysis_mag", "synthesis_wave"):
        cnt, tot = named.get(k, (0, 0.0))
        if cnt:
            st[k] = {"ms": tot / cnt, "ns_per_frame": 1e6 * tot / cnt / (n * T), "band_bins": nb, "launches": cnt}
    del mag, ph, x
    torch.cuda.empty_cache()
    return res


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--clips", type=int, nargs="+", default=[256, 1024])
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "desync.jsonl"))
    args = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("profile_desync.py needs a CUDA device")
    if args.iters < 20:
        raise SystemExit("--iters must be at least 20")
    emb, _ = load()
    eng = emb.engine
    A.set_engine(eng)
    rec = {"script": "tests/profile_desync.py", "time": time.strftime("%Y-%m-%dT%H:%M:%S"), "card": card(),
           "sample_rate": SR, "seconds": SECONDS, "iters": args.iters, "sizes": []}
    print("card:", rec["card"], flush=True)
    for n in args.clips:
        r = profile_size(eng, n, args.iters)
        rec["sizes"].append(r)
        print("%d x %g s @ %d Hz:" % (n, SECONDS, SR))
        for k, v in r["stages"].items():
            print("  %-24s %s" % (k, ", ".join("%s %.4g" % kv for kv in v.items())))
        for k, v in r["attacks"].items():
            print("  %-24s %.2f ms  %.0f audio-s/s" % (k, v["ms"], v["audio_s_per_s"]))
        sys.stdout.flush()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        f.write(json.dumps(rec) + "\n")
    print("wrote", args.out)


if __name__ == "__main__":
    main()

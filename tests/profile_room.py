"""Throughput of the reverberation / echo convolution (aw_attack_convolve) and of its two CUDA stages on one GPU.

    python tests/profile_room.py [--clips 1024] [--iters 20] [--direct-clips 16] [--out profiles/room.jsonl]

For 10 s clips (synthetic, aware_b200.synth) at 44.1 kHz and at 16 kHz and each RT60 in {0.3, 0.7, 1.2} s
(one synthetic response of `attacks.Reverb`, shared by the batch), plus the 50 ms echo, it warms every shape
up, then times `--iters` back-to-back launches with CUDA events:
  * the whole convolution, reported as attacked audio-seconds per second;
  * each stage (conv_fwd, conv_mac_inv), read through the engine's per-kernel timeline in a separate pass;
  * the existing direct-form FIR kernel (attack_upfirdn, flipped taps) on the same response, on a batch of
    `--direct-clips` clips small enough to finish, compared per clip.
Each stage is compared with its own floor: the larger of its algorithmic FLOP over the FP32 peak (SM count x
128 lanes x 2 x the card's maximum SM clock) and its algorithmic bytes over 7.7 TB/s of HBM (the data sheet's
figure).  FLOP: 5 n log2 n = 51 200 per 1024-point complex FFT, one per two blocks in each stage, and
8 FLOP per bin and partition of the complex multiply-accumulate (8 NB K 513 per clip).  Bytes, the algorithmic
floor: conv_fwd reads the clip and writes the packed block spectra (NB x 512 x 8); conv_mac_inv reads those
spectra and the partition spectra once and writes the clip.  conv_mac_inv's CTAs fetch each block spectrum
once per CTA that needs it, about ceil((K + 15) / 16) times, partly from L2; `X_fetched_GB` records that
count (computed from the shapes, not measured).  Every working set exceeds the 126 MB L2 (3.5 MB of spectra per
44.1 kHz clip).  The card's name and power limit are read in the same run.  One JSON line is appended to
--out."""
import argparse
import json
import math
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

SECONDS = 10.0
HBM_BYTES_PER_S = 7.7e12
FFT_FLOP = 5 * 1024 * 10


def card():
    out = {"name": torch.cuda.get_device_name(0), "sms": torch.cuda.get_device_properties(0).multi_processor_count}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        name, power, clock = [s.strip() for s in q.stdout.strip().splitlines()[0].split(",")]
        out.update(smi_name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # noqa: BLE001
        out["smi_error"] = repr(e)
    return out


def fp32_peak(c):
    """FP32 FLOP/s: SMs x 128 lanes x 2 (FMA) x the maximum SM clock (1 965 MHz when nvidia-smi is silent)."""
    mhz = 1965.0
    try:
        mhz = float(c["max_sm_clock"].split()[0])
    except (KeyError, ValueError, IndexError):
        pass
    return c["sms"] * 128 * 2 * mhz * 1e6


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


def x_rows_fetched(NB, K, R=16):
    """Block-spectrum rows one clip's conv_mac_inv CTAs load: the R blocks of each CTA's initial register
    ring, then one per partition step while the block lies in the clip (conv.cuh)."""
    return sum(min(R, NB - b0) + min(min(K, b0 + R), b0) for b0 in range(0, NB, R))


def floor_ms(flop, nbytes, peak):
    t_f, t_b = flop / peak * 1e3, nbytes / HBM_BYTES_PER_S * 1e3
    return (t_f, "fp32") if t_f >= t_b else (t_b, "hbm")


def stage(ms, flop, nbytes, peak):
    fl, bound = floor_ms(flop, nbytes, peak)
    return {"ms": ms, "GFLOP": flop / 1e9, "GB": nbytes / 1e9, "floor_ms": fl, "bound": bound,
            "share_of_floor": fl / ms}


def profile_case(eng, x, sr, att, iters, n_direct, peak):
    n, N = x.shape
    h = att.responses(sr)[0]
    M = len(h)
    NB, K = -(-N // 512), -(-M // 512)
    spec = torch.from_numpy(A.conv_spectra(h)).to(eng.device)
    y = eng.attack_convolve(x, spec)
    assert torch.isfinite(y[:4]).all()
    del y
    ms = timed(lambda: eng.attack_convolve(x, spec), iters)
    res = {"attack": att.name, "taps": M, "parts": K, "blocks": NB, "ms": ms,
           "audio_s_per_s": n * SECONDS / (ms / 1e3), "stages": {}}
    # per stage, from the engine's timeline (a separate pass: the event marks cost host time)
    torch.cuda.synchronize()
    eng.profile(True)
    eng.profile_read_named()
    for _ in range(iters):
        eng.attack_convolve(x, spec)
    eng.attack_pcm(x[:1], 16)                              # closes the last conv_mac_inv interval
    named = eng.profile_read_named()
    eng.profile(False)
    fwd_flop = n * math.ceil(NB / 2) * FFT_FLOP
    fwd_bytes = n * (4 * N + NB * 512 * 8)
    mac_flop = n * (8 * NB * K * 513 + math.ceil(NB / 2) * FFT_FLOP)
    mac_bytes = n * (NB * 512 * 8 + 4 * N) + K * 513 * 8
    for key, flop, nbytes in (("conv_fwd", fwd_flop, fwd_bytes), ("conv_mac_inv", mac_flop, mac_bytes)):
        cnt, tot = named.get(key, (0, 0.0))
        if cnt:
            res["stages"][key] = dict(stage(tot / cnt, flop, nbytes, peak), launches=cnt)
    if "conv_mac_inv" in res["stages"]:
        res["stages"]["conv_mac_inv"]["X_fetched_GB"] = n * x_rows_fetched(NB, K) * 512 * 8 / 1e9
    # the direct form on the same taps, a few clips
    if n_direct:
        xs = x[:n_direct].contiguous()
        h_tf = torch.from_numpy(np.ascontiguousarray(h[::-1])).to(eng.device)
        d_iters = 3 if M > 1024 else iters
        ms_d = timed(lambda: eng.attack_upfirdn(xs, h_tf, M, 1, 1, 0, N), d_iters)
        per_clip_direct = ms_d / n_direct
        res["direct_fir"] = {"clips": n_direct, "iters": d_iters, "ms": ms_d, "ms_per_clip": per_clip_direct,
                             "GFLOP_per_s": n_direct * 2.0 * M * N / (ms_d / 1e3) / 1e9,
                             "speedup_of_convolve": per_clip_direct / (ms / n)}
        del xs
    del spec
    torch.cuda.empty_cache()
    return res


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--clips", type=int, default=1024)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--direct-clips", type=int, default=16)
    ap.add_argument("--rates", type=int, nargs="+", default=[44100, 16000])
    ap.add_argument("--rt60", type=float, nargs="+", default=[0.3, 0.7, 1.2])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "room.jsonl"))
    args = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("profile_room.py needs a CUDA device")
    if args.iters < 20:
        raise SystemExit("--iters must be at least 20")
    emb, _ = load()
    eng = emb.engine
    A.set_engine(eng)
    c = card()
    peak = fp32_peak(c)
    rec = {"script": "tests/profile_room.py", "time": time.strftime("%Y-%m-%dT%H:%M:%S"), "card": c,
           "fp32_peak_TFLOP_s": peak / 1e12, "hbm_TB_s": HBM_BYTES_PER_S / 1e12, "seconds": SECONDS,
           "n_clips": args.clips, "iters": args.iters, "rates": []}
    print("card:", c, "FP32 peak %.1f TFLOP/s" % (peak / 1e12), flush=True)
    for sr in args.rates:
        x = torch.from_numpy(synth_batch(args.clips, SECONDS, sr)).to(eng.device)
        cases = []
        for att in [A.Reverb(t, seed=0) for t in args.rt60] + [A.Echo(0.05, 0.5)]:
            r = profile_case(eng, x, sr, att, args.iters, args.direct_clips, peak)
            cases.append(r)
            print("%d x %g s @ %d Hz, %s (M %d, K %d, NB %d): %.3f ms, %.0f audio-s/s" % (
                args.clips, SECONDS, sr, r["attack"], r["taps"], r["parts"], r["blocks"], r["ms"], r["audio_s_per_s"]))
            for k, v in r["stages"].items():
                print("    %-13s %.3f ms  floor %.3f ms (%s)  %.0f %% of floor" % (k, v["ms"], v["floor_ms"], v["bound"],
                                                                               100 * v["share_of_floor"]))
            if "direct_fir" in r:
                d = r["direct_fir"]
                print("    direct FIR    %.3f ms per clip (%.0f GFLOP/s); the convolution is %.0fx faster" % (
                    d["ms_per_clip"], d["GFLOP_per_s"], d["speedup_of_convolve"]))
            sys.stdout.flush()
        rec["rates"].append({"sample_rate": sr, "n_samples": x.shape[1], "cases": cases})
        del x
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        f.write(json.dumps(rec) + "\n")
    print("wrote", args.out)


if __name__ == "__main__":
    main()

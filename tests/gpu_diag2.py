"""Round-2 GPU diagnostics (development aid, not a test): python tests/gpu_diag2.py <what>"""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import numpy as np, torch


def big_detect():
    from aware_b200.synth import synth_batch, synth_bits
    from aware_b200.utils.models import load
    from aware_b200 import attacks as A
    emb, det = load(); emb.verbose = False
    eng = emb.engine; A.set_engine(eng)
    sr = 44100
    x = torch.from_numpy(synth_batch(256, 10.0, sr)).cuda()
    pat = torch.from_numpy(2 * synth_bits(256) - 1)
    for tc in (False, True):
        eng.set_tc_spectral(tc)
        y = eng.embed(x, sr, pat, iters=6, scale="signed_max", precision="fp16")
        torch.cuda.synchronize()
        print("embed tc=%s ok" % tc, flush=True)
        for n in (256, 512, 1024):
            yy = y.repeat(n // 256, 1)
            try:
                v = eng.detect(yy, sr)
                torch.cuda.synchronize()
                print("  detect n=%d ok" % n, float(v.abs().min()), flush=True)
            except Exception as e:  # noqa: BLE001
                print("  detect n=%d FAILED: %s" % (n, e), flush=True)


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "big_detect":
    big_detect()


def tl(tag=""):
    """per-kernel-class timeline of a few embed iterations (128 clips), TC spectral path on / off"""
    from aware_b200.synth import synth_batch, synth_bits
    from aware_b200.utils.models import load
    emb, det = load(); emb.verbose = False
    eng = emb.engine
    sr = 44100
    n = int(os.environ.get("CLIPS", "256"))
    x = torch.from_numpy(synth_batch(n, 10.0, sr)).cuda()
    pat = torch.from_numpy(2 * synth_bits(n) - 1)
    for tc in (True, False):
        eng.set_tc_spectral(tc)
        eng.embed(x, sr, pat, iters=4, precision="fp16")
        eng.profile(True)
        eng.embed(x, sr, pat, iters=10, precision="fp16")
        torch.cuda.synchronize()
        eng.profile(False)
        eng.profile_read()
        t = eng.profile_read_named()
        tot = sum(v[1] for v in t.values())
        print("tc=%s total %.2f ms per iteration" % (tc, tot / 10))
        for k, v in sorted(t.items(), key=lambda kv: -kv[1][1])[:40]:
            print("   %-28s %4d launches %8.3f ms/iter" % (k, v[0], v[1] / 10))


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "tl":
    tl()


def tcprof():
    """short fp16 embed on the TC spectral path for ncu (64 clips x 10 s, 6 iterations, eager launches)"""
    from aware_b200.synth import synth_batch, synth_bits
    from aware_b200.utils.models import load
    emb, det = load(); emb.verbose = False
    eng = emb.engine
    sr = 44100
    n = int(os.environ.get("CLIPS", "64"))
    x = torch.from_numpy(synth_batch(n, 10.0, sr)).cuda()
    pat = torch.from_numpy(2 * synth_bits(n) - 1)
    eng.embed(x, sr, pat, iters=int(os.environ.get("ITERS", "6")), precision="fp16")
    torch.cuda.synchronize()
    print("tcprof ok", eng.launch_count())


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "tcprof":
    tcprof()


def pair():
    """K >= 512 layers on CTA pairs vs one CTA per tile: instrumented per-kernel times and the
    un-instrumented (graph replay) time of 100 iterations, 256 clips x 10 s, fp16 and tf32 loops"""
    from aware_b200.synth import synth_batch, synth_bits
    from aware_b200.utils.models import load
    emb, det = load(); emb.verbose = False
    eng = emb.engine
    sr = 44100
    n = int(os.environ.get("CLIPS", "256"))
    x = torch.from_numpy(synth_batch(n, 10.0, sr)).cuda()
    pat = torch.from_numpy(2 * synth_bits(n) - 1)
    for prec in ("fp16", "tf32"):
        for on in (True, False, True, False):
            eng.set_pair_gemm(on)
            eng.embed(x, sr, pat, iters=4, precision=prec)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            eng.embed(x, sr, pat, iters=100, precision=prec)
            b.record()
            torch.cuda.synchronize()
            print("%s pair=%s: %.3f ms per iteration (graph replay)" % (prec, on, a.elapsed_time(b) / 100))
        for on in (True, False):
            eng.set_pair_gemm(on)
            eng.profile(True)
            eng.embed(x, sr, pat, iters=10, precision=prec)
            torch.cuda.synchronize()
            eng.profile(False)
            eng.profile_read()
            t = eng.profile_read_named()
            tot = sum(v[1] for v in t.values())
            print("%s pair=%s instrumented total %.2f ms per iteration" % (prec, on, tot / 10))
            for k, v in sorted(t.items(), key=lambda kv: -kv[1][1])[:12]:
                print("   %-28s %4d launches %8.3f ms/iter" % (k, v[0], v[1] / 10))


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "pair":
    pair()


def quick():
    """fp16 loop at 256 clips x 10 s: graph-replay ms per iteration (100 iterations, twice) and the
    instrumented per-class times of 10 iterations"""
    from aware_b200.synth import synth_batch, synth_bits
    from aware_b200.utils.models import load
    emb, det = load(); emb.verbose = False
    eng = emb.engine
    sr = 44100
    n = int(os.environ.get("CLIPS", "256"))
    x = torch.from_numpy(synth_batch(n, 10.0, sr)).cuda()
    pat = torch.from_numpy(2 * synth_bits(n) - 1)
    if "BWD64" in os.environ:
        eng.set_bwd64_stream(os.environ["BWD64"] == "1")
    eng.embed(x, sr, pat, iters=4, precision="fp16")
    torch.cuda.synchronize()
    for _ in range(2):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        eng.embed(x, sr, pat, iters=100, precision="fp16")
        b.record()
        torch.cuda.synchronize()
        print("fp16: %.3f ms per iteration (graph replay, 100 iterations)" % (a.elapsed_time(b) / 100), flush=True)
    eng.profile(True)
    eng.embed(x, sr, pat, iters=10, precision="fp16")
    torch.cuda.synchronize()
    eng.profile(False)
    eng.profile_read()
    t = eng.profile_read_named()
    tot = sum(v[1] for v in t.values())
    print("instrumented total %.2f ms per iteration" % (tot / 10))
    for k, v in sorted(t.items(), key=lambda kv: -kv[1][1])[:40]:
        print("   %-28s %4d launches %8.3f ms/iter" % (k, v[0], v[1] / 10))


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "quick":
    quick()

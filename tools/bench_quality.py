"""What measuring enlargement quality costs on the GPU, all in one process on one GPU:

  evaluate  Net.evaluate_frames_host: 256 frames of 960x540 RGBA8 + their 1920x1080 RGBA8
            references up, 1920x1080 RGB8 + 4 doubles a frame down (x2)
  frames    Net.upscale_frames_host on the same frames (the enlargement alone)

for 9-1-5 128/64 and 64/32, Lanczos and bicubic, on pinned host buffers.  The two entries are
timed alternately (host clock around whole synchronous calls, each repeated for at least
`--seconds` after a warm-up call) and their RGB8 results compared byte for byte first.  Then the
quality kernel alone (srcnn_image_quality, both launches) on 32 frame pairs of 1920x1080, an RGB8
and an RGBA8 result against RGBA8 references: 32 * 2.07 Mpx * 7 or 8 bytes = 464 or 531 MB per
call, well over the 126 MB L2, so every call reads HBM.  Its rate counts each input byte once
(the halo re-reads of neighbouring tiles hit L2); the FP64 count is that of the kernel's loops:
per region pixel 26/16 horizontal rows of 5 x 11 FMAs, 5 x 11 vertical FMAs, 3 products for the
maps and ~12 operations for the SSIM of a window (an FMA counted as 2).

    python tools/bench_quality.py [--seconds 2.0] > profiles/quality_b200.txt
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import _pkg  # noqa: E402
from bench_upscale import card, timed  # noqa: E402
from helpers import make_params  # noqa: E402

pkg = _pkg.load()
NETS = {"9-1-5 128/64": (128, 64, 9, 1, 5), "9-1-5 64/32": (64, 32, 9, 1, 5)}
N, w, h, S = 256, 960, 540, 2
W, H = S * w, S * h
HBM_PEAK = 7.7e12          # bytes/s, NVIDIA's HGX B200 data sheet, one GPU
FLOP_PX = (26 / 16 * 5 * 11 + 5 * 11) * 2 + 3 + 12


def kernel_rate(ctx, seconds):
    K, border = 32, 6
    rng = np.random.default_rng(11)
    frame = rng.integers(0, 256, (H, W, 4), dtype=np.uint8)
    mres, mref = ctx.alloc(K * W * H * 4), ctx.alloc(K * W * H * 4)
    for i in range(K):   # every frame its own bytes
        ctx.write(mres, np.roll(frame, i, 1), offset=i * W * H * 4)
        ctx.write(mref, np.roll(frame, 3 * i + 1, 0), offset=i * W * H * 4)
    out = ctx.alloc(16 * K)
    L, hctx = ctx.L, ctx.h
    for bpp in (3, 4):
        def call(reps=20):
            for _ in range(reps):
                pkg._check(L.srcnn_image_quality(hctx, mres, bpp, mref, W, H, K, border, out))
            ctx.block()

        call(2)
        ms, n = timed(call, seconds)
        per = ms / 20 / 1e3
        nbytes = K * W * H * (bpp + 4)
        flop = K * (W - 2 * border) * (H - 2 * border) * FLOP_PX
        print("quality kernel, %d frame pairs %dx%d, result %s: %.4f ms a call (%.4f ms a frame "
              "pair), %.0f GB/s = %.1f%% of %.1f TB/s HBM, %.2f TFLOP/s FP64 (%d x 20 calls)"
              % (K, W, H, "RGB8" if bpp == 3 else "RGBA8", per * 1e3, per * 1e3 / K,
                 nbytes / per / 1e9, 100 * nbytes / per / HBM_PEAK, HBM_PEAK / 1e12,
                 flop / per / 1e12, n))
    for m in (mres, mref, out):
        ctx.release(m)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=2.0)
    a = ap.parse_args()
    rng = np.random.default_rng(7)
    print("card (name, power limit): %s" % card())
    with pkg.Context(0) as ctx:
        print("device: %s, %d SMs" % ctx.device_info()[:2])
        src = pkg.PinnedBuffer((N, h, w, 4), np.uint8)
        ref = pkg.PinnedBuffer((N, H, W, 4), np.uint8)
        base = rng.integers(0, 256, (H, W, 4), dtype=np.uint8)
        for i in range(N):   # every frame different
            ref.array[i] = np.roll(base, 7 * i, 1)
            src.array[i] = ref.array[i, ::S, ::S]
        out_e = pkg.PinnedBuffer((N, H, W, 3), np.uint8)
        out_f = pkg.PinnedBuffer((N, H, W, 3), np.uint8)
        print("\n%d frames %dx%d -> %dx%d (x%d) with %dx%d RGBA8 references, pinned host "
              "buffers; ms a frame" % (N, w, h, W, H, S, W, H))
        for name, cfg in NETS.items():
            net = pkg.Net(ctx, *cfg, make_params(rng, *cfg))
            print("\n== %s ==" % name)
            for f in ("lanczos", "bicubic"):
                def evaluate():
                    return net.evaluate_frames_host(src.array, ref.array, W, H, f, out=out_e.array)

                def frames():
                    net.upscale_frames_host(src.array, W, H, f, out=out_f.array)

                _, met = evaluate()
                frames()
                same = np.array_equal(out_e.array, out_f.array)
                print("%s: evaluate entry's RGB8 == frames entry's, all %d frames: %s" % (f, N, same))
                assert same
                print("%s: mean network PSNR %.4f dB SSIM %.6f, baseline PSNR %.4f dB SSIM %.6f"
                      % (f, np.mean(10 * np.log10(1 / met[:, 0])), met[:, 1].mean(),
                         np.mean(10 * np.log10(1 / met[:, 2])), met[:, 3].mean()))
                res = {"frames entry": [], "evaluate entry": []}
                for _ in range(2):   # alternate the two entries
                    for label, fn in (("frames entry", frames), ("evaluate entry", evaluate)):
                        ms, n = timed(fn, a.seconds / 2)
                        res[label].append((ms / N, n))
                for label, r in res.items():
                    print("%s, %s: %s ms/frame (%s calls of %d frames)"
                          % (f, label, " / ".join("%.4f" % v for v, _ in r),
                             " / ".join(str(n) for _, n in r), N))
                fr = np.mean([v for v, _ in res["frames entry"]])
                ev = np.mean([v for v, _ in res["evaluate entry"]])
                print("%s: evaluation adds %.4f ms/frame (%.1f%%)" % (f, ev - fr, 100 * (ev - fr) / fr))
        print()
        kernel_rate(ctx, a.seconds)
        for b in (src, ref, out_e, out_f):
            b.free()
    print("\ncard after the run (name, power limit): %s" % card())


if __name__ == "__main__":
    main()

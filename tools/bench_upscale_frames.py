"""Wall clock per frame of the frames entry srcnn_upscale_frames_host (enlarge -> SRCNN -> RGB8 for
a set of frames) on pinned host buffers, next to the ways the same or similar work runs without
it, all in one process on one GPU:

  frames    Net.upscale_frames_host: 256 frames of 960x540 RGBA8 up, 1920x1080 RGB8 down (x2)
  loop      Net.upscale_image_host called once per frame on the same frames
  c5        Net.infer_frames_host on 256 float luma frames of 1920x1080 (BASELINE config C5's
            shape; float luma up and down)

for 9-1-5 128/64 and 64/32, Lanczos and bicubic.  Each timing is a host clock around whole
synchronous calls (all 256 frames), repeated for at least `--seconds` after a warm-up call of
every shape.  The frames entry's and the loop's results are compared byte for byte first.  The
pinned H2D / D2H copy rates are measured in the same run; a frame's copy floor is its bytes up /
H2D rate + bytes down / D2H rate (both directions one after the other), and the overlapped floor
the larger of the two terms.

    python tools/bench_upscale_frames.py [--seconds 2.0] > profiles/upscale_frames_b200.txt
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
from bench_upscale import card, copy_rates, timed  # noqa: E402
from helpers import make_params  # noqa: E402

pkg = _pkg.load()
NETS = {"9-1-5 128/64": (128, 64, 9, 1, 5), "9-1-5 64/32": (64, 32, 9, 1, 5)}
N, w, h, S = 256, 960, 540, 2
W, H = S * w, S * h


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=2.0)
    a = ap.parse_args()
    rng = np.random.default_rng(7)
    print("card (name, power limit): %s" % card())
    with pkg.Context(0) as ctx:
        print("device: %s, %d SMs" % ctx.device_info()[:2])
        h2d, d2h = copy_rates(ctx, a.seconds)
        print("pinned copy rates (64 MiB, one direction at a time): H2D %.1f GB/s, D2H %.1f GB/s"
              % (h2d, d2h))
        src = pkg.PinnedBuffer((N, h, w, 4), np.uint8)
        for i in range(N):   # every frame different (its own Q1 mean)
            src.array[i] = rng.integers(0, 256 - i // 2, (h, w, 4), dtype=np.uint8)
        dst = pkg.PinnedBuffer((N, H, W, 3), np.uint8)
        ref = pkg.PinnedBuffer((N, H, W, 3), np.uint8)
        lin = pkg.PinnedBuffer((N, H, W), np.float32)
        base = rng.uniform(-0.5, 0.5, (H, W)).astype(np.float32)
        for i in range(N):
            lin.array[i] = base + np.float32(i * 1e-3)
        up_rgb, down_rgb = w * h * 4, W * H * 3
        print("\n%d frames %dx%d -> %dx%d (x%d), pinned host buffers; per frame: ms, output "
              "MPix/s, PCIe bytes, copy floor" % (N, w, h, W, H, S))
        for name, cfg in NETS.items():
            net = pkg.Net(ctx, *cfg, make_params(rng, *cfg))
            (_, _), (_, _), (w3, h3) = net.out_dims(W, H)
            lout = pkg.PinnedBuffer((N, h3, w3), np.float32)
            print("\n== %s ==" % name)
            for f in ("lanczos", "bicubic"):
                def frames():
                    net.upscale_frames_host(src.array, W, H, f, out=dst.array)

                def loop():
                    for i in range(N):
                        net.upscale_image_host(src.array[i], W, H, f, out=ref.array[i])

                frames()
                loop()
                same = np.array_equal(dst.array, ref.array)
                print("%s: frames entry == per-frame loop, all %d frames: %s" % (f, N, same))
                assert same
                floor_s = up_rgb / h2d / 1e6 + down_rgb / d2h / 1e6
                floor_o = max(up_rgb / h2d / 1e6, down_rgb / d2h / 1e6)
                for label, fn in (("frames entry", frames), ("image-entry loop", loop)):
                    ms, n = timed(fn, a.seconds)
                    per = ms / N
                    print("%s, %s: %.4f ms/frame (%d calls of %d frames), %.0f MPix/s out, PCIe "
                          "%.2f MB up + %.2f MB down, copy floor %.4f ms (overlapped %.4f ms)"
                          % (f, label, per, n, N, W * H / per / 1e3, up_rgb / 1e6,
                             down_rgb / 1e6, floor_s, floor_o))
            net.infer_frames_host(lin.array, W, H, lout.array)
            ms, n = timed(lambda: net.infer_frames_host(lin.array, W, H, lout.array), a.seconds)
            per = ms / N
            up_f, down_f = W * H * 4, w3 * h3 * 4
            print("c5 infer_frames_host, float luma %dx%d: %.4f ms/frame (%d calls of %d frames), "
                  "%.0f MPix/s out, PCIe %.2f MB up + %.2f MB down, copy floor %.4f ms "
                  "(overlapped %.4f ms)"
                  % (W, H, per, n, N, w3 * h3 / per / 1e3, up_f / 1e6, down_f / 1e6,
                     up_f / h2d / 1e6 + down_f / d2h / 1e6, max(up_f / h2d, down_f / d2h) / 1e6))
            lout.free()
        for b in (src, dst, ref, lin):
            b.free()
        print("\ncard after the run (name, power limit): %s" % card())


if __name__ == "__main__":
    main()

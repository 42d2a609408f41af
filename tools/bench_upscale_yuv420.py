"""Wall clock per frame of the I420 frames entry srcnn_upscale_yuv420_frames_host (planar 4:2:0
video in and out) next to the RGBA8 frames entry srcnn_upscale_frames_host on the same content, on
pinned host buffers, all in one process on one GPU:

  yuv420    Net.upscale_yuv420_frames_host: 256 I420 frames of 960x540 up, 1920x1080 I420 down (x2)
  rgba      Net.upscale_frames_host: the same frames as RGBA8 (JFIF Y'CbCr -> RGB, chroma repeated
            2x2) up, 1920x1080 RGB8 down

for 9-1-5 128/64 and 64/32, Lanczos and bicubic.  Each timing is a host clock around whole
synchronous calls (all 256 frames), repeated for at least `--seconds` after a warm-up call of
every shape.  The pinned H2D / D2H copy rates are measured in the same run; an entry's copy floor
per frame is its own bytes up / H2D rate + bytes down / D2H rate (both directions one after the
other), and the overlapped floor the larger of the two terms.

    python tools/bench_upscale_yuv420.py [--seconds 2.0] > profiles/upscale_yuv420_b200.txt

`--trace DIR` instead runs one call of each entry for 9-1-5 64/32 (Lanczos) under torch.profiler
(a run of its own: tracing slows the host), writes DIR/<entry>.pt.trace.json and prints the device
time per kernel and copy direction.
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


def frames(rng, yuv, rgba):
    """smooth planes plus noise, every frame different (its own Q1 mean); rgba: the same frames
    through the JFIF conversion of swap_luma.cl"""
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    base = 110 + 80 * np.sin(xx / 23.0) * np.cos(yy / 17.0)
    for i in range(N):
        y = np.clip(base + i % 40 + rng.normal(0, 6, (h, w)), 0, 255).astype(np.uint8)
        cb = rng.integers(96, 160, (h // 2, w // 2), dtype=np.uint8)
        cr = rng.integers(96, 160, (h // 2, w // 2), dtype=np.uint8)
        yuv[i] = np.concatenate([y.ravel(), cb.ravel(), cr.ravel()])
        Y = y.astype(np.float32)
        Cb = np.repeat(np.repeat(cb, 2, 0), 2, 1).astype(np.float32) - 128
        Cr = np.repeat(np.repeat(cr, 2, 0), 2, 1).astype(np.float32) - 128
        rgb = np.stack([Y + 1.402 * Cr, Y - 0.344 * Cb - 0.714 * Cr, Y + 1.772 * Cb], -1)
        rgba[i, ..., :3] = np.clip(rgb, 0, 255).astype(np.uint8)
        rgba[i, ..., 3] = 255


def trace(ctx, net, calls, out_dir):
    import torch
    from torch.profiler import ProfilerActivity, profile
    os.makedirs(out_dir, exist_ok=True)
    for name, fn in calls:
        fn()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as p:
            fn()
            torch.cuda.synchronize()
        p.export_chrome_trace(os.path.join(out_dir, name + ".pt.trace.json"))
        print("\n== one call of the %s entry, 9-1-5 64/32, lanczos, %d frames ==" % (name, N))
        print(p.key_averages().table(sort_by="self_cuda_time_total", row_limit=14))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=2.0)
    ap.add_argument("--trace", default=None)
    a = ap.parse_args()
    rng = np.random.default_rng(7)
    print("card (name, power limit): %s" % card())
    with pkg.Context(0) as ctx:
        print("device: %s, %d SMs" % ctx.device_info()[:2])
        yuv_in = pkg.PinnedBuffer((N, w * h * 3 // 2), np.uint8)
        yuv_out = pkg.PinnedBuffer((N, W * H * 3 // 2), np.uint8)
        rgba_in = pkg.PinnedBuffer((N, h, w, 4), np.uint8)
        rgb_out = pkg.PinnedBuffer((N, H, W, 3), np.uint8)
        frames(rng, yuv_in.array, rgba_in.array)
        bytes_of = {"yuv420 entry": (w * h * 3 // 2, W * H * 3 // 2),
                    "rgba frames entry": (w * h * 4, W * H * 3)}
        if a.trace:
            cfg = NETS["9-1-5 64/32"]
            net = pkg.Net(ctx, *cfg, make_params(rng, *cfg))
            trace(ctx, net, [
                ("yuv420", lambda: net.upscale_yuv420_frames_host(yuv_in.array, w, h, W, H,
                                                                  out=yuv_out.array)),
                ("rgba", lambda: net.upscale_frames_host(rgba_in.array, W, H, out=rgb_out.array))],
                a.trace)
        else:
            h2d, d2h = copy_rates(ctx, a.seconds)
            print("pinned copy rates (64 MiB, one direction at a time): H2D %.1f GB/s, D2H %.1f GB/s"
                  % (h2d, d2h))
            print("\n%d frames %dx%d -> %dx%d (x%d), pinned host buffers; per frame: ms, output "
                  "MPix/s, PCIe bytes, copy floor" % (N, w, h, W, H, S))
            for name, cfg in NETS.items():
                net = pkg.Net(ctx, *cfg, make_params(rng, *cfg))
                print("\n== %s ==" % name)
                for f in ("lanczos", "bicubic"):
                    def yuv():
                        net.upscale_yuv420_frames_host(yuv_in.array, w, h, W, H, f, out=yuv_out.array)

                    def rgba():
                        net.upscale_frames_host(rgba_in.array, W, H, f, out=rgb_out.array)

                    for label, fn in (("yuv420 entry", yuv), ("rgba frames entry", rgba)):
                        up, down = bytes_of[label]
                        ms, n = timed(fn, a.seconds)
                        per = ms / N
                        print("%s, %s: %.4f ms/frame (%d calls of %d frames), %.0f MPix/s out, "
                              "PCIe %.2f MB up + %.2f MB down, copy floor %.4f ms (overlapped "
                              "%.4f ms)" % (f, label, per, n, N, W * H / per / 1e3, up / 1e6,
                                            down / 1e6, up / h2d / 1e6 + down / d2h / 1e6,
                                            max(up / h2d, down / d2h) / 1e6))
        for b in (yuv_in, yuv_out, rgba_in, rgb_out):
            b.free()
        print("\ncard after the run (name, power limit): %s" % card())


if __name__ == "__main__":
    main()

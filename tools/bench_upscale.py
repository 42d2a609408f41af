"""Wall clock of the image entry srcnn_upscale_image_host (enlarge -> SRCNN -> RGB8) on pinned host
buffers, next to the ways the same or similar work runs without it, all in one process on one GPU:

  upscale   Net.upscale_image_host: RGBA8 w x h up, RGB8 W x H down (s = 2 both filters, s = 3)
  rows      srcnn_infer_rows_host on a W x H float luma image (float luma up and down)
  unpiped   the existing calls one after another (upload, resample, extract_luma, sum read to the
            host, sub_from_all, forward, swap_luma) plus a full D2H of the RGB8 result
  resample  the resampling kernel alone (CUDA events), with its bytes per second

Each timing is a host clock around synchronous calls, over at least a second of calls after a
warm-up of every shape.  The pinned H2D / D2H copy rates are measured in the same run; the copy
floor of a call is its bytes up / H2D rate + bytes down / D2H rate.

    python tools/bench_upscale.py [--seconds 1.0] > profiles/upscale_b200.txt
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import _pkg  # noqa: E402
from helpers import make_params  # noqa: E402

pkg = _pkg.load()
CFG = (64, 32, 9, 1, 5)


def timed(fn, seconds):
    fn()
    n, t0 = 0, time.perf_counter()
    while True:
        fn()
        n += 1
        el = time.perf_counter() - t0
        if el >= seconds:
            return el / n * 1e3, n


def card():
    try:
        return subprocess.check_output(
            ["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
            text=True).strip().splitlines()[0]
    except Exception as e:   # the name still comes from the context below
        return "nvidia-smi unavailable (%s)" % e


def copy_rates(ctx, seconds):
    nbytes = 64 << 20
    pin = pkg.PinnedBuffer((nbytes,), np.uint8)
    m = ctx.alloc(nbytes)
    L, h, p = ctx.L, ctx.h, pkg.C.c_void_p(pin.ptr)
    up, _ = timed(lambda: pkg._check(L.srcnn_write(h, m, 0, nbytes, p, 1)), seconds)
    down, _ = timed(lambda: pkg._check(L.srcnn_read(h, m, 0, nbytes, p, 1)), seconds)
    ctx.release(m)
    pin.free()
    return nbytes / up / 1e6, nbytes / down / 1e6   # GB/s


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=1.0)
    a = ap.parse_args()
    rng = np.random.default_rng(7)
    print("card (name, power limit): %s" % card())
    with pkg.Context(0) as ctx:
        print("device: %s, %d SMs" % ctx.device_info()[:2])
        net = pkg.Net(ctx, *CFG, make_params(rng, *CFG))
        h2d, d2h = copy_rates(ctx, a.seconds)
        print("pinned copy rates (64 MiB, one direction at a time): H2D %.1f GB/s, D2H %.1f GB/s"
              % (h2d, d2h))
        cases = [(2048, 2048, 2, "lanczos"), (2048, 2048, 2, "bicubic"), (1365, 1365, 3, "lanczos")]
        bufs = {}
        for w, h, s, f in cases:   # warm every shape first
            W, H = s * w, s * h
            src = pkg.PinnedBuffer((h, w, 4), np.uint8)
            src.array[...] = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
            dst = pkg.PinnedBuffer((H, W, 3), np.uint8)
            bufs[(w, h, s, f)] = (src, dst)
            net.upscale_image_host(src.array, W, H, f, out=dst.array)
        print("\n== upscale_image_host (9-1-5 64/32, pinned) ==")
        for (w, h, s, f), (src, dst) in bufs.items():
            W, H = s * w, s * h
            ms, n = timed(lambda: net.upscale_image_host(src.array, W, H, f, out=dst.array),
                          a.seconds)
            up, down = w * h * 4, W * H * 3
            floor = up / h2d / 1e6 + down / d2h / 1e6
            print("%dx%d -> %dx%d (x%d, %s): %.3f ms/call (%d calls), %.0f MPix/s out, "
                  "PCIe %.1f MB up + %.1f MB down, copy floor %.3f ms = %.0f%% of the call"
                  % (w, h, W, H, s, f, ms, n, W * H / ms / 1e3, up / 1e6, down / 1e6, floor,
                     100 * floor / ms))
        print("\n== comparison at 4096x4096 output ==")
        W = H = 4096
        lin = pkg.PinnedBuffer((H, W), np.float32)
        lin.array[...] = rng.uniform(0, 1, (H, W)).astype(np.float32)
        (_, _), (_, _), (w3, h3) = net.out_dims(W, H)
        lout = pkg.PinnedBuffer((h3, w3), np.float32)
        ms, n = timed(lambda: net.infer_rows_host(lin.array, W, H, 0, h3, lout.array), a.seconds)
        print("infer_rows_host, float luma %dx%d: %.3f ms/call (%d calls), PCIe %.1f MB up + "
              "%.1f MB down" % (W, H, ms, n, W * H * 4 / 1e6, w3 * h3 * 4 / 1e6))
        src, dst = bufs[(2048, 2048, 2, "lanczos")]
        n_px = W * H
        ms_ = [ctx.alloc(2048 * 2048 * 4), ctx.alloc(n_px * 4), ctx.alloc(4 * n_px), ctx.alloc(4),
               ctx.alloc(4 * w3 * h3), ctx.alloc(3 * n_px)]
        mi, mb, ml, msum, mo, mr = ms_
        L, hh = ctx.L, ctx.h
        one = np.empty(1, np.float32)

        def unpiped():
            pkg._check(L.srcnn_write(hh, mi, 0, 2048 * 2048 * 4, pkg.C.c_void_p(src.ptr), 0))
            ctx.resample(mi, 2048, 2048, mb, W, H, "lanczos")
            ctx.extract_luma(mb, ml, W, H, True)
            ctx.sum(ml, n_px, True, msum)
            pkg._check(L.srcnn_read(hh, msum, 0, 4, pkg._np_ptr(one), 1))
            ctx.sub_from_all(ml, np.float32(one[0]) / np.float32(n_px), n_px)
            net.forward_fused(ml, mo, W, H, 1)
            ctx.swap_luma(mb, mo, mr, W, H, w3, h3)
            pkg._check(L.srcnn_read(hh, mr, 0, 3 * n_px, pkg.C.c_void_p(dst.ptr), 1))

        ms, n = timed(unpiped, a.seconds)
        print("existing calls one after another + full D2H (2048^2 -> 4096^2, lanczos): %.3f ms/call "
              "(%d calls)" % (ms, n))
        import torch
        for f in ("lanczos", "bicubic"):
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 200
            stream = torch.cuda.ExternalStream(ctx.stream())
            ctx.resample(mi, 2048, 2048, mb, W, H, f, ml)
            ctx.block()
            ev0.record(stream)
            for _ in range(reps):
                ctx.resample(mi, 2048, 2048, mb, W, H, f, ml)
            ev1.record(stream)
            ev1.synchronize()
            k_ms = ev0.elapsed_time(ev1) / reps
            nbytes = 2048 * 2048 * 4 + n_px * 8
            print("resample kernel alone (%s, 2048^2 -> 4096^2, RGBA + luma out): %.4f ms, "
                  "%.1f MB moved (%.0f GB/s)" % (f, k_ms, nbytes / 1e6, nbytes / k_ms / 1e6))
        for m in ms_:
            ctx.release(m)
        for src, dst in bufs.values():
            src.free()
            dst.free()
        lin.free()
        lout.free()


if __name__ == "__main__":
    main()

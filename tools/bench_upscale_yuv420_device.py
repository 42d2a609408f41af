"""Time per frame of the device-buffer 4:2:0 entry srcnn_upscale_yuv420_frames next to the host
entry srcnn_upscale_yuv420_frames_host on the same content, all in one process on one GPU:

  i420 dense      Net.upscale_yuv420_frames on 256 dense I420 frames of 960x540 -> 1920x1080
  nv12 dense      the same frames as dense NV12
  nv12 pitched    NV12 as decoders lay it out: 1024-byte input rows and 2048-byte output rows, the
                  CbCr plane after a 16-row-aligned Y plane (544 and 1088 rows)
  host entry      Net.upscale_yuv420_frames_host on pinned I420 buffers (upload, device work,
                  download; synchronous)
  ... left, ... topleft   i420 dense, nv12 pitched and the host entry with left- and top-left-sited
                  chroma kept as it is (chroma_siting of both layouts, of both host arguments):
                  the same launches and kernel with other chroma taps, so the same time is expected

for 9-1-5 128/64 and 64/32, Lanczos and bicubic (the frames of tools/bench_upscale_yuv420.py).
The device entry is timed with CUDA events on the context stream around `--reps` calls after a
warm-up call of every shape (its input and output, 0.2 GB and 0.8 GB, are larger than the L2);
the host entry with a host clock around whole synchronous calls.  The enqueue time is the host
time until one call returns (median of 20 calls, each followed by a synchronise).  The last lines
give the RGBA8 resampling kernel alone (ctx.resample, 2048^2 -> 4096^2, RGBA + luma out, CUDA
events), as tools/bench_upscale.py measures it, because the plane resampler took row pitches.

    python tools/bench_upscale_yuv420_device.py [--reps 20] [--seconds 2.0] \
        > profiles/chroma_siting_b200.txt
"""
import argparse
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import _pkg  # noqa: E402
from bench_upscale import card, timed  # noqa: E402
from bench_upscale_yuv420 import NETS, H, N, W, frames, h, w  # noqa: E402
from helpers import make_params  # noqa: E402

pkg = _pkg.load()


def nv12_of(i420, w, h, layout):
    """dense I420 frames [n][w*h*3//2] -> one buffer of NV12 frames in `layout`"""
    n = len(i420)
    ny, nc = w * h, (w // 2) * (h // 2)
    buf = np.zeros((n - 1) * layout.frame_stride + layout.frame_stride, np.uint8)
    for i, f in enumerate(i420):
        base = i * layout.frame_stride
        y = f[:ny].reshape(h, w)
        cbcr = np.stack([f[ny:ny + nc], f[ny + nc:]], -1).reshape(h // 2, w)
        for r in range(h):
            buf[base + r * layout.y_pitch:base + r * layout.y_pitch + w] = y[r]
        for r in range(h // 2):
            o = base + layout.cb_offset + r * layout.c_pitch
            buf[o:o + w] = cbcr[r]
    return buf


def event_ms(ctx, fn, reps):
    """CUDA-event time of one of `reps` calls of fn on the context stream"""
    import torch
    stream = torch.cuda.ExternalStream(ctx.stream())
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    ctx.block()
    ev0.record(stream)
    for _ in range(reps):
        fn()
    ev1.record(stream)
    ev1.synchronize()
    return ev0.elapsed_time(ev1) / reps


def enqueue_ms(ctx, fn):
    t = []
    for _ in range(20):
        t0 = time.perf_counter()
        fn()
        t.append(time.perf_counter() - t0)
        ctx.block()
    return statistics.median(t) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--seconds", type=float, default=2.0)
    a = ap.parse_args()
    rng = np.random.default_rng(7)
    print("card (name, power limit): %s" % card())
    with pkg.Context(0) as ctx:
        print("device: %s, %d SMs" % ctx.device_info()[:2])
        yuv_in = pkg.PinnedBuffer((N, w * h * 3 // 2), np.uint8)
        yuv_out = pkg.PinnedBuffer((N, W * H * 3 // 2), np.uint8)
        frames(rng, yuv_in.array, np.empty((N, h, w, 4), np.uint8))
        Lay = pkg.yuv420_layout
        def nv12_pitched(s):
            return ("nv12", Lay("nv12", w, h, 1024, 1024, 544 * 1024, chroma_siting=s),
                    Lay("nv12", W, H, 2048, 2048, 1088 * 2048, chroma_siting=s))

        layouts = {
            "i420 dense": ("i420", Lay("i420", w, h), Lay("i420", W, H)),
            "nv12 dense": ("nv12", Lay("nv12", w, h), Lay("nv12", W, H)),
            "nv12 pitched": nv12_pitched("center"),
        }
        for s in ("left", "topleft"):
            layouts["i420 dense " + s] = ("i420", Lay("i420", w, h, chroma_siting=s),
                                          Lay("i420", W, H, chroma_siting=s))
            layouts["nv12 pitched " + s] = nv12_pitched(s)
        mems = {}
        for label, (fmt, li, lo) in layouts.items():
            src = yuv_in.array.reshape(-1) if fmt == "i420" else nv12_of(yuv_in.array, w, h, li)
            mems[label] = (ctx.upload(src, np.uint8), ctx.alloc(N * lo.frame_stride))
        print("\n%d frames %dx%d -> %dx%d; ms per frame (device entry: CUDA events over %d calls; "
              "host entry: host clock over >= %.1f s of calls, pinned buffers)" % (N, w, h, W, H,
                                                                                  a.reps, a.seconds))
        for name, cfg in NETS.items():
            net = pkg.Net(ctx, *cfg, make_params(rng, *cfg))
            print("\n== %s ==" % name)
            for f in ("lanczos", "bicubic"):
                host = {}
                for s in ("center", "left", "topleft"):
                    host[s] = net.upscale_yuv420_frames_host(yuv_in.array, w, h, W, H, f,
                                                             out=yuv_out.array,
                                                             chroma_siting=s).copy()
                sitings = {v: k for k, v in pkg.CHROMA_SITINGS.items()}
                for label, (fmt, li, lo) in layouts.items():
                    m_in, m_out = mems[label]

                    def call():
                        net.upscale_yuv420_frames(m_in, w, h, N, m_out, W, H, f, fmt, li, lo)

                    ms = event_ms(ctx, call, a.reps)
                    enq = enqueue_ms(ctx, call)
                    same = ""
                    if fmt == "i420":   # the bytes are the host entry's
                        got = ctx.read(m_out, (N, W * H * 3 // 2), np.uint8)
                        same = ", bytes == host entry: %s" % np.array_equal(
                            got, host[sitings[li.chroma_siting]])
                    print("%s, device entry %s: %.4f ms/frame, enqueue of one call %.3f ms%s"
                          % (f, label, ms / N, enq, same))
                ms, n = timed(lambda: net.upscale_yuv420_frames_host(yuv_in.array, w, h, W, H, f,
                                                                     out=yuv_out.array), a.seconds)
                print("%s, host entry (pinned): %.4f ms/frame (%d calls of %d frames)"
                      % (f, ms / N, n, N))
                ms, n = timed(lambda: net.upscale_yuv420_frames_host(
                    yuv_in.array, w, h, W, H, f, out=yuv_out.array, chroma_siting="left"), a.seconds)
                print("%s, host entry left (pinned): %.4f ms/frame (%d calls of %d frames)"
                      % (f, ms / N, n, N))
        for m_in, m_out in mems.values():
            ctx.release(m_in)
            ctx.release(m_out)
        yuv_in.free()
        yuv_out.free()
        print("\n== RGBA8 resampling kernel alone (ctx.resample, 2048^2 -> 4096^2, RGBA + luma out) ==")
        n_px = 4096 * 4096
        mi, mb, ml = ctx.alloc(2048 * 2048 * 4), ctx.alloc(n_px * 4), ctx.alloc(n_px * 4)
        for f in ("lanczos", "bicubic"):
            k = event_ms(ctx, lambda: ctx.resample(mi, 2048, 2048, mb, 4096, 4096, f, ml), 200)
            print("%s: %.4f ms" % (f, k))
        for m in (mi, mb, ml):
            ctx.release(m)
    print("\ncard after the run (name, power limit): %s" % card())


if __name__ == "__main__":
    main()

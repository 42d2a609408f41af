"""Time per frame of the 10-bit 4:2:0 entries next to the 8-bit ones on the same content, all in
one process on one GPU:

  i420 / nv12 dense        the 8-bit device entry (srcnn_upscale_yuv420_frames) on dense frames
  nv12 pitched             8-bit NV12 as decoders lay it out: 1024-byte input rows and 2048-byte
                           output rows, the CbCr plane after a 16-row-aligned Y plane
  host entry               srcnn_upscale_yuv420_frames_host on pinned I420 buffers
  i010 / p010 dense        the device entry with bit_depth 10 on dense I010 and P010 frames
  i010 / p010 pitched      the same as decoders lay it out: 2048-byte input rows and 4096-byte
                           output rows, the chroma after a 16-row-aligned Y plane
  host entry 10-bit        srcnn_upscale_yuv420p10_frames_host on pinned I010 buffers (twice the
                           bytes of the 8-bit host entry each way)

for 256 frames of 960x540 -> 1920x1080, 9-1-5 128/64 and 64/32, Lanczos and bicubic.  The 10-bit
frames are the 8-bit ones of tools/bench_upscale_yuv420.py widened to 10 bits (v << 2 | v >> 6).
The device entry is timed with CUDA events on the context stream around `--reps` calls after a
warm-up call (its input and output are larger than the L2), the host entries with a host clock
around whole synchronous calls.  Each 10-bit device result is also compared with the 10-bit host
entry's words.

    python tools/bench_upscale_yuv420p10.py [--reps 20] [--seconds 2.0] \\
        > profiles/upscale_yuv420p10_b200.txt
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
from bench_upscale_yuv420 import NETS, H, N, W, frames, h, w  # noqa: E402
from bench_upscale_yuv420_device import event_ms, nv12_of  # noqa: E402
from helpers import make_params  # noqa: E402

pkg = _pkg.load()


def frame_index(layout, w, h, b):
    """the sample index, in units of b bytes, of every sample of one dense I420 frame in a frame
    of `layout` (NV12 / P010: Cb and Cr interleaved)"""
    nv12 = layout.format == pkg.YUV420_FORMATS["nv12"]
    yp, cp, cbo, cro = (v // b for v in (layout.y_pitch, layout.c_pitch, layout.cb_offset,
                                         layout.cr_offset))
    ys, xs = np.mgrid[0:h, 0:w]
    cy, cx = np.mgrid[0:h // 2, 0:w // 2]
    cb = cbo + cy * cp + (2 * cx if nv12 else cx)
    cr = cb + 1 if nv12 else cro + cy * cp + cx
    return np.concatenate([(ys * yp + xs).ravel(), cb.ravel(), cr.ravel()])


def pack10(values, layout, w, h):
    """dense 10-bit frames [n][w*h*3//2] -> one buffer of words in `layout` (P010: v << 6)"""
    shift = 6 if layout.format == pkg.YUV420_FORMATS["nv12"] else 0
    stride = layout.frame_stride // 2
    buf = np.zeros(len(values) * stride, np.uint16)
    idx = frame_index(layout, w, h, 2)
    for i, f in enumerate(values):
        buf[i * stride + idx] = f << shift
    return buf


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
        v8 = yuv_in.array.astype(np.uint16)
        p10_in = pkg.PinnedBuffer((N, w * h * 3 // 2), np.uint16)
        p10_out = pkg.PinnedBuffer((N, W * H * 3 // 2), np.uint16)
        p10_in.array[...] = (v8 << 2) | (v8 >> 6)
        Lay = pkg.yuv420_layout

        def pitched(fmt, bits, bi, bo):
            return (fmt, bits, Lay(fmt, w, h, bi, bi, -(-h // 16) * 16 * bi, bit_depth=bits),
                    Lay(fmt, W, H, bo, bo, -(-H // 16) * 16 * bo, bit_depth=bits))

        layouts = {
            "i420 dense": ("i420", 8, Lay("i420", w, h), Lay("i420", W, H)),
            "nv12 dense": ("nv12", 8, Lay("nv12", w, h), Lay("nv12", W, H)),
            "nv12 pitched": pitched("nv12", 8, 1024, 2048),
            "i010 dense": ("i420", 10, Lay("i420", w, h, bit_depth=10), Lay("i420", W, H, bit_depth=10)),
            "p010 dense": ("nv12", 10, Lay("nv12", w, h, bit_depth=10), Lay("nv12", W, H, bit_depth=10)),
            "i010 pitched": pitched("i420", 10, 2048, 4096),
            "p010 pitched": pitched("nv12", 10, 2048, 4096),
        }
        mems = {}
        for label, (fmt, bits, li, lo) in layouts.items():
            if bits == 8:
                src = yuv_in.array.reshape(-1) if fmt == "i420" else nv12_of(yuv_in.array, w, h, li)
                m_in = ctx.upload(src, np.uint8)
            else:
                m_in = ctx.upload(pack10(p10_in.array, li, w, h), np.uint16)
            mems[label] = (m_in, ctx.alloc(N * lo.frame_stride))
        print("\n%d frames %dx%d -> %dx%d; ms per frame (device entry: CUDA events over %d calls; "
              "host entries: host clock over >= %.1f s of calls, pinned buffers)"
              % (N, w, h, W, H, a.reps, a.seconds))
        for name, cfg in NETS.items():
            net = pkg.Net(ctx, *cfg, make_params(rng, *cfg))
            print("\n== %s ==" % name)
            for f in ("lanczos", "bicubic"):
                ref10 = net.upscale_yuv420p10_frames_host(p10_in.array, w, h, W, H, f,
                                                          out=p10_out.array).copy()
                for label, (fmt, bits, li, lo) in layouts.items():
                    m_in, m_out = mems[label]

                    def call():
                        net.upscale_yuv420_frames(m_in, w, h, N, m_out, W, H, f, fmt, li, lo)

                    ms = event_ms(ctx, call, a.reps)
                    same = ""
                    if bits == 10:
                        got = ctx.read(m_out, (N * lo.frame_stride // 2,), np.uint16)
                        idx = frame_index(lo, W, H, 2)
                        shift = 6 if fmt == "nv12" else 0
                        ok = all(np.array_equal(got[i * lo.frame_stride // 2 + idx] >> shift, ref10[i])
                                 for i in range(N))
                        same = ", words == 10-bit host entry: %s" % ok
                    print("%s, device entry %s: %.4f ms/frame%s" % (f, label, ms / N, same))
                ms, n = timed(lambda: net.upscale_yuv420_frames_host(yuv_in.array, w, h, W, H, f,
                                                                     out=yuv_out.array), a.seconds)
                print("%s, host entry 8-bit (pinned): %.4f ms/frame (%d calls of %d frames)"
                      % (f, ms / N, n, N))
                ms, n = timed(lambda: net.upscale_yuv420p10_frames_host(
                    p10_in.array, w, h, W, H, f, out=p10_out.array), a.seconds)
                print("%s, host entry 10-bit (pinned): %.4f ms/frame (%d calls of %d frames)"
                      % (f, ms / N, n, N))
        for m_in, m_out in mems.values():
            ctx.release(m_in)
            ctx.release(m_out)
        for b in (yuv_in, yuv_out, p10_in, p10_out):
            b.free()
    print("\ncard after the run (name, power limit): %s" % card())


if __name__ == "__main__":
    main()

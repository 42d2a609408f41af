"""A/B of the RGBA8 resampling kernel (srcnn_resample, 2048^2 -> 4096^2, RGBA + luma out) between
two builds of the library, e.g. the parent commit's and this tree's: each library runs in a fresh
process of its own, alternating, `--rounds` times, and reports CUDA-event time per launch over
`--reps` launches after a warm-up launch.  Only entries every build has are called (raw ctypes,
not the Python binding), so an older library needs no matching binding.  The working set (16 MB
in, 64 + 64 MB out) is larger than the 126 MB L2.

    python tools/ab_resample.py OTHER.so [THIS.so] [--rounds 4] [--reps 400]

THIS.so defaults to the library this tree builds.
"""
import argparse
import ctypes as C
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W_IN, W_OUT = 2048, 4096


def one(lib, reps):
    """times both filters with one library in this process; prints 'lanczos T bicubic T'"""
    import torch
    L = C.CDLL(lib)
    vp, u64 = C.c_void_p, C.c_uint64
    L.srcnn_ctx_create.argtypes = [C.c_int, C.c_int, C.POINTER(vp)]
    L.srcnn_alloc.argtypes = [vp, C.c_size_t, C.POINTER(u64)]
    L.srcnn_resample.argtypes = [vp, u64, C.c_int, C.c_int, u64, u64, C.c_int, C.c_int, C.c_int]
    L.srcnn_stream.argtypes = [vp, C.POINTER(vp)]
    L.srcnn_block.argtypes = [vp]
    L.srcnn_ctx_destroy.argtypes = [vp]
    ctx, stream = vp(), vp()
    assert L.srcnn_ctx_create(0, 0, C.byref(ctx)) == 0
    assert L.srcnn_stream(ctx, C.byref(stream)) == 0
    mems = []
    for nbytes in (W_IN * W_IN * 4, W_OUT * W_OUT * 4, W_OUT * W_OUT * 4):
        m = u64()
        assert L.srcnn_alloc(ctx, nbytes, C.byref(m)) == 0
        mems.append(m.value)
    mi, mb, ml = mems
    s = torch.cuda.ExternalStream(stream.value)
    out = []
    for name, f in (("lanczos", 1), ("bicubic", 0)):
        def call():
            assert L.srcnn_resample(ctx, mi, W_IN, W_IN, mb, ml, W_OUT, W_OUT, f) == 0
        call()
        assert L.srcnn_block(ctx) == 0
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(s)
        for _ in range(reps):
            call()
        ev1.record(s)
        ev1.synchronize()
        out.append("%s %.4f" % (name, ev0.elapsed_time(ev1) / reps))
    L.srcnn_ctx_destroy(ctx)
    print(" ".join(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("other")
    ap.add_argument("this", nargs="?",
                    default=os.path.join(ROOT, "cnn-super-resolution_b200", "libsrcnn_b200.so"))
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--reps", type=int, default=400)
    ap.add_argument("--one", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.one:
        return one(a.one, a.reps)
    print("resample kernel, 2048^2 -> 4096^2, RGBA + luma out, ms per launch over %d launches"
          % a.reps)
    for rnd in range(a.rounds):
        for label, lib in (("other", a.other), ("this", a.this)):
            r = subprocess.run([sys.executable, __file__, a.other, "--one", lib, "--reps",
                                str(a.reps)], capture_output=True, text=True)
            print("round %d, %s (%s): %s" % (rnd, label, os.path.basename(lib),
                                             r.stdout.strip() or r.stderr.strip()[-400:]),
                  flush=True)


if __name__ == "__main__":
    main()

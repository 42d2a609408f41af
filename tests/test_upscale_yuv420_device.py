"""4:2:0 video frames in device memory: srcnn_upscale_yuv420_frames (Net.upscale_yuv420_frames)
on I420 and NV12 buffers with pitched rows.

A frame's bytes are defined as those of srcnn_upscale_yuv420_frames_host (tested against the
composed definition in test_upscale_yuv420.py; one small case here is checked against that
definition directly).  A layout is restated as the byte index, in the buffer, of every byte of the
dense I420 frames (`plane_index`), so that packing, unpacking and the bytes no plane covers follow
from one function."""
import os
import subprocess
import sys

import numpy as np
import pytest

import _pkg
from test_upscale import FILTERS, NETS, make_net
from test_upscale_frames import forward_launches
from test_upscale_yuv420 import CASES, expected, size_for, yuv_frames

pkg = _pkg.load()

SWITCHED = [k for k in ("SRCNN_FUSED_IMPL", "SRCNN_C5_IMPL", "SRCNN_B3_IMPL", "SRCNN_GW_IMPL",
                        "SRCNN_D1_IMPL") if os.environ.get(k)]
EINVAL, EHANDLE, ERANGE = -1, -4, -5


def plane_index(layout, w, h, n):
    """int64 [n][w*h*3//2]: where each byte of n dense I420 frames of w x h lies in a buffer of
    `layout` (NV12: Cb and Cr interleaved in the CbCr plane)"""
    nv12 = layout.format == pkg.YUV420_FORMATS["nv12"]
    ys, xs = np.mgrid[0:h, 0:w]
    cy, cx = np.mgrid[0:h // 2, 0:w // 2]
    y = ys * layout.y_pitch + xs
    if nv12:
        cb = layout.cb_offset + cy * layout.c_pitch + 2 * cx
        cr = cb + 1
    else:
        cb = layout.cb_offset + cy * layout.c_pitch + cx
        cr = layout.cr_offset + cy * layout.c_pitch + cx
    one = np.concatenate([y.ravel(), cb.ravel(), cr.ravel()]).astype(np.int64)
    return one[None, :] + layout.frame_stride * np.arange(n, dtype=np.int64)[:, None]


def needed(layout, w, h, n):
    """the bytes the header says a buffer must hold: (n - 1) * frame_stride + the frame's extent"""
    nv12 = layout.format == pkg.YUV420_FORMATS["nv12"]
    c_end = (h // 2 - 1) * layout.c_pitch + (w if nv12 else w // 2)
    ends = [(h - 1) * layout.y_pitch + w, layout.cb_offset + c_end]
    if not nv12:
        ends.append(layout.cr_offset + c_end)
    return (n - 1) * layout.frame_stride + max(ends)


def pack(frames, layout, w, h, fill):
    """dense I420 frames -> a buffer of `layout`, the bytes outside the planes set to `fill`"""
    n = len(frames)
    buf = np.array(fill, np.uint8) if np.ndim(fill) else np.full(needed(layout, w, h, n), fill, np.uint8)
    buf[plane_index(layout, w, h, n)] = frames
    return buf


def unpack(buf, layout, w, h, n):
    return buf[plane_index(layout, w, h, n)]


def outside(buf, layout, w, h, n):
    """the bytes of buf no plane covers"""
    keep = np.ones(buf.size, bool)
    keep[plane_index(layout, w, h, n).ravel()] = False
    return buf[keep]


def run_device(ctx, net, frames, w, h, W, H, filt, fmt="i420", li=None, lo=None, in_fill=0,
               out_fill=0):
    """frames through the device entry in the given layouts (dense by default): (the result
    unpacked to dense I420, the whole output buffer)"""
    n = len(frames)
    li = li or pkg.yuv420_layout(fmt, w, h)
    lo = lo or pkg.yuv420_layout(fmt, W, H)
    m_in = ctx.upload(pack(frames, li, w, h, in_fill), np.uint8)
    out0 = np.full(needed(lo, W, H, n), out_fill, np.uint8) if np.ndim(out_fill) == 0 else out_fill
    m_out = ctx.upload(out0, np.uint8)
    try:
        net.upscale_yuv420_frames(m_in, w, h, n, m_out, W, H, filt, fmt, li, lo)
        buf = ctx.read(m_out, (out0.size,), np.uint8)
    finally:
        ctx.release(m_in)
        ctx.release(m_out)
    return unpack(buf, lo, W, H, n), buf


def default_group(net, W, H, n):
    """the device entry's group size the header documents: ~128 MB of scratch per frame group"""
    env = int(os.environ.get("SRCNN_FRAMES_GROUP", "0") or 0)
    if not net.fused_supported():
        return 1
    npx = W * H
    red = 8 * min(-(-npx // 256), 1024) + 4
    frame = npx * 4 + (W - net.padding) * (H - net.padding) * 4 + red
    return min(env if env > 0 else max(1, (128 << 20) // frame), n)


@pytest.fixture(scope="module")
def ctx():
    with pkg.Context(0) as c:
        yield c


# ----------------------------------------------------------------------------- CPU

def test_layout_helper_defaults_are_dense():
    """yuv420_layout's defaults are the dense layouts the header gives"""
    w, h = 38, 46
    for fmt, c_pitch, cr in (("i420", w // 2, w * h * 5 // 4), ("nv12", w, 0)):
        l = pkg.yuv420_layout(fmt, w, h)
        assert (l.format, l.frame_stride, l.y_pitch, l.c_pitch, l.cb_offset, l.cr_offset) == \
            (pkg.YUV420_FORMATS[fmt], w * h * 3 // 2, w, c_pitch, w * h, cr)
        idx = plane_index(l, w, h, 3)
        assert np.array_equal(np.sort(idx.ravel()), np.arange(3 * w * h * 3 // 2))
    with pytest.raises(ValueError):
        pkg.yuv420_layout("p010", w, h)


# ----------------------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("net_name", list(NETS))
def test_device_matches_host_entry(ctx, net_name, case):
    """dense I420 and NV12 in device memory give the host entry's bytes, both filters"""
    net, _ = make_net(ctx, net_name)
    h, w, H, W, n = size_for(net, case)
    frames = yuv_frames(np.random.default_rng(list(CASES).index(case) + 700), n, h, w)
    if case.startswith("1080p") and net.fused_supported() and not os.environ.get("SRCNN_FRAMES_GROUP"):
        g = default_group(net, W, H, n)
        assert -(-n // g) >= 2 and n % g != 0, g
    for filt in FILTERS:
        exp = net.upscale_yuv420_frames_host(frames, w, h, W, H, filt)
        for fmt in ("i420", "nv12"):
            got, _ = run_device(ctx, net, frames, w, h, W, H, filt, fmt)
            for i in range(n):
                assert np.array_equal(got[i], exp[i]), (fmt, filt, i)


@pytest.mark.gpu
@pytest.mark.parametrize("net_name", list(NETS))
def test_device_matches_composed_definition(ctx, net_name):
    net, _ = make_net(ctx, net_name)
    h, w, H, W, n = size_for(net, "40x40_n2")
    frames = yuv_frames(np.random.default_rng(77), n, h, w)
    for filt in FILTERS:
        exp = expected(ctx, net, frames, w, h, W, H, filt)
        for fmt in ("i420", "nv12"):
            got, _ = run_device(ctx, net, frames, w, h, W, H, filt, fmt)
            assert np.array_equal(got, exp), (fmt, filt)


def pitched(fmt, w, h, extra_y, extra_c, gap, pitch=None):
    """rows wider than their bytes, chroma after a 16-row-aligned Y plane, a gap between frames"""
    nv12 = fmt == "nv12"
    y_pitch = pitch or w + extra_y
    c_pitch = pitch or (w if nv12 else w // 2) + extra_c
    cb = -(-h // 16) * 16 * y_pitch
    dense = pkg.yuv420_layout(fmt, w, h, y_pitch, c_pitch, cb)
    return pkg.yuv420_layout(fmt, w, h, y_pitch, c_pitch, cb, dense.frame_stride + gap)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["i420", "nv12"])
@pytest.mark.parametrize("net_name,case", [("915_64_32", "x3_n2"), ("955_64_32", "x3_n2"),
                                           ("915_64_32", "1080p_n10")])
def test_device_pitch_and_placement(ctx, net_name, case, fmt):
    """pitched rows (odd extra bytes for I420, even for NV12; 2048-byte rows at 1080p, as
    decoders lay them out), padding bytes of random content in the input, a sentinel in the
    output's: the planes are the dense result and every sentinel survives"""
    net, _ = make_net(ctx, net_name)
    h, w, H, W, n = size_for(net, case)
    rng = np.random.default_rng(91)
    frames = yuv_frames(rng, n, h, w)
    odd = fmt == "i420"
    big = case.startswith("1080p")
    li = pitched(fmt, w, h, 3 if odd else 6, 5 if odd else 10, 37 if odd else 38,
                 1024 if big else None)
    lo = pitched(fmt, W, H, 7 if odd else 4, 1 if odd else 2, 53 if odd else 64,
                 2048 if big else None)
    in_fill = rng.integers(0, 256, needed(li, w, h, n), dtype=np.uint8)
    out_fill = np.full(needed(lo, W, H, n) + 512, 0xA7, np.uint8)   # + bytes after the last plane
    for filt in FILTERS:
        dense, _ = run_device(ctx, net, frames, w, h, W, H, filt, fmt)
        got, buf = run_device(ctx, net, frames, w, h, W, H, filt, fmt, li, lo, in_fill, out_fill)
        assert np.array_equal(got, dense), filt
        rest = outside(buf, lo, W, H, n)
        assert rest.size > 512 and (rest == 0xA7).all(), (filt, int((rest != 0xA7).sum()))


@pytest.mark.gpu
def test_device_stream_order_and_graph_capture():
    """a context on a torch stream: a torch fill right before the call and a torch read right after
    it, with no synchronise between, see the call's order; a call captured with torch.cuda.graph
    (no host synchronisation, no allocation) replays on new input contents"""
    import torch
    s = torch.cuda.Stream()
    with pkg.Context(0, stream=s.cuda_stream) as c:
        h, w, H, W, n = 270, 480, 540, 960, 5
        rng = np.random.default_rng(5)
        for net_name in ("915_64_32", "955_64_32"):
            net, _ = make_net(c, net_name)
            for fmt in ("nv12", "i420"):
                li, lo = pitched(fmt, w, h, 64, 32, 0, 512 if fmt == "nv12" else None), \
                    pkg.yuv420_layout(fmt, W, H)
                sets = [yuv_frames(rng, n, h, w) for _ in range(3)]
                exps = [net.upscale_yuv420_frames_host(f, w, h, W, H) for f in sets]
                srcs = [torch.from_numpy(pack(f, li, w, h, 0)).cuda() for f in sets]
                t_in = torch.zeros(srcs[0].numel(), dtype=torch.uint8, device="cuda")
                t_out = torch.zeros(needed(lo, W, H, n), dtype=torch.uint8, device="cuda")
                torch.cuda.synchronize()
                m_in, m_out = c.wrap(t_in.data_ptr(), t_in.numel()), c.wrap(t_out.data_ptr(), t_out.numel())

                def call():
                    net.upscale_yuv420_frames(m_in, w, h, n, m_out, W, H, "lanczos", fmt, li, lo)

                with torch.cuda.stream(s):
                    t_in.copy_(srcs[0])
                    call()
                    res = t_out.clone()
                s.synchronize()
                assert np.array_equal(unpack(res.cpu().numpy(), lo, W, H, n), exps[0]), (net_name, fmt)
                if net.fused_supported():
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=s):
                        call()
                    for k in (1, 2):
                        with torch.cuda.stream(s):
                            t_in.copy_(srcs[k])
                            g.replay()
                            res = t_out.clone()
                        s.synchronize()
                        assert np.array_equal(unpack(res.cpu().numpy(), lo, W, H, n), exps[k]), k
                    del g
                c.release(m_in)
                c.release(m_out)


def check_launch_count(net_name):
    """launches of a repeated call == the header's formula, and 1 more after a parameter write"""
    with pkg.Context(0) as c:
        net, params = make_net(c, net_name)
        for (h, w, H, W, n) in ((20, 20, 40, 40, 3), (540, 960, 1080, 1920, 10)):
            frames = yuv_frames(np.random.default_rng(n), n, h, w)
            F = forward_launches(c, net, W, H)
            for fmt in ("i420", "nv12"):
                li, lo = pkg.yuv420_layout(fmt, w, h), pkg.yuv420_layout(fmt, W, H)
                m_in = c.upload(pack(frames, li, w, h, 0), np.uint8)
                m_out = c.alloc(needed(lo, W, H, n))
                call = lambda: net.upscale_yuv420_frames(m_in, w, h, n, m_out, W, H, "lanczos", fmt)
                call()
                before = c.launch_count()
                call()
                launches = c.launch_count() - before
                nv12 = fmt == "nv12"
                if net.fused_supported():
                    expect = -(-n // default_group(net, W, H, n)) * (5 + nv12 + F)
                else:
                    expect = n * (4 + F + 1 + nv12)
                assert launches == expect, (fmt, W, H, launches, expect)
                if net.fused_supported():
                    c.write(net.c.w[0], params["w1"])   # the packed operand image is rebuilt
                    before = c.launch_count()
                    call()
                    assert c.launch_count() - before == expect + 1, fmt
                c.block()
                c.release(m_in)
                c.release(m_out)


# SRCNN_FRAMES_GROUP as the test process started (other tests set it in-process, after the
# library has read it)
START_GROUP = os.environ.get("SRCNN_FRAMES_GROUP")


@pytest.mark.gpu
@pytest.mark.skipif(bool(SWITCHED), reason="launch counts assume the default kernel selection")
@pytest.mark.parametrize("net_name", ["915_64_32", "915_128_64", "955_64_32"])
def test_device_launch_count(net_name):
    """in a process of its own, so that the group size the library reads once per process is the
    one default_group computes"""
    env = {k: v for k, v in os.environ.items() if k != "SRCNN_FRAMES_GROUP"}
    if START_GROUP is not None:
        env["SRCNN_FRAMES_GROUP"] = START_GROUP
    tests = os.path.dirname(os.path.abspath(__file__))
    code = ("import sys; sys.path[:0] = [%r, %r]\nfrom test_upscale_yuv420_device import "
            "check_launch_count\ncheck_launch_count(%r)\nprint('OK')" % (os.path.dirname(tests),
                                                                          tests, net_name))
    r = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["i420", "nv12"])
def test_device_rejects_bad_arguments(ctx, fmt):
    """each rule of the header's error list returns its code before any launch, and the output
    buffer stays untouched"""
    net, _ = make_net(ctx, "915_64_32")
    L, pnet = ctx.L, pkg.C.byref(net.c)
    w, h, W, H, n = 10, 10, 20, 20, 2
    nv12 = fmt == "nv12"
    Lay = pkg.yuv420_layout
    li, lo = Lay(fmt, w, h), Lay(fmt, W, H)
    m_in = ctx.upload(np.zeros(needed(li, w, h, n) + 64, np.uint8), np.uint8)
    out_bytes = needed(lo, W, H, n) + 64
    m_out = ctx.upload(np.full(out_bytes, 7, np.uint8), np.uint8)
    base_in, base_out = ctx.mem_ptr(m_in), ctx.mem_ptr(m_out)

    def call(li=li, lo=lo, w=w, h=h, n=n, W=W, H=H, f=1, m_in=m_in, m_out=m_out, c=ctx.h, nt=pnet):
        return L.srcnn_upscale_yuv420_frames(c, nt, m_in, None if li is None else pkg.C.byref(li),
                                             w, h, n, m_out, None if lo is None else pkg.C.byref(lo),
                                             W, H, f)

    def mod(l, **kw):
        x = pkg.CYuv420Layout.from_buffer_copy(l)
        for k, v in kw.items():
            setattr(x, k, v)
        return x

    c_row, c_row_out = (w if nv12 else w // 2), (W if nv12 else W // 2)
    before = ctx.launch_count()
    cases = {
        # everything the host entry rejects
        "size": (call(W=9), EINVAL), "odd in": (call(w=9, li=Lay(fmt, 9, h)), EINVAL),
        "odd out": (call(H=21, lo=Lay(fmt, W, 21)), EINVAL), "shrink": (call(W=8), EINVAL),
        "filter": (call(f=5), EINVAL), "n=0": (call(n=0), EINVAL), "n<0": (call(n=-3), EINVAL),
        "null net": (call(nt=None), EINVAL), "too small": (call(W=12, H=12), EINVAL),
        # layouts and formats
        "null in layout": (call(li=None), EINVAL), "null out layout": (call(lo=None), EINVAL),
        "unknown format": (call(li=mod(li, format=2), lo=mod(lo, format=2)), EINVAL),
        "negative format": (call(li=mod(li, format=-1), lo=mod(lo, format=-1)), EINVAL),
        "mismatched": (call(lo=Lay("i420" if nv12 else "nv12", W, H)), EINVAL),
        "y pitch": (call(li=mod(li, y_pitch=w - 1)), EINVAL),
        "c pitch": (call(lo=mod(lo, c_pitch=c_row_out - 2)), EINVAL),
        "huge pitch": (call(lo=mod(lo, y_pitch=1 << 31)), EINVAL),
        "cb in y": (call(li=mod(li, cb_offset=w * h - 1)), EINVAL),
        "stride": (call(lo=mod(lo, frame_stride=lo.frame_stride - 1)), EINVAL),
        # unknown and short buffers
        "handle": (call(m_in=123456), EHANDLE),
        "short": (call(m_out=ctx.wrap(base_out, needed(lo, W, H, n) - 1)), ERANGE),
        "short pitched": (call(li=mod(li, frame_stride=li.frame_stride + 66)), ERANGE),
        # the same buffer, or overlapping views of it, as input and output
        "same": (call(m_in=m_out), EINVAL),
        "overlap": (call(m_in=ctx.wrap(base_out + out_bytes - needed(li, w, h, n) - 2,
                                       needed(li, w, h, n))), EINVAL),
    }
    if nv12:
        cases.update({
            "cr offset": (call(li=mod(li, cr_offset=1)), EINVAL),
            "odd c pitch": (call(li=mod(li, c_pitch=c_row + 1, frame_stride=li.frame_stride + 10)),
                            EINVAL),
            "odd plane": (call(li=mod(li, cb_offset=w * h + 1, frame_stride=li.frame_stride + 2)), EINVAL),
            "odd buffer": (call(m_in=ctx.wrap(base_in + 1, needed(li, w, h, n))), EINVAL),
            "odd stride": (call(lo=mod(lo, frame_stride=lo.frame_stride + 1)), EINVAL),
        })
    else:
        cases.update({
            "cr in cb": (call(li=mod(li, cr_offset=li.cb_offset + c_row)), EINVAL),
            "cr in y": (call(lo=mod(lo, cr_offset=10)), EINVAL),
        })
    got = {k: v[0] for k, v in cases.items()}
    assert got == {k: v[1] for k, v in cases.items()}, got
    assert ctx.launch_count() == before
    assert (ctx.read(m_out, (out_bytes,), np.uint8) == 7).all()
    # the null-context check, and a frame stride that only one frame never uses is accepted
    assert call(c=None) == EINVAL
    assert call(n=1, li=mod(li, frame_stride=0), lo=mod(lo, frame_stride=0)) == 0
    ctx.release(m_in)
    ctx.release(m_out)


@pytest.mark.gpu
@pytest.mark.parametrize("net_name", ["915_64_32", "955_64_32"])
def test_device_state_between_calls(ctx, net_name):
    """the device entry interleaved on one context with the host 4:2:0 and RGBA frames entries,
    at other sizes too: each gives its own bytes, call after call"""
    from test_upscale_frames import frames_of, per_frame
    net, _ = make_net(ctx, net_name)
    rng = np.random.default_rng(23)
    h, w, H, W = 90, 70, 256 + net.padding, 140
    frames, small = yuv_frames(rng, 5, h, w), yuv_frames(rng, 3, 20, 20)
    exp = net.upscale_yuv420_frames_host(frames, w, h, W, H)
    small_exp = net.upscale_yuv420_frames_host(small, 20, 20, 40, 40, "bicubic")
    rgba = frames_of(rng, 3, 20, 20)
    rgba_exp = per_frame(net, rgba, 40, 40, "bicubic")
    for _ in range(2):
        assert np.array_equal(run_device(ctx, net, frames, w, h, W, H, "lanczos", "nv12")[0], exp)
        assert np.array_equal(net.upscale_yuv420_frames_host(small, 20, 20, 40, 40, "bicubic"), small_exp)
        assert np.array_equal(run_device(ctx, net, small, 20, 20, 40, 40, "bicubic")[0], small_exp)
        assert np.array_equal(net.upscale_frames_host(rgba, 40, 40, "bicubic"), rgba_exp)
        assert np.array_equal(net.upscale_yuv420_frames_host(frames, w, h, W, H), exp)
        assert np.array_equal(run_device(ctx, net, frames, w, h, W, H, "lanczos", "i420")[0], exp)

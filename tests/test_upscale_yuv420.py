"""Planar Y'CbCr 4:2:0 video frames: srcnn_upscale_yuv420_frames_host
(Net.upscale_yuv420_frames_host) and `cnn -i IN.y4m`.

Per frame the result is defined by parts that are already tested: Pillow's enlargement of each
plane (oracle/resample.py), and for the interior of Y the existing device-layer calls on the
enlarged Y' / 255 (sum of squares, sub_from_all, forward_fused), converted to a byte as swap_luma
converts a pixel with zero chroma.  Every frame of a set has its own content, so that a frame,
plane or ring-slot mix-up shows."""
import os
import subprocess
import sys

import numpy as np
import pytest

import _pkg
from oracle import resample as R
from test_upscale import FILTERS, NETS, make_net, photo
from test_upscale_frames import forward_launches

pkg = _pkg.load()

SWITCHED = [k for k in ("SRCNN_FUSED_IMPL", "SRCNN_C5_IMPL", "SRCNN_B3_IMPL", "SRCNN_GW_IMPL",
                        "SRCNN_D1_IMPL") if os.environ.get(k)]

# (h, w, H, W, n_frames); H of the h3_* cases is + the network's padding: network-output heights
# either side of the sub-band threshold (256) of the image entry, even because 4:2:0 sizes are and
# the padding is; "1080p" gives the default group size at least 3 groups and a partial last one
# (see default_group)
CASES = {"40x40_n1": (20, 20, 40, 40, 1), "40x40_n2": (20, 20, 40, 40, 2),
         "h3_254_n2": (90, 70, 254, 140, 2), "h3_256_n2": (90, 70, 256, 140, 2),
         "same_size_n2": (54, 62, 54, 62, 2), "x3_n2": (30, 42, 90, 126, 2),
         "1080p_n10": (540, 960, 1080, 1920, 10)}


def yuv_frames(rng, n, h, w):
    """n different I420 frames [n][w*h*3//2]: the planes of a photo-like image"""
    out = []
    for i in range(n):
        rgb = photo(rng, h, w).astype(np.float32) / (1 + i % 3) + 7 * i
        y = np.clip(rgb @ np.float32([0.299, 0.587, 0.114]), 0, 255).astype(np.uint8)
        sub = rgb.reshape(h // 2, 2, w // 2, 2, 3).mean((1, 3))
        cb = np.clip(128 + sub @ np.float32([-0.1687, -0.3313, 0.5]), 0, 255).astype(np.uint8)
        cr = np.clip(128 + sub @ np.float32([0.5, -0.4187, -0.0813]), 0, 255).astype(np.uint8)
        out.append(np.concatenate([y.ravel(), cb.ravel(), cr.ravel()]))
    return np.stack(out)


def planes(frame, w, h):
    """(Y [h][w], Cb, Cr [h/2][w/2]) views of one I420 frame"""
    n, c = w * h, (w // 2) * (h // 2)
    return (frame[:n].reshape(h, w), frame[n:n + c].reshape(h // 2, w // 2),
            frame[n + c:].reshape(h // 2, w // 2))


def luma_byte(o3):
    """swap_luma's byte for a pixel with zero chroma: clamp(y * 255) truncated, in float32"""
    return np.clip(o3.astype(np.float32) * np.float32(255), 0, 255).astype(np.uint8)


def net_luma(ctx, net, big_y):
    """the network's output for an enlarged Y plane through the existing device-layer calls"""
    H, W = big_y.shape
    (w1, h1), (w2, h2), (w3, h3) = net.out_dims(W, H)
    n = W * H
    ml, ms = ctx.upload(big_y.astype(np.float32) / np.float32(255)), ctx.alloc(4)
    ctx.sum(ml, n, True, ms)
    s = ctx.read(ms, (1,))[0]
    ctx.sub_from_all(ml, np.float32(s) / np.float32(n), n)
    mo = ctx.alloc(4 * w3 * h3)
    scratch = [] if net.fused_supported() else [ctx.alloc(4 * w1 * h1 * net.n1),
                                                ctx.alloc(4 * w2 * h2 * net.n2)]
    net.forward_fused(ml, mo, W, H, 1, *scratch)
    o3 = ctx.read(mo, (h3, w3))
    for m in [ml, ms, mo] + scratch:
        ctx.release(m)
    return o3


def expected(ctx, net, frames, w, h, W, H, filt, enlarged=None):
    """the composed definition of every frame; `enlarged`: the planes of each frame enlarged by
    the restatement, when the caller has them already"""
    pad = net.padding // 2
    out = []
    for i, f in enumerate(frames):
        y, cb, cr = enlarged[i] if enlarged else enlarge(f, w, h, W, H, filt)
        y = y.copy()
        o3 = net_luma(ctx, net, y)
        y[pad:pad + o3.shape[0], pad:pad + o3.shape[1]] = luma_byte(o3)
        out.append(np.concatenate([y.ravel(), cb.ravel(), cr.ravel()]))
    return np.stack(out)


def enlarge(frame, w, h, W, H, filt):
    y, cb, cr = planes(frame, w, h)
    return (R.resize(y, W, H, filt), R.resize(cb, W // 2, H // 2, filt),
            R.resize(cr, W // 2, H // 2, filt))


def default_group(net, w, h, W, H, n):
    """the group size the header documents: ~128 MB of device staging per group"""
    env = int(os.environ.get("SRCNN_FRAMES_GROUP", "0") or 0)
    if not net.fused_supported():
        return 1
    pad = net.padding
    frame = 3 * (w * h * 3 // 2 + W * H * 3 // 2) + W * H * 4 + (W - pad) * (H - pad) * 4
    return min(env if env > 0 else max(1, (128 << 20) // frame), n, 21845)


def size_for(net, case):
    h, w, H, W, n = CASES[case]
    return h, w, H + (net.padding if case.startswith("h3_") else 0), W, n


@pytest.fixture(scope="module")
def ctx():
    with pkg.Context(0) as c:
        yield c


# the restated enlargements of a case's frames, shared by the networks (the 1080p ones are slow)
_ENLARGED = {}


def enlarged_for(case, frames, w, h, W, H, filt):
    key = (case, H, filt)
    if key not in _ENLARGED:
        _ENLARGED[key] = [enlarge(f, w, h, W, H, filt) for f in frames]
    return _ENLARGED[key]


# ----------------------------------------------------------------------------- CPU

def write_y4m(path, header, frames, marker=b"FRAME\n", tail=b""):
    with open(path, "wb") as fh:
        fh.write(header + b"\n")
        for f in frames:
            fh.write(marker + np.ascontiguousarray(f, np.uint8).tobytes())
        fh.write(tail)


def read_y4m(path):
    data = open(path, "rb").read()
    header, rest = data.split(b"\n", 1)
    tags = header.split(b" ")[1:]
    w = int([t for t in tags if t[:1] == b"W"][0][1:])
    h = int([t for t in tags if t[:1] == b"H"][0][1:])
    fb = w * h * 3 // 2
    frames = []
    while rest:
        assert rest[:6] == b"FRAME\n"
        frames.append(np.frombuffer(rest[6:6 + fb], np.uint8))
        rest = rest[6 + fb:]
    return header, np.stack(frames)


def test_cli_y4m_rejections(tmp_path):
    """every rejected header, frame marker, truncation and mode stops with one message before any
    device work"""
    from test_host_cpp import CNN, HOST, run
    pkg.build()
    subprocess.check_call(["make", "-C", HOST, "-s"])
    cfg = os.path.join(os.path.dirname(__file__), "golden", "ref_config", "config.json")
    frames = np.zeros((2, 24), np.uint8)   # 4x4 I420
    src = str(tmp_path / "in.y4m")
    cases = [
        (b"YUV4MPEG2 W4 H4 C420mpeg2", {}, "chroma siting 'C420mpeg2' is left-sited"),
        (b"YUV4MPEG2 W4 H4 C420paldv", {}, "chroma siting 'C420paldv' is left-sited"),
        (b"YUV4MPEG2 W4 H4 C444", {}, "colourspace 'C444' is not supported"),
        (b"YUV4MPEG2 W4 H4 C420p10", {}, "colourspace 'C420p10' is not supported"),
        (b"YUV4MPEG2 W4 H4 Cmono", {}, "colourspace 'Cmono' is not supported"),
        (b"YUV4MPEG2 W4 H4 It", {}, "interlacing 'It' is not supported"),
        (b"YUV4MPEG2 W4 H4 Ib", {}, "interlacing 'Ib' is not supported"),
        (b"YUV4MPEG2 W4 H4 Im", {}, "interlacing 'Im' is not supported"),
        (b"YUV4MPEG2 W5 H4", {}, "frame size 5x4 is odd"),
        (b"YUV4MPEG2 W4 H3", {}, "frame size 4x3 is odd"),
        (b"YUV4MPEG2 W4", {}, "the header gives no W or no H"),
        (b"P6 4 4 255", {}, "not a YUV4MPEG2 stream"),
        (b"YUV4MPEG2 W4 H4", {"marker": b"FRAMES\n"}, "frame 0 does not start with FRAME"),
        (b"YUV4MPEG2 W4 H4", {"tail": b"FRAMX\n" + bytes(24)}, "frame 2 does not start with FRAME"),
        (b"YUV4MPEG2 W4 H4", {"tail": b"FRAME\n" + bytes(23)}, "frame 2 is truncated"),
        (b"YUV4MPEG2 W4 H4", {"tail": b"FRAME"}, "frame 2 is truncated"),
    ]
    for header, kw, msg in cases:
        write_y4m(src, header, frames, **kw)
        r = run([CNN, "dry", "-c", cfg, "-i", src])
        assert r.returncode != 0 and msg in r.stdout, (header, kw, r.stdout)
        assert "no CUDA device" not in r.stdout and "GPU ERROR" not in r.stdout, r.stdout
    write_y4m(src, b"YUV4MPEG2 W4 H4", frames)
    for mode in ("train", "eval"):
        r = run([CNN, mode, "-c", cfg, "-i", src, "-o", str(tmp_path / "out")])
        assert r.returncode != 0 and "A .y4m input applies to the forward mode only" in r.stdout


# ----------------------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("net_name", list(NETS))
def test_yuv420_matches_composed_definition(ctx, net_name, case):
    net, _ = make_net(ctx, net_name)
    h, w, H, W, n = size_for(net, case)
    rng = np.random.default_rng(list(CASES).index(case) + 300)
    frames = yuv_frames(rng, n, h, w)
    if case.startswith("1080p") and net.fused_supported():
        g = default_group(net, w, h, W, H, n)
        if not os.environ.get("SRCNN_FRAMES_GROUP"):
            assert -(-n // g) >= 3 and n % g != 0, g
    for filt in FILTERS:
        got = net.upscale_yuv420_frames_host(frames, w, h, W, H, filt)
        exp = expected(ctx, net, frames, w, h, W, H, filt,
                       enlarged_for(case, frames, w, h, W, H, filt))
        assert got.shape == (n, W * H * 3 // 2)
        for i in range(n):
            assert np.array_equal(got[i], exp[i]), (filt, i, int(np.abs(got[i].astype(int) - exp[i]).max()))


@pytest.mark.gpu
@pytest.mark.parametrize("group", [1, 2])
def test_yuv420_ring_wrap_around(ctx, tmp_path, group):
    """7 frames through groups of 1 and 2 (SRCNN_FRAMES_GROUP is read once per process, so in a
    process of its own): every ring slot is reused, and the bytes are those of this process"""
    tests = os.path.dirname(os.path.abspath(__file__))
    code = r"""
import sys
import numpy as np
sys.path[:0] = [%r, %r]
import _pkg
from test_upscale import make_net
from test_upscale_yuv420 import yuv_frames
pkg = _pkg.load()
with pkg.Context(0) as ctx:
    for name in ("915_64_32", "915_128_64"):
        net, _ = make_net(ctx, name)
        frames = yuv_frames(np.random.default_rng(5), 7, 46, 38)
        for filt in ("lanczos", "bicubic"):
            np.save("%s/%%s_%%s.npy" %% (name, filt), net.upscale_yuv420_frames_host(frames, 38, 46, 90, 114, filt))
print("OK")
""" % (os.path.dirname(tests), tests, str(tmp_path))
    env = dict(os.environ, SRCNN_FRAMES_GROUP=str(group))
    r = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout
    frames = yuv_frames(np.random.default_rng(5), 7, 46, 38)
    for name in ("915_64_32", "915_128_64"):
        net, _ = make_net(ctx, name)
        for filt in ("lanczos", "bicubic"):
            got = np.load(str(tmp_path / ("%s_%s.npy" % (name, filt))))
            assert np.array_equal(got, net.upscale_yuv420_frames_host(frames, 38, 46, 90, 114, filt)), (name, filt)


def check_launch_count(net_name):
    """launches of a repeated call == the documented formula"""
    with pkg.Context(0) as c:
        net, _ = make_net(c, net_name)
        for (h, w, H, W, n) in ((20, 20, 40, 40, 3), (540, 960, 1080, 1920, 6)):
            frames = yuv_frames(np.random.default_rng(n), n, h, w)
            F = forward_launches(c, net, W, H)
            net.upscale_yuv420_frames_host(frames, w, h, W, H)
            before = c.launch_count()
            net.upscale_yuv420_frames_host(frames, w, h, W, H)
            launches = c.launch_count() - before
            if net.fused_supported():
                expect = -(-n // default_group(net, w, h, W, H, n)) * (5 + F)
            else:
                expect = n * (4 + F + 1)
            assert launches == expect, (W, H, launches, expect)


START_GROUP = os.environ.get("SRCNN_FRAMES_GROUP")


@pytest.mark.gpu
@pytest.mark.skipif(bool(SWITCHED), reason="launch counts assume the default kernel selection")
@pytest.mark.parametrize("net_name", ["915_64_32", "915_128_64", "955_64_32"])
def test_yuv420_launch_count(net_name):
    """in a process of its own, so that the group size the library reads once per process is the
    one default_group computes"""
    env = {k: v for k, v in os.environ.items() if k != "SRCNN_FRAMES_GROUP"}
    if START_GROUP is not None:
        env["SRCNN_FRAMES_GROUP"] = START_GROUP
    tests = os.path.dirname(os.path.abspath(__file__))
    code = ("import sys; sys.path[:0] = [%r, %r]\nfrom test_upscale_yuv420 import check_launch_count\n"
            "check_launch_count(%r)\nprint('OK')" % (os.path.dirname(tests), tests, net_name))
    r = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("net_name", ["915_64_32", "955_64_32"])
def test_yuv420_state_between_calls(ctx, net_name):
    from test_upscale_frames import frames_of, per_frame
    net, params = make_net(ctx, net_name)
    h, w, H, W = 90, 70, 256 + net.padding, 140
    rng = np.random.default_rng(21)
    frames = yuv_frames(rng, 5, h, w)
    first = net.upscale_yuv420_frames_host(frames, w, h, W, H)
    assert np.array_equal(net.upscale_yuv420_frames_host(frames, w, h, W, H), first)   # repeat
    assert np.array_equal(first, expected(ctx, net, frames, w, h, W, H, "lanczos"))
    # new weights through srcnn_write: the next call uses them
    new = {k: (v * np.float32(1.25)).astype(np.float32) for k, v in params.items()}
    for l in range(3):
        ctx.write(net.c.w[l], new["w%d" % (l + 1)])
        ctx.write(net.c.b[l], new["b%d" % (l + 1)])
    got = net.upscale_yuv420_frames_host(frames, w, h, W, H)
    exp = expected(ctx, net, frames, w, h, W, H, "lanczos")
    assert np.array_equal(got, exp) and not np.array_equal(got, first)
    # pinned and pageable host buffers give the same bytes
    pin_in, pin_out = pkg.PinnedBuffer(frames.shape, np.uint8), pkg.PinnedBuffer(exp.shape, np.uint8)
    try:
        pin_in.array[...] = frames
        for _ in range(2):
            net.upscale_yuv420_frames_host(pin_in.array, w, h, W, H, out=pin_out.array)
            assert np.array_equal(pin_out.array, exp)
    finally:
        pin_in.free()
        pin_out.free()
    # the RGBA frames and image entries interleaved with this one on one context, other sizes
    # too: each matches its own reference
    rgba = frames_of(rng, 3, 20, 20)
    rgba_exp = per_frame(net, rgba, 40, 40, "bicubic")
    image_exp = net.upscale_image_host(rgba[1], W, H)
    small = yuv_frames(rng, 3, 20, 20)
    small_exp = expected(ctx, net, small, 20, 20, 40, 40, "bicubic")
    for _ in range(2):
        assert np.array_equal(net.upscale_yuv420_frames_host(small, 20, 20, 40, 40, "bicubic"), small_exp)
        assert np.array_equal(net.upscale_frames_host(rgba, 40, 40, "bicubic"), rgba_exp)
        assert np.array_equal(net.upscale_yuv420_frames_host(frames, w, h, W, H), exp)
        assert np.array_equal(net.upscale_image_host(rgba[1], W, H), image_exp)
        assert np.array_equal(net.upscale_image_host(rgba[2], 40, 40, "bicubic"), rgba_exp[2])


@pytest.mark.gpu
def test_yuv420_rejects_bad_arguments(ctx):
    """each bad argument fails with SRCNN_EINVAL, and the output buffer stays untouched"""
    net, _ = make_net(ctx, "915_64_32")
    src = np.zeros((2, 10 * 10 * 3 // 2), np.uint8)
    out = np.full(2 * 40 * 40 * 3 // 2, 7, np.uint8)
    L, h, pnet = ctx.L, ctx.h, pkg.C.byref(net.c)

    def call(W, H, f, n=2, w=10, hh=10, src=pkg._np_ptr(src), dst=pkg._np_ptr(out), c=h, nt=pnet):
        return L.srcnn_upscale_yuv420_frames_host(c, nt, src, w, hh, n, W, H, f, dst)

    bad = [call(W, H, f) for W, H, f in ((9, 20, 1), (20, 9, 1), (12, 12, 0), (0, 20, 1),
                                        (70000, 70000, 1), (20, 20, 5), (20, 20, -1),
                                        (21, 20, 1), (20, 21, 1), (8, 20, 1))]
    bad += [call(20, 20, 1, w=9), call(20, 20, 1, hh=9), call(20, 20, 1, n=0),
            call(20, 20, 1, n=-3), call(20, 20, 1, src=None), call(20, 20, 1, dst=None),
            call(20, 20, 1, c=None), call(20, 20, 1, nt=None)]
    assert bad == [-1] * len(bad), bad
    assert (out == 7).all()
    with pytest.raises(pkg.SrcnnError):
        pkg._check(call(21, 20, 1))
    with pytest.raises(ValueError):
        net.upscale_yuv420_frames_host(src, 10, 10, 20, 20, "nearest")


@pytest.mark.gpu
@pytest.mark.parametrize("size", ["40x40_n1", "h3_256_n2"])
@pytest.mark.parametrize("net_name", ["915_64_32", "955_64_32"])
def test_yuv420_matches_oracle_chain(ctx, port, net_name, size):
    """the plain-C oracle's subtract_mean (Q1) and three layers on the restated enlargement of Y:
    chroma exact, Y within 1 on fewer than 0.1 % of the pixels"""
    from oracle.loader import NetState
    net, params = make_net(ctx, net_name, seed=9)
    h, w, H, W, n = size_for(net, size)
    frames = yuv_frames(np.random.default_rng(11), n, h, w)
    pad = net.padding
    for filt in FILTERS:
        got = net.upscale_yuv420_frames_host(frames, w, h, W, H, filt)
        for i, f in enumerate(frames):
            y, cb, cr = enlarge(f, w, h, W, H, filt)
            luma = y.astype(np.float32) / np.float32(255)
            port.subtract_mean(luma.reshape(-1), with_event=True)
            _, _, o3 = port.net_forward(NetState(*NETS[net_name], params), luma, W, H, 1)
            y = y.copy()
            y[pad // 2:H - pad // 2, pad // 2:W - pad // 2] = luma_byte(o3[0].reshape(H - pad, W - pad))
            gy, gcb, gcr = planes(got[i], W, H)
            assert np.array_equal(gcb, cb) and np.array_equal(gcr, cr), (filt, i)
            diff = np.abs(gy.astype(int) - y.astype(int))
            assert diff.max() <= 1 and (diff > 0).mean() < 1e-3, (filt, i, diff.max(), (diff > 0).mean())


@pytest.mark.gpu
@pytest.mark.parametrize("net_name", ["915_64_32", "955_64_32"])
def test_cnn_cli_y4m(ctx, tmp_path, net_name):
    """`cnn -i IN.y4m -o OUT.y4m --scale 2`: 70 frames (more than one batch of 64), the header's
    W and H doubled and its other tags copied, every frame byte-equal to the entry's; `dry` writes
    nothing"""
    from helpers import make_params
    from test_host_cpp import CNN, HOST, run, write_config, write_params
    pkg.build()
    subprocess.check_call(["make", "-C", HOST, "-s"])
    cfg = NETS[net_name]
    rng = np.random.default_rng(51)
    params = make_params(rng, *cfg)
    pfile, cfile = str(tmp_path / "params.json"), str(tmp_path / "config.json")
    write_params(pfile, params)
    write_config(cfile, cfg, pfile)
    h, w = 22, 18
    frames = yuv_frames(rng, 70, h, w)
    src, dst = tmp_path / "in.y4m", tmp_path / "out.y4m"
    write_y4m(src, b"YUV4MPEG2 W18 H22 F30000:1001 Ip A1:1 C420jpeg XYSCSS=420JPEG", frames,
              marker=b"FRAME Ixyz\n")
    r = run([CNN, "-c", cfile, "-i", str(src), "-o", str(dst), "--scale", "2", "--resample",
             "bicubic"])
    assert r.returncode == 0, r.stdout
    assert "Input video: " in r.stdout and "Video: 18x22, 70 frames" in r.stdout, r.stdout
    header, got = read_y4m(dst)
    assert header == b"YUV4MPEG2 W36 H44 F30000:1001 Ip A1:1 C420jpeg XYSCSS=420JPEG", header
    net = pkg.Net(ctx, *cfg, params)
    exp = net.upscale_yuv420_frames_host(frames, w, h, 2 * w, 2 * h, "bicubic")
    assert got.shape == exp.shape and np.array_equal(got, exp)
    os.remove(dst)
    r = run([CNN, "dry", "-c", cfile, "-i", str(src), "-o", str(dst)])
    assert r.returncode == 0 and not dst.exists() and "Saving result" not in r.stdout, r.stdout

"""10-bit 4:2:0 video frames: srcnn_upscale_yuv420p10_frames_host
(Net.upscale_yuv420p10_frames_host), srcnn_upscale_yuv420_frames on I010 and P010 buffers
(bit_depth 10 in the layouts) and `cnn -i IN.y4m --bit-depth 10`.

Per frame the result is defined by parts that are tested on their own: Pillow's 16-bit enlargement
of each plane, capped at 1023 (oracle/resample16.py, checked against Pillow's "I;16" resize here),
and for the interior of Y the existing device-layer calls on the enlarged v / 1023, written back as
clamp(out * 1023) truncated.  Inputs carry junk in the bits outside their 10-bit values, so that a
read that does not mask or shift them shows."""
import os
import subprocess
import sys

import numpy as np
import pytest

import _pkg
from oracle import resample16 as R16
from test_upscale import FILTERS, NETS, make_net, photo
from test_upscale_frames import forward_launches
from test_upscale_yuv420 import CASES, size_for, write_y4m
from test_upscale_yuv420_device import plane_index

pkg = _pkg.load()

SWITCHED = [k for k in ("SRCNN_FUSED_IMPL", "SRCNN_C5_IMPL", "SRCNN_B3_IMPL", "SRCNN_GW_IMPL",
                        "SRCNN_D1_IMPL") if os.environ.get(k)]
EINVAL = -1
SITING_NAMES = list(pkg.CHROMA_SITINGS)


def yuv10_frames(rng, n, h, w):
    """n different I010 frames [n][w*h*3//2] of values in [0, 1023]: the planes of a photo-like
    image, with a row and a column at each of the hard edges 0 and 1023"""
    out = []
    for i in range(n):
        rgb = photo(rng, h, w).astype(np.float32) * np.float32(4.0 / (1 + i % 3)) + 29 * i
        rgb += rng.integers(0, 4, rgb.shape)
        y = np.clip(rgb @ np.float32([0.299, 0.587, 0.114]), 0, 1023)
        sub = rgb.reshape(h // 2, 2, w // 2, 2, 3).mean((1, 3))
        cb = np.clip(512 + sub @ np.float32([-0.1687, -0.3313, 0.5]), 0, 1023)
        cr = np.clip(512 + sub @ np.float32([0.5, -0.4187, -0.0813]), 0, 1023)
        for p in (y, cb, cr):
            p[:, p.shape[1] // 3] = 1023
            p[p.shape[0] // 2, :] = 0
            p[:, -1] = 1023 * (i % 2)
        out.append(np.concatenate([y.ravel(), cb.ravel(), cr.ravel()]).astype(np.uint16))
    return np.stack(out)


def with_junk(rng, frames, shift=0):
    """the words of 10-bit values at bit `shift` (I010: 0, P010: 6) with every other bit random"""
    junk = rng.integers(0, 1 << 16, frames.shape, dtype=np.uint16) & np.uint16(~(0x3FF << shift) & 0xFFFF)
    return ((frames.astype(np.uint16) << shift) | junk).astype(np.uint16)


def planes10(frame, w, h):
    n, c = w * h, (w // 2) * (h // 2)
    return (frame[:n].reshape(h, w), frame[n:n + c].reshape(h // 2, w // 2),
            frame[n + c:].reshape(h // 2, w // 2))


def enlarge10(frame, w, h, W, H, filt, s_in="center", s_out="center"):
    y, cb, cr = planes10(frame, w, h)
    return (R16.resize10(y, W, H, filt),
            R16.resize10_sited(cb, W // 2, H // 2, filt, s_in, s_out),
            R16.resize10_sited(cr, W // 2, H // 2, filt, s_in, s_out))


def net_luma10(ctx, net, big_y):
    """the network's output for an enlarged 10-bit Y plane (its v / 1023) through the existing
    device-layer calls"""
    H, W = big_y.shape
    (w1, h1), (w2, h2), (w3, h3) = net.out_dims(W, H)
    n = W * H
    ml, ms = ctx.upload(big_y.astype(np.float32) / np.float32(1023)), ctx.alloc(4)
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


def luma_word(o3):
    """the 10-bit Y write: clamp(y * 1023, 0, 1023) truncated, in float32"""
    return np.clip(o3.astype(np.float32) * np.float32(1023), 0, 1023).astype(np.uint16)


def expected10(ctx, net, frames, w, h, W, H, filt, enlarged):
    """the composed definition of every frame from its restated planes `enlarged`"""
    pad = net.padding // 2
    out = []
    for y, cb, cr in enlarged:
        y = y.copy()
        o3 = net_luma10(ctx, net, y)
        y[pad:pad + o3.shape[0], pad:pad + o3.shape[1]] = luma_word(o3)
        out.append(np.concatenate([y.ravel(), cb.ravel(), cr.ravel()]))
    return np.stack(out)


def default_group10(net, w, h, W, H, n):
    """the host entry's group size: the 8-bit rule with every frame twice the bytes"""
    env = int(os.environ.get("SRCNN_FRAMES_GROUP", "0") or 0)
    if not net.fused_supported():
        return 1
    pad = net.padding
    frame = 3 * (w * h * 3 + W * H * 3) + W * H * 4 + (W - pad) * (H - pad) * 4
    return min(env if env > 0 else max(1, (128 << 20) // frame), n, 21845)


# 10-bit layouts in 16-bit words: plane_index and the byte counts of test_upscale_yuv420_device
# apply to them with every offset, pitch and stride halved
def in_words(layout):
    x = pkg.CYuv420Layout.from_buffer_copy(layout)
    for k in ("frame_stride", "y_pitch", "c_pitch", "cb_offset", "cr_offset"):
        assert getattr(x, k) % 2 == 0
        setattr(x, k, getattr(x, k) // 2)
    return x


def needed_words(layout, w, h, n):
    lw = in_words(layout)
    nv12 = lw.format == pkg.YUV420_FORMATS["nv12"]
    c_end = (h // 2 - 1) * lw.c_pitch + (w if nv12 else w // 2)
    ends = [(h - 1) * lw.y_pitch + w, lw.cb_offset + c_end] + ([] if nv12 else [lw.cr_offset + c_end])
    return (n - 1) * lw.frame_stride + max(ends)


def run_device10(ctx, net, frames, w, h, W, H, filt, fmt, rng, li=None, lo=None, out_fill=None,
                 s_in="center", s_out="center"):
    """10-bit frames (values) through the device entry as I010 ("i420") or P010 ("nv12"), the
    input's other bits and padding random: (the result's values as dense I010, the whole output
    buffer of words)"""
    n = len(frames)
    shift = 6 if fmt == "nv12" else 0
    li = li or pkg.yuv420_layout(fmt, w, h, chroma_siting=s_in, bit_depth=10)
    lo = lo or pkg.yuv420_layout(fmt, W, H, chroma_siting=s_out, bit_depth=10)
    buf = rng.integers(0, 1 << 16, needed_words(li, w, h, n), dtype=np.uint16)
    buf[plane_index(in_words(li), w, h, n)] = with_junk(rng, frames, shift)
    out0 = np.zeros(needed_words(lo, W, H, n), np.uint16) if out_fill is None else out_fill
    m_in, m_out = ctx.upload(buf, np.uint16), ctx.upload(out0, np.uint16)
    try:
        net.upscale_yuv420_frames(m_in, w, h, n, m_out, W, H, filt, fmt, li, lo)
        got = ctx.read(m_out, (out0.size,), np.uint16)
    finally:
        ctx.release(m_in)
        ctx.release(m_out)
    words = got[plane_index(in_words(lo), W, H, n)]
    assert (words & np.uint16(~(0x3FF << shift) & 0xFFFF) == 0).all(), "bits outside the value"
    return words >> shift, got


@pytest.fixture(scope="module")
def ctx():
    with pkg.Context(0) as c:
        yield c


# ----------------------------------------------------------------------------- CPU

def pillow_shapes(rng, count):
    """(h, w, H, W): ratio-1 axes, x2, x3 and uneven ratios"""
    fixed = [(7, 9, 7, 18), (6, 5, 18, 5), (8, 8, 8, 8), (5, 11, 10, 33), (9, 4, 23, 13)]
    for s in fixed:
        yield s
    for _ in range(count - len(fixed)):
        h, w = (int(v) for v in rng.integers(2, 30, 2))
        yield (h, w, h * int(rng.integers(1, 4)) + int(rng.integers(0, 3)),
               w * int(rng.integers(1, 4)) + int(rng.integers(0, 3)))


def i16(Image, a):
    """a uint16 plane as a Pillow "I;16" image"""
    im = Image.fromarray(a)
    assert im.mode == "I;16"
    return im


def edgy_plane(rng, h, w):
    a = rng.integers(0, 1024, (h, w)).astype(np.uint16)
    a[:, ::3] = 0
    a[::2, :] = np.where(rng.random(w) < 0.5, 1023, 0)
    return a


def test_restatement_matches_pillow_i16():
    """oracle/resample16.py equals Pillow's "I;16" resize, both filters, plain and with a box of a
    fractional start inside the image (the restatement given the box's scale as Pillow computes
    it: the box in single precision, the scale in double); capped at 1023 it is resize10"""
    Image = pytest.importorskip("PIL.Image")
    from test_chroma_siting import pillow_box
    rng = np.random.default_rng(1010)
    n = 0
    for h, w, H, W in pillow_shapes(rng, 40):
        a = edgy_plane(rng, h, w)
        x0, y0 = float(rng.uniform(0, 1)), float(rng.choice([0.0, 0.25, rng.uniform(0, 1)]))
        box = (x0, y0, w - float(rng.uniform(0, 0.5)), h - 0.25)
        for filt, f in (("bicubic", Image.BICUBIC), ("lanczos", Image.LANCZOS)):
            exp = np.asarray(i16(Image, a).resize((W, H), f))
            got = R16.resize_box(a, W, H, filt)
            assert got.dtype == np.uint16 and np.array_equal(got, exp), (h, w, H, W, filt)
            assert np.array_equal(R16.resize10(a, W, H, filt), np.minimum(exp, 1023))
            exp = np.asarray(i16(Image, a).resize((W, H), f, box=box))
            got = R16.resize_box(a, W, H, filt, *pillow_box(box, W, H))
            assert np.array_equal(got, exp), (h, w, H, W, box, filt)
            n += 2
    assert n == 160


def test_restatement_is_not_the_8bit_one():
    """on values that fit 8 bits the 16-bit path still differs from the 8-bit one somewhere (the
    weights are not rounded to 22 bits, the rounding is half away from zero), so a 10-bit entry
    that ran the 8-bit arithmetic would show"""
    from oracle import resample as R
    rng = np.random.default_rng(3)
    a = rng.integers(0, 256, (40, 40)).astype(np.uint8)
    diff = sum(int((R16.resize_box(a.astype(np.uint16), 113, 97, f) != R.resize(a, 113, 97, f)).sum())
               for f in FILTERS)
    assert diff > 0


def test_layout_helper_10bit_defaults():
    """yuv420_layout(..., bit_depth=10) is the dense I010 / P010 layout the header gives; other bit
    depths and a "p010" format name are refused"""
    w, h = 38, 46
    for fmt, c_pitch, cr in (("i420", w, 2 * w * h * 5 // 4), ("nv12", 2 * w, 0)):
        l = pkg.yuv420_layout(fmt, w, h, bit_depth=10)
        assert (l.format, l.frame_stride, l.y_pitch, l.c_pitch, l.cb_offset, l.cr_offset,
                l.chroma_siting, l.bit_depth) == \
            (pkg.YUV420_FORMATS[fmt], w * h * 3, 2 * w, c_pitch, 2 * w * h, cr, 0, 10)
        idx = plane_index(in_words(l), w, h, 3)
        assert np.array_equal(np.sort(idx.ravel()), np.arange(3 * w * h * 3 // 2))
        assert pkg.yuv420_layout(fmt, w, h).bit_depth == 8
    for bad in (0, 9, 12, 16):
        with pytest.raises(ValueError):
            pkg.yuv420_layout("i420", w, h, bit_depth=bad)
    with pytest.raises(ValueError):
        pkg.yuv420_layout("p010", w, h, bit_depth=10)


def test_cli_10bit_rejections(tmp_path):
    """C420p10 without --bit-depth 10 (the 8-bit message, then a hint), --bit-depth 10 on an 8-bit
    header, a --bit-depth other than 8 or 10, --bit-depth without a forward-mode .y4m input, a
    --chroma-siting a C420p10 tag cannot state, and a truncated 10-bit frame: one line each,
    before any device work; a complete C420p10 file with the flag passes the header and frame
    checks"""
    from helpers import make_params
    from test_host_cpp import CNN, HOST, run, write_config, write_params
    pkg.build()
    subprocess.check_call(["make", "-C", HOST, "-s"])
    pfile, cfg = str(tmp_path / "params.json"), str(tmp_path / "config.json")
    write_params(pfile, make_params(np.random.default_rng(1), *NETS["915_32_16"]))
    write_config(cfg, NETS["915_32_16"], pfile)
    src = str(tmp_path / "in.y4m")
    ten = np.zeros((2, 48), np.uint8)   # two 4x4 I010 frames
    cases = [
        (b"YUV4MPEG2 W4 H4 C420p10", ten, {}, [],
         "colourspace 'C420p10' is not supported; only 8-bit 4:2:0 (C420jpeg, C420) is; "
         "--bit-depth 10 reads 10-bit 4:2:0"),
        (b"YUV4MPEG2 W4 H4 C420p10", ten, {}, ["--bit-depth", "8"], "colourspace 'C420p10' is not"),
        (b"YUV4MPEG2 W4 H4 C420jpeg", ten[:, :24], {}, ["--bit-depth", "10"],
         "--bit-depth 10 needs a 10-bit (C420p10) input"),
        (b"YUV4MPEG2 W4 H4", ten[:, :24], {}, ["--bit-depth", "10"], "--bit-depth 10 needs a 10-bit"),
        (b"YUV4MPEG2 W4 H4 C420p10", ten, {}, ["--bit-depth", "10", "--chroma-siting", "420mpeg2"],
         "--chroma-siting must be keep or 420jpeg for a 10-bit input"),
        (b"YUV4MPEG2 W4 H4 C420p10", ten, {}, ["--bit-depth", "10", "--chroma-siting", "420paldv"],
         "--chroma-siting must be keep or 420jpeg for a 10-bit input"),
        (b"YUV4MPEG2 W4 H4 C420p10", ten, {"tail": b"FRAME\n" + bytes(47)}, ["--bit-depth", "10"],
         "frame 2 is truncated"),
        (b"YUV4MPEG2 W4 H4 C420p10", ten[:1, :24], {}, ["--bit-depth", "10"], "frame 0 is truncated"),
    ]
    for bad in ("9", "16", "", "ten"):
        cases.append((b"YUV4MPEG2 W4 H4 C420p10", ten, {}, ["--bit-depth", bad],
                      "--bit-depth must be 8 or 10, got '%s'" % bad))
    for header, frames, kw, opts, msg in cases:
        write_y4m(src, header, frames, **kw)
        r = run([CNN, "dry", "-c", cfg, "-i", src] + opts)
        assert r.returncode != 0 and msg in r.stdout, (header, opts, r.stdout)
        assert "no CUDA device" not in r.stdout and "GPU ERROR" not in r.stdout, r.stdout
    ppm = str(tmp_path / "in.ppm")
    with open(ppm, "wb") as f:
        f.write(b"P6 4 4 255\n" + bytes(48))
    for cmd in ([CNN, "dry", "-c", cfg, "-i", ppm, "--bit-depth", "10"],
                [CNN, "train", "-c", cfg, "-i", str(tmp_path), "-o", str(tmp_path / "p"),
                 "--bit-depth", "8"]):
        r = run(cmd)
        assert r.returncode != 0 and "--bit-depth applies to a .y4m input in the forward mode " \
            "only" in r.stdout, r.stdout
    write_y4m(src, b"YUV4MPEG2 W32 H32 C420p10", np.zeros((2, 32 * 32 * 3), np.uint8))
    for opts in ([], ["--chroma-siting", "keep"], ["--chroma-siting", "420jpeg"]):
        r = run([CNN, "dry", "-c", cfg, "-i", src, "--bit-depth", "10"] + opts)
        assert "Video: 32x32, 2 frames" in r.stdout, r.stdout
        assert r.returncode != 0 if "no CUDA device" in r.stdout else r.returncode == 0, r.stdout


# ----------------------------------------------------------------------------- GPU

# the restated enlargements of a case's frames, shared by the networks (the 1080p ones are slow)
_ENLARGED = {}


def enlarged_for(key, frames, w, h, W, H, filt, s_in="center", s_out="center"):
    key = key + (H, filt, s_in, s_out)
    if key not in _ENLARGED:
        _ENLARGED[key] = [enlarge10(f, w, h, W, H, filt, s_in, s_out) for f in frames]
    return _ENLARGED[key]


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("net_name", list(NETS))
def test_p10_host_matches_composed_definition(ctx, net_name, case):
    net, _ = make_net(ctx, net_name)
    h, w, H, W, n = size_for(net, case)
    rng = np.random.default_rng(list(CASES).index(case) + 1000)
    frames = yuv10_frames(rng, n, h, w)
    if case.startswith("1080p") and net.fused_supported() and not os.environ.get("SRCNN_FRAMES_GROUP"):
        g = default_group10(net, w, h, W, H, n)
        assert g == 3 and -(-n // g) >= 3 and n % g != 0, g
    src = with_junk(rng, frames)
    for filt in FILTERS:
        got = net.upscale_yuv420p10_frames_host(src, w, h, W, H, filt)
        exp = expected10(ctx, net, frames, w, h, W, H, filt,
                         enlarged_for((case,), frames, w, h, W, H, filt))
        assert got.dtype == np.uint16 and got.shape == (n, W * H * 3 // 2)
        for i in range(n):
            assert np.array_equal(got[i], exp[i]), (filt, i, int(np.abs(got[i].astype(int) - exp[i]).max()))


@pytest.mark.gpu
@pytest.mark.parametrize("net_name", ["915_64_32", "955_64_32"])
def test_p10_all_siting_pairs(ctx, net_name):
    """the nine pairs of input and output siting, both filters: chroma as restated from the
    sitings' box starts, Y as without a siting"""
    net, _ = make_net(ctx, net_name)
    h, w, H, W, n = size_for(net, "x3_n2")
    rng = np.random.default_rng(1101)
    frames = yuv10_frames(rng, n, h, w)
    src = with_junk(rng, frames)
    ny = W * H
    for filt in FILTERS:
        plain = net.upscale_yuv420p10_frames_host(src, w, h, W, H, filt)
        assert np.array_equal(plain, expected10(ctx, net, frames, w, h, W, H, filt,
                                                enlarged_for(("x3",), frames, w, h, W, H, filt)))
        for s_in in SITING_NAMES:
            for s_out in SITING_NAMES:
                got = net.upscale_yuv420p10_frames_host(src, w, h, W, H, filt, chroma_siting=s_in,
                                                        out_chroma_siting=s_out)
                assert np.array_equal(got[:, :ny], plain[:, :ny]), (filt, s_in, s_out)
                for i, f in enumerate(frames):
                    _, cb, cr = enlarge10(f, w, h, W, H, filt, s_in, s_out)
                    exp = np.concatenate([cb.ravel(), cr.ravel()])
                    assert np.array_equal(got[i, ny:], exp), (filt, s_in, s_out, i)


@pytest.mark.gpu
@pytest.mark.parametrize("net_name,case", [("915_64_32", "x3_n2"), ("955_64_32", "x3_n2"),
                                           ("915_128_64", "h3_256_n2"), ("915_64_32", "1080p_n10")])
def test_p10_device_matches_host_entry(ctx, net_name, case):
    """I010 and P010 in device memory, dense and pitched (2048-byte-aligned rows at 1080p, as
    decoders lay them out), random bits outside the input values and random input padding: the
    values are the host entry's, the bits outside them 0, the output padding untouched"""
    net, _ = make_net(ctx, net_name)
    h, w, H, W, n = size_for(net, case)
    rng = np.random.default_rng(1202)
    frames = yuv10_frames(rng, n, h, w)
    big = case.startswith("1080p")
    for filt in FILTERS:
        exp = net.upscale_yuv420p10_frames_host(with_junk(rng, frames), w, h, W, H, filt)
        for fmt in ("i420", "nv12"):
            got, _ = run_device10(ctx, net, frames, w, h, W, H, filt, fmt, rng)
            assert np.array_equal(got, exp), (fmt, filt, "dense")
            # rows 4-byte multiples for P010, 2 for I010; a gap between frames
            li = pitched10(fmt, w, h, 6 if fmt == "i420" else 8, 2 if fmt == "i420" else 4,
                           38 if fmt == "i420" else 44, 4096 if big else None)
            lo = pitched10(fmt, W, H, 14, 2 if fmt == "i420" else 12, 66 if fmt == "i420" else 68,
                           4096 if big else None)
            fill = np.full(needed_words(lo, W, H, n) + 256, 0xA7C3, np.uint16)
            got, buf = run_device10(ctx, net, frames, w, h, W, H, filt, fmt, rng, li, lo, fill)
            assert np.array_equal(got, exp), (fmt, filt, "pitched")
            keep = np.ones(buf.size, bool)
            keep[plane_index(in_words(lo), W, H, n).ravel()] = False
            assert keep.sum() > 256 and (buf[keep] == 0xA7C3).all(), (fmt, filt)


def pitched10(fmt, w, h, extra_y, extra_c, gap, pitch=None):
    """rows wider than their bytes, chroma after a 16-row-aligned Y plane, a gap between frames
    (as test_upscale_yuv420_device's pitched(), for 10-bit layouts)"""
    nv12 = fmt == "nv12"
    y_pitch = pitch or 2 * w + extra_y
    c_pitch = pitch or 2 * (w if nv12 else w // 2) + extra_c
    cb = -(-h // 16) * 16 * y_pitch
    dense = pkg.yuv420_layout(fmt, w, h, y_pitch, c_pitch, cb, bit_depth=10)
    return pkg.yuv420_layout(fmt, w, h, y_pitch, c_pitch, cb, dense.frame_stride + gap,
                             bit_depth=10)


@pytest.mark.gpu
def test_p10_device_composed_definition_and_sitings(ctx):
    """one small case of the device entry straight against the composed definition, with a
    siting conversion"""
    net, _ = make_net(ctx, "915_32_16")
    h, w, H, W, n = size_for(net, "40x40_n2")
    rng = np.random.default_rng(1303)
    frames = yuv10_frames(rng, n, h, w)
    for filt in FILTERS:
        enl = [enlarge10(f, w, h, W, H, filt, "left", "topleft") for f in frames]
        exp = expected10(ctx, net, frames, w, h, W, H, filt, enl)
        for fmt in ("i420", "nv12"):
            got, _ = run_device10(ctx, net, frames, w, h, W, H, filt, fmt, rng, s_in="left",
                                  s_out="topleft")
            assert np.array_equal(got, exp), (fmt, filt)


def check_launch_count10(net_name):
    """launches of a repeated 10-bit call == the 8-bit formulas, with the host entry's group of
    10-bit frames and the device entry's group of 8-bit ones"""
    from test_upscale_yuv420_device import default_group as device_group
    with pkg.Context(0) as c:
        net, _ = make_net(c, net_name)
        for (h, w, H, W, n) in ((20, 20, 40, 40, 3), (540, 960, 1080, 1920, 10)):
            frames = yuv10_frames(np.random.default_rng(n), n, h, w)
            F = forward_launches(c, net, W, H)
            fused = net.fused_supported()

            def launches(call):
                call()
                before = c.launch_count()
                call()
                c.block()
                return c.launch_count() - before

            got = launches(lambda: net.upscale_yuv420p10_frames_host(frames, w, h, W, H))
            expect = -(-n // default_group10(net, w, h, W, H, n)) * (5 + F) if fused else n * (4 + F + 1)
            assert got == expect, ("host", W, H, got, expect)
            for fmt in ("i420", "nv12"):
                li = pkg.yuv420_layout(fmt, w, h, bit_depth=10)
                lo = pkg.yuv420_layout(fmt, W, H, bit_depth=10)
                m_in = c.upload(np.zeros(needed_words(li, w, h, n), np.uint16), np.uint16)
                m_out = c.alloc(2 * needed_words(lo, W, H, n))
                nv12 = fmt == "nv12"
                got = launches(lambda: net.upscale_yuv420_frames(m_in, w, h, n, m_out, W, H, "lanczos",
                                                                 fmt, bit_depth=10))
                if fused:
                    expect = -(-n // device_group(net, W, H, n)) * (5 + nv12 + F)
                else:
                    expect = n * (4 + F + 1 + nv12)
                assert got == expect, (fmt, W, H, got, expect)
                c.release(m_in)
                c.release(m_out)


START_GROUP = os.environ.get("SRCNN_FRAMES_GROUP")


@pytest.mark.gpu
@pytest.mark.skipif(bool(SWITCHED), reason="launch counts assume the default kernel selection")
@pytest.mark.parametrize("net_name", ["915_64_32", "915_128_64", "955_64_32"])
def test_p10_launch_count(net_name):
    """in a process of its own, so that the group size the library reads once per process is the
    one the test computes"""
    env = {k: v for k, v in os.environ.items() if k != "SRCNN_FRAMES_GROUP"}
    if START_GROUP is not None:
        env["SRCNN_FRAMES_GROUP"] = START_GROUP
    tests = os.path.dirname(os.path.abspath(__file__))
    code = ("import sys; sys.path[:0] = [%r, %r]\nfrom test_upscale_yuv420p10 import "
            "check_launch_count10\ncheck_launch_count10(%r)\nprint('OK')" % (os.path.dirname(tests),
                                                                              tests, net_name))
    r = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("net_name", ["915_64_32", "955_64_32"])
def test_p10_and_8bit_tables_apart(ctx, net_name):
    """on a fresh context, 8-bit calls of one shape right after 10-bit ones (and the other way
    round) give the bytes of a context that only ran the one bit depth: the resample table cache
    keeps the two apart"""
    from test_upscale_yuv420 import yuv_frames
    from test_upscale_yuv420_device import run_device
    net, params = make_net(ctx, net_name)
    h, w, H, W, n = size_for(net, "x3_n2")
    rng = np.random.default_rng(1404)
    f8, f10 = yuv_frames(rng, n, h, w), yuv10_frames(rng, n, h, w)
    exp8 = {f: net.upscale_yuv420_frames_host(f8, w, h, W, H, f) for f in FILTERS}
    exp8s = {f: net.upscale_yuv420_frames_host(f8, w, h, W, H, f, chroma_siting="left") for f in FILTERS}
    exp10 = {f: net.upscale_yuv420p10_frames_host(f10, w, h, W, H, f) for f in FILTERS}
    for first in (10, 8):
        with pkg.Context(0) as c:
            net2 = pkg.Net(c, *NETS[net_name], params)
            for _ in range(2):
                for f in FILTERS:
                    if first == 10:
                        assert np.array_equal(net2.upscale_yuv420p10_frames_host(f10, w, h, W, H, f), exp10[f])
                    assert np.array_equal(net2.upscale_yuv420_frames_host(f8, w, h, W, H, f), exp8[f])
                    assert np.array_equal(net2.upscale_yuv420_frames_host(
                        f8, w, h, W, H, f, chroma_siting="left"), exp8s[f])
                    assert np.array_equal(run_device(c, net2, f8, w, h, W, H, f, "nv12")[0], exp8[f])
                    got, _ = run_device10(c, net2, f10, w, h, W, H, f, "nv12", rng)
                    assert np.array_equal(got, exp10[f]), (first, f)
                    assert np.array_equal(net2.upscale_yuv420p10_frames_host(f10, w, h, W, H, f), exp10[f])


@pytest.mark.gpu
def test_p10_rejects_bad_arguments(ctx):
    """the host entry rejects what the 8-bit one does; the device entry each 10-bit layout rule:
    SRCNN_EINVAL before any launch, the output untouched"""
    net, _ = make_net(ctx, "915_64_32")
    L, pnet = ctx.L, pkg.C.byref(net.c)
    src = np.zeros((2, 10 * 10 * 3 // 2), np.uint16)
    out = np.full(2 * 20 * 20 * 3 // 2, 7, np.uint16)

    def host(W=20, H=20, f=1, n=2, w=10, hh=10, s_in=0, s_out=0, s=pkg._np_ptr(src),
             d=pkg._np_ptr(out), c=ctx.h, nt=pnet):
        return L.srcnn_upscale_yuv420p10_frames_host(c, nt, s, w, hh, n, W, H, f, s_in, s_out, d)

    bad = [host(W=9), host(H=21), host(W=8), host(f=5), host(w=9), host(n=0), host(s_in=3),
           host(s_out=-1), host(s=None), host(d=None), host(c=None), host(nt=None), host(W=12, H=12)]
    assert bad == [EINVAL] * len(bad), bad
    assert (out == 7).all()
    with pytest.raises(pkg.SrcnnError):
        net.upscale_yuv420p10_frames_host(src, 10, 10, 21, 20)

    w, h, W, H, n = 10, 10, 20, 20, 2
    for fmt in ("i420", "nv12"):
        nv12 = fmt == "nv12"

        def lay(w, h, **kw):
            """a 10-bit layout whose only fault is what kw asks for: its frame_stride a multiple
            of 4 unless given"""
            d = pkg.yuv420_layout(fmt, w, h, bit_depth=10, **kw)
            if "frame_stride" not in kw:
                d.frame_stride = -(-d.frame_stride // 4) * 4
            return d

        def mod(l, **kw):
            x = pkg.CYuv420Layout.from_buffer_copy(l)
            for k, v in kw.items():
                setattr(x, k, v)
            return x

        li, lo = lay(w, h), lay(W, H)
        m_in = ctx.upload(np.zeros(needed_words(li, w, h, n) + 256, np.uint16), np.uint16)
        out_words = needed_words(lo, W, H, n) + 256
        m_out = ctx.upload(np.full(out_words, 7, np.uint16), np.uint16)
        base_in, base_out = ctx.mem_ptr(m_in), ctx.mem_ptr(m_out)

        def dev(li=li, lo=lo, n=n, m_in=m_in, m_out=m_out):
            return L.srcnn_upscale_yuv420_frames(ctx.h, pnet, m_in, pkg.C.byref(li), w, h, n, m_out,
                                                 pkg.C.byref(lo), W, H, 1)

        c_row, c_row_out = (2 * w, 2 * W) if nv12 else (w, W)
        before = ctx.launch_count()
        cases = {
            "depth 9": dev(li=mod(li, bit_depth=9), lo=mod(lo, bit_depth=9)),
            "depth 16": dev(li=mod(li, bit_depth=16), lo=mod(lo, bit_depth=16)),
            "depth -1": dev(li=mod(li, bit_depth=-1)),
            "depths differ": dev(lo=mod(lo, bit_depth=8)),
            "depths differ 0": dev(li=mod(li, bit_depth=0)),
            "y pitch below 2w": dev(li=lay(w, h, y_pitch=2 * w - 2)),
            "c pitch below row": dev(lo=lay(W, H, c_pitch=c_row_out - 4)),
            "odd y pitch": dev(li=lay(w, h, y_pitch=2 * w + 1)),
            "odd c pitch": dev(lo=lay(W, H, c_pitch=c_row_out + 1)),
            "odd cb offset": dev(li=lay(w, h, cb_offset=2 * w * h + 1)),
            "odd stride": dev(lo=mod(lo, frame_stride=lo.frame_stride + 1)),
            "odd buffer": dev(m_in=ctx.wrap(base_in + 1, 2 * needed_words(li, w, h, n))),
            "odd out buffer": dev(m_out=ctx.wrap(base_out + 1, 2 * needed_words(lo, W, H, n))),
        }
        if nv12:
            cases.update({
                "p010 c pitch 4k+2": dev(lo=lay(W, H, c_pitch=c_row_out + 2)),
                "p010 plane off 4": dev(li=lay(w, h, cb_offset=2 * w * h + 2)),
                "p010 stride 4k+2": dev(lo=mod(lo, frame_stride=lo.frame_stride + 2)),
                "p010 buffer off 4": dev(m_in=ctx.wrap(base_in + 2, 2 * needed_words(li, w, h, n))),
            })
        else:
            cases["odd cr offset"] = dev(li=mod(li, cr_offset=li.cr_offset + 1,
                                                frame_stride=li.frame_stride + 64))
        assert cases == {k: EINVAL for k in cases}, (fmt, cases)
        assert ctx.launch_count() == before
        assert (ctx.read(m_out, (out_words,), np.uint16) == 7).all()
        # layouts that keep the rules are accepted: wider rows by 4 bytes, one frame without a
        # stride, and an I010 plane (or buffer) at 2 mod 4
        assert dev() == 0
        assert dev(li=lay(w, h, y_pitch=2 * w + 4, c_pitch=c_row + 4)) == 0
        assert dev(n=1, li=mod(li, frame_stride=0), lo=mod(lo, frame_stride=0)) == 0
        if not nv12:
            assert dev(li=lay(w, h, cb_offset=2 * w * h + 2)) == 0
            assert dev(m_in=ctx.wrap(base_in + 2, 2 * needed_words(li, w, h, n))) == 0
        ctx.block()
        ctx.release(m_in)
        ctx.release(m_out)


@pytest.mark.gpu
def test_p10_device_stream_order_and_graph_capture():
    """as for 8-bit frames: a context on a torch stream sees a torch fill right before the call and
    a torch read right after it in order; a captured call replays on new input contents"""
    import torch
    s = torch.cuda.Stream()
    with pkg.Context(0, stream=s.cuda_stream) as c:
        h, w, H, W, n = 270, 480, 540, 960, 5
        rng = np.random.default_rng(1505)
        for net_name in ("915_64_32", "955_64_32"):
            net, _ = make_net(c, net_name)
            for fmt in ("nv12", "i420"):
                shift = 6 if fmt == "nv12" else 0
                li = pitched10(fmt, w, h, 64, 32, 0, 1024 if fmt == "nv12" else None)
                lo = pkg.yuv420_layout(fmt, W, H, bit_depth=10)
                sets = [yuv10_frames(rng, n, h, w) for _ in range(3)]
                exps = [net.upscale_yuv420p10_frames_host(f, w, h, W, H) for f in sets]
                idx_in, idx_out = plane_index(in_words(li), w, h, n), plane_index(in_words(lo), W, H, n)
                srcs = []
                for f in sets:
                    buf = np.zeros(needed_words(li, w, h, n), np.uint16)
                    buf[idx_in] = with_junk(rng, f, shift)
                    srcs.append(torch.from_numpy(buf.view(np.int16)).cuda())
                t_in = torch.zeros(srcs[0].numel(), dtype=torch.int16, device="cuda")
                t_out = torch.zeros(needed_words(lo, W, H, n), dtype=torch.int16, device="cuda")
                torch.cuda.synchronize()
                m_in = c.wrap(t_in.data_ptr(), 2 * t_in.numel())
                m_out = c.wrap(t_out.data_ptr(), 2 * t_out.numel())

                def call():
                    net.upscale_yuv420_frames(m_in, w, h, n, m_out, W, H, "lanczos", fmt, li, lo)

                def result(t):
                    return t.cpu().numpy().view(np.uint16)[idx_out] >> shift

                with torch.cuda.stream(s):
                    t_in.copy_(srcs[0])
                    call()
                    res = t_out.clone()
                s.synchronize()
                assert np.array_equal(result(res), exps[0]), (net_name, fmt)
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
                        assert np.array_equal(result(res), exps[k]), (net_name, fmt, k)
                    del g
                c.release(m_in)
                c.release(m_out)


def read_y4m10(path):
    data = open(path, "rb").read()
    header, rest = data.split(b"\n", 1)
    tags = header.split(b" ")[1:]
    w = int([t for t in tags if t[:1] == b"W"][0][1:])
    h = int([t for t in tags if t[:1] == b"H"][0][1:])
    fb = w * h * 3
    frames = []
    while rest:
        assert rest[:6] == b"FRAME\n"
        frames.append(np.frombuffer(rest[6:6 + fb], "<u2"))
        rest = rest[6 + fb:]
    return header, np.stack(frames)


@pytest.mark.gpu
@pytest.mark.parametrize("net_name", ["915_64_32", "955_64_32"])
def test_cnn_cli_y4m_10bit(ctx, tmp_path, net_name):
    """`cnn -i IN.y4m -o OUT.y4m --scale 2 --bit-depth 10` on a 70-frame C420p10 file (more than
    one batch of 64): the header's W and H doubled and its other tags copied, every frame the
    entry's words, written little-endian"""
    from helpers import make_params
    from test_host_cpp import CNN, HOST, run, write_config, write_params
    pkg.build()
    subprocess.check_call(["make", "-C", HOST, "-s"])
    cfg = NETS[net_name]
    rng = np.random.default_rng(1606)
    params = make_params(rng, *cfg)
    pfile, cfile = str(tmp_path / "params.json"), str(tmp_path / "config.json")
    write_params(pfile, params)
    write_config(cfile, cfg, pfile)
    h, w = 22, 18
    frames = with_junk(rng, yuv10_frames(rng, 70, h, w))
    src, dst = tmp_path / "in.y4m", tmp_path / "out.y4m"
    write_y4m(src, b"YUV4MPEG2 W18 H22 F25:1 Ip A1:1 C420p10 XYSCSS=420P10",
              frames.astype("<u2").view(np.uint8), marker=b"FRAME Ixyz\n")
    for opts in ([], ["--chroma-siting", "keep"]):
        r = run([CNN, "-c", cfile, "-i", str(src), "-o", str(dst), "--scale", "2", "--resample",
                 "bicubic", "--bit-depth", "10"] + opts)
        assert r.returncode == 0, r.stdout
        assert "Video: 18x22, 70 frames" in r.stdout, r.stdout
        header, got = read_y4m10(dst)
        assert header == b"YUV4MPEG2 W36 H44 F25:1 Ip A1:1 C420p10 XYSCSS=420P10", header
        net = pkg.Net(ctx, *cfg, params)
        exp = net.upscale_yuv420p10_frames_host(frames, w, h, 2 * w, 2 * h, "bicubic")
        assert got.shape == exp.shape and np.array_equal(got, exp)
        os.remove(dst)

"""4:2:0 chroma siting: srcnn_upscale_yuv420_frames_host_sited, the chroma_siting of
srcnn_yuv420_layout and `cnn --chroma-siting`.

The definition is Pillow's enlargement of a box with a fractional start (oracle/resample_sited.py;
tests/golden/pil_box_resample.npz holds Pillow's own output), with the start each siting pair
gives.  A frame's Y is that of the centre-sited entries; only its chroma changes.  Byte equality
with a restatement cannot catch a sign error in the siting itself, so a ramp sampled at the sited
positions checks the direction."""
import os
import subprocess

import numpy as np
import pytest

import _pkg
from conftest import load_npz
from oracle import resample as R
from oracle import resample_sited as S
from test_upscale import FILTERS, NETS, make_net
from test_upscale_yuv420 import (CASES, expected, planes, read_y4m, size_for, write_y4m,
                                 yuv_frames)
from test_upscale_yuv420_device import needed, outside, pitched, run_device

pkg = _pkg.load()

EINVAL = -1
SIT = pkg.CHROMA_SITINGS
# (input siting, output siting): kept at left and top-left, and converted both ways
PAIRS = [("left", "left"), ("topleft", "topleft"), ("left", "center"), ("center", "topleft")]


def sited_chroma(frame, w, h, W, H, filt, s_in, s_out):
    _, cb, cr = planes(frame, w, h)
    return (S.resize_sited(cb, W // 2, H // 2, filt, s_in, s_out),
            S.resize_sited(cr, W // 2, H // 2, filt, s_in, s_out))


def expected_sited(ctx, net, frames, w, h, W, H, filt, pairs):
    """the composed definition of every frame for each siting pair: {pair: [n][W*H*3//2]}.  Y
    does not depend on the siting, so the network runs once per frame."""
    enl = [(R.resize(planes(f, w, h)[0], W, H, filt),) + sited_chroma(f, w, h, W, H, filt, *pairs[0])
           for f in frames]
    first = expected(ctx, net, frames, w, h, W, H, filt, enl)
    out = {pairs[0]: first}
    ny = W * H
    for p in pairs[1:]:
        e = first.copy()
        for i, f in enumerate(frames):
            cb, cr = sited_chroma(f, w, h, W, H, filt, *p)
            e[i, ny:] = np.concatenate([cb.ravel(), cr.ravel()])
        out[p] = e
    return out


def host_sited(ctx, net, frames, w, h, W, H, filt, s_in, s_out):
    """the sited host entry called directly (the binding calls the plain one for centre/centre)"""
    out = np.empty((len(frames), W * H * 3 // 2), np.uint8)
    pkg._check(ctx.L.srcnn_upscale_yuv420_frames_host_sited(
        ctx.h, pkg.C.byref(net.c), pkg._np_ptr(frames), w, h, len(frames), W, H,
        pkg.RESAMPLE_FILTERS[filt], SIT[s_in], SIT[s_out], pkg._np_ptr(out)))
    return out


@pytest.fixture(scope="module")
def ctx():
    with pkg.Context(0) as c:
        yield c


# ----------------------------------------------------------------------------- CPU

def box_cases():
    g = load_npz("pil_box_resample.npz")
    for k in sorted(g):
        if k.endswith("_in"):
            name = k[:-3]
            yield name, g[k], g[name + "_box"], g[name + "_size"], {f: g[name + "_" + f] for f in FILTERS}


def pillow_box(box, W, H):
    """(x0, y0, sx, sy) as Pillow computes them: the box and its extent in single precision, the
    scale in double"""
    x0, y0, x1, y1 = (np.float32(v) for v in box)
    return float(x0), float(y0), float(x1 - x0) / W, float(y1 - y0) / H


def test_box_restatement_matches_pillow_golden():
    n = 0
    for name, img, box, (W, H), exp in box_cases():
        for filt in FILTERS:
            got = S.resize_box(img, int(W), int(H), filt, *pillow_box(box, W, H))
            assert got.dtype == np.uint8 and np.array_equal(got, exp[filt]), (name, filt)
            n += 1
    assert n == 96


def test_box_restatement_matches_live_pillow():
    Image = pytest.importorskip("PIL.Image")
    rng = np.random.default_rng(777)
    for _ in range(24):
        h, w = (int(v) for v in rng.integers(4, 16, 2))
        W, H = w * int(rng.integers(1, 4)) + int(rng.integers(0, 3)), h * int(rng.integers(1, 4))
        x0, y0 = float(rng.uniform(0, 1)), float(rng.choice([0.0, rng.uniform(0, 1)]))
        box = (x0, y0, w - float(rng.uniform(0, 0.5)), float(h) if y0 == 0.0 else h - 0.25)
        img = rng.integers(0, 256, (h, w), dtype=np.uint8)
        for filt, f in (("bicubic", Image.BICUBIC), ("lanczos", Image.LANCZOS)):
            exp = np.asarray(Image.fromarray(img, "L").resize((W, H), f, box=box))
            got = S.resize_box(img, W, H, filt, *pillow_box(box, W, H))
            assert np.array_equal(got, exp), (h, w, H, W, box, filt)


def test_centre_and_equal_sitings_start_at_zero():
    """in0 is exactly 0.0 for equal sitings at ratio 1 and for centre to centre at every ratio, so
    resize_sited(center, center) is Pillow's plain enlargement bit for bit"""
    for s in (0.25, 0.5):
        for n in (1, 7, 12, 540):
            assert S.chroma_in0(n, n, s, s) == 0.0
    for n in range(1, 40):
        for N in range(n, 4 * n + 3):
            assert S.chroma_in0(n, N, 0.5, 0.5) == 0.0
    rng = np.random.default_rng(31)
    for h, w, H, W in ((7, 9, 14, 27), (10, 10, 40, 30), (6, 5, 6, 13), (8, 8, 8, 8)):
        img = rng.integers(0, 256, (h, w), dtype=np.uint8)
        for filt in FILTERS:
            assert np.array_equal(S.resize_sited(img, W, H, filt, "center", "center"),
                                  R.resize(img, W, H, filt)), (h, w, H, W, filt)


def ramp_error(s, filt, s_in, s_out, axis, sited):
    """a chroma ramp of 8 levels per input chroma sample along `axis` (0: horizontal), sampled at
    s_in's positions and enlarged s times: the interior's error against the ramp at s_out's
    positions, enlarged with the sitings or as if both were centred"""
    wc, Wc = 14, 14 * s
    a_in, a_out = S.SITINGS[s_in][axis], S.SITINGS[s_out][axis]
    vals = np.round(8 * (np.arange(wc) + a_in)).astype(np.uint8)
    plane = np.repeat(vals[None, :], wc, 0) if axis == 0 else np.repeat(vals[:, None], wc, 1)
    out = S.resize_sited(plane, Wc, Wc, filt, *((s_in, s_out) if sited else ("center", "center")))
    truth = 8 * (np.arange(Wc) + a_out) * (wc / Wc)
    prof = out[Wc // 2, :] if axis == 0 else out[:, Wc // 2]
    return (prof.astype(np.float64) - truth)[3 * s:-3 * s]


@pytest.mark.parametrize("s", [2, 3, 4])
@pytest.mark.parametrize("filt", FILTERS)
def test_siting_direction_on_a_ramp(s, filt):
    """with the siting, the interior is within rounding (0.5) of the ramp at the output's sited
    positions; treated as centre-sited, every interior sample is off by at least 1.0 (left to
    centre: 2.0 on average), one way"""
    for s_in, s_out, axes, shift in (("left", "left", (0,), 2 * (1 - 1 / s)),
                                     ("topleft", "topleft", (0, 1), 2 * (1 - 1 / s)),
                                     ("left", "center", (0,), 2.0)):
        for axis in axes:
            good = ramp_error(s, filt, s_in, s_out, axis, True)
            bad = ramp_error(s, filt, s_in, s_out, axis, False)
            assert np.abs(good).max() <= 0.5, (s_in, s_out, axis, good)
            assert np.abs(bad).min() >= 1.0 and (bad < 0).all(), (s_in, s_out, axis, bad)
            assert abs(bad.mean() + shift) < 0.2, (s_in, s_out, axis, bad.mean(), shift)


def test_cli_chroma_siting_rejections(tmp_path):
    """an unknown --chroma-siting value, or the option without a forward-mode .y4m input, stops
    with one line before any device work; with `keep`, a C420mpeg2 header passes the header check
    (and stops at the device on a machine without one); without the option it is still refused"""
    from helpers import make_params
    from test_host_cpp import CNN, HOST, run, write_config, write_params
    pkg.build()
    subprocess.check_call(["make", "-C", HOST, "-s"])
    # a network with its parameters, so that a machine with a device runs the video through
    pfile, cfg = str(tmp_path / "params.json"), str(tmp_path / "config.json")
    write_params(pfile, make_params(np.random.default_rng(1), *NETS["915_32_16"]))
    write_config(cfg, NETS["915_32_16"], pfile)
    src = str(tmp_path / "in.y4m")
    write_y4m(src, b"YUV4MPEG2 W4 H4 C420mpeg2", np.zeros((2, 24), np.uint8))
    for bad in ("left", "mpeg2", "", "KEEP"):
        r = run([CNN, "dry", "-c", cfg, "-i", src, "--chroma-siting", bad])
        assert r.returncode != 0 and "--chroma-siting must be keep, 420jpeg, 420mpeg2 or 420paldv" \
            in r.stdout, (bad, r.stdout)
    ppm = str(tmp_path / "in.ppm")
    with open(ppm, "wb") as f:
        f.write(b"P6 4 4 255\n" + bytes(48))
    for cmd in ([CNN, "dry", "-c", cfg, "-i", ppm, "--chroma-siting", "keep"],
                [CNN, "dry", "-c", cfg, "-i", str(tmp_path), "--chroma-siting", "420jpeg"]):
        r = run(cmd)
        assert r.returncode != 0 and "--chroma-siting applies to a .y4m input in the forward mode " \
            "only" in r.stdout, r.stdout
    r = run([CNN, "train", "-c", cfg, "-i", str(tmp_path), "-o", str(tmp_path / "p"),
             "--chroma-siting", "keep"])
    assert r.returncode != 0 and "--chroma-siting applies" in r.stdout, r.stdout
    for tag in (b"C420mpeg2", b"C420paldv"):
        write_y4m(src, b"YUV4MPEG2 W32 H32 " + tag, np.zeros((2, 32 * 32 * 3 // 2), np.uint8))
        r = run([CNN, "dry", "-c", cfg, "-i", src])
        assert r.returncode != 0 and ("chroma siting '%s' is left-sited" % tag.decode()) in r.stdout
        assert "--chroma-siting keep enlarges it at its own siting" in r.stdout, r.stdout
        for opt in ("keep", "420jpeg", "420paldv"):
            r = run([CNN, "dry", "-c", cfg, "-i", src, "--chroma-siting", opt])
            assert "Video: 32x32, 2 frames" in r.stdout and "left-sited" not in r.stdout, r.stdout
            if "no CUDA device" in r.stdout:
                assert r.returncode != 0
            else:
                assert r.returncode == 0, r.stdout


# ----------------------------------------------------------------------------- GPU

# the composed definitions of a case, shared by the networks with the same output size
_EXPECTED = {}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("net_name", list(NETS))
def test_host_sited_matches_composed_definition(ctx, net_name, case):
    """every siting pair, both filters: the fused ring route and the frame-by-frame route (9-5-5);
    same_size_n2 resamples the chroma of a siting conversion whose size does not change"""
    net, _ = make_net(ctx, net_name)
    h, w, H, W, n = size_for(net, case)
    frames = yuv_frames(np.random.default_rng(list(CASES).index(case) + 900), n, h, w)
    for filt in FILTERS:
        exp = expected_sited(ctx, net, frames, w, h, W, H, filt, PAIRS)
        for s_in, s_out in PAIRS:
            got = net.upscale_yuv420_frames_host(frames, w, h, W, H, filt, chroma_siting=s_in,
                                                 out_chroma_siting=s_out)
            for i in range(n):
                assert np.array_equal(got[i], exp[s_in, s_out][i]), (filt, s_in, s_out, i)
        if case == "same_size_n2":
            # equal sitings copy the chroma; a conversion changes it
            c0 = frames[:, W * H:]
            assert np.array_equal(exp["left", "left"][:, W * H:], c0)
            assert not np.array_equal(exp["left", "center"][:, W * H:], c0)


@pytest.mark.gpu
@pytest.mark.parametrize("net_name", ["915_64_32", "955_64_32"])
def test_host_sited_centre_is_the_plain_entry(ctx, net_name):
    """centre/centre through the sited entry: the plain entry's bytes and launches"""
    net, _ = make_net(ctx, net_name)
    h, w, H, W = 90, 70, 256 + net.padding, 140
    frames = yuv_frames(np.random.default_rng(41), 5, h, w)
    for filt in FILTERS:
        plain = net.upscale_yuv420_frames_host(frames, w, h, W, H, filt)
        b = ctx.launch_count()
        net.upscale_yuv420_frames_host(frames, w, h, W, H, filt)
        n_plain = ctx.launch_count() - b
        b = ctx.launch_count()
        sited = host_sited(ctx, net, frames, w, h, W, H, filt, "center", "center")
        assert ctx.launch_count() - b == n_plain
        assert np.array_equal(sited, plain), filt


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["i420", "nv12"])
@pytest.mark.parametrize("net_name,case", [("915_64_32", "x3_n2"), ("955_64_32", "x3_n2"),
                                           ("915_64_32", "1080p_n10")])
def test_device_sited_matches_host_sited(ctx, net_name, case, fmt):
    """left and top-left, dense and pitched (random input padding, a sentinel in the output's):
    the planes are the sited host entry's bytes (NV12: the same bytes, interleaved), every
    sentinel survives, and a left -> centre conversion goes through the two layouts"""
    net, _ = make_net(ctx, net_name)
    h, w, H, W, n = size_for(net, case)
    rng = np.random.default_rng(93)
    frames = yuv_frames(rng, n, h, w)
    odd = fmt == "i420"
    big = case.startswith("1080p")
    li = pitched(fmt, w, h, 3 if odd else 6, 5 if odd else 10, 37 if odd else 38, 1024 if big else None)
    lo = pitched(fmt, W, H, 7 if odd else 4, 1 if odd else 2, 53 if odd else 64, 2048 if big else None)
    in_fill = rng.integers(0, 256, needed(li, w, h, n), dtype=np.uint8)
    out_fill = np.full(needed(lo, W, H, n) + 512, 0xA7, np.uint8)
    for filt in FILTERS:
        for s_in, s_out in (("left", "left"), ("topleft", "topleft"), ("left", "center")):
            exp = net.upscale_yuv420_frames_host(frames, w, h, W, H, filt, chroma_siting=s_in,
                                                 out_chroma_siting=s_out)
            dli, dlo = pkg.yuv420_layout(fmt, w, h), pkg.yuv420_layout(fmt, W, H)
            dli.chroma_siting, dlo.chroma_siting = SIT[s_in], SIT[s_out]
            dense, _ = run_device(ctx, net, frames, w, h, W, H, filt, fmt, dli, dlo)
            assert np.array_equal(dense, exp), (filt, s_in, s_out)
            li.chroma_siting, lo.chroma_siting = SIT[s_in], SIT[s_out]
            got, buf = run_device(ctx, net, frames, w, h, W, H, filt, fmt, li, lo, in_fill,
                                  out_fill.copy())
            assert np.array_equal(got, exp), (filt, s_in, s_out)
            rest = outside(buf, lo, W, H, n)
            assert rest.size > 512 and (rest == 0xA7).all(), (filt, int((rest != 0xA7).sum()))


@pytest.mark.gpu
@pytest.mark.parametrize("net_name", ["915_64_32", "955_64_32"])
def test_table_cache_keys_the_siting(ctx, net_name):
    """calls of one shape with different sitings, interleaved with the RGBA frames and image
    entries on one context: each gives its own bytes, call after call"""
    from test_upscale_frames import frames_of, per_frame
    net, _ = make_net(ctx, net_name)
    rng = np.random.default_rng(29)
    h, w, H, W = 30, 42, 90, 126
    frames = yuv_frames(rng, 3, h, w)
    pairs = [("center", "center")] + PAIRS
    exp = {p: expected_sited(ctx, net, frames, w, h, W, H, "lanczos", [p])[p] for p in pairs}
    assert len({e.tobytes() for e in exp.values()}) == len(pairs)
    rgba = frames_of(rng, 2, h, w)
    rgba_exp = per_frame(net, rgba, W, H, "lanczos")
    for _ in range(2):
        for p in pairs:
            assert np.array_equal(net.upscale_yuv420_frames_host(
                frames, w, h, W, H, chroma_siting=p[0], out_chroma_siting=p[1]), exp[p]), p
            for fmt in ("nv12", "i420"):
                li, lo = (pkg.yuv420_layout(fmt, w, h, chroma_siting=p[0]),
                          pkg.yuv420_layout(fmt, W, H, chroma_siting=p[1]))
                assert np.array_equal(run_device(ctx, net, frames, w, h, W, H, "lanczos", fmt, li,
                                                 lo)[0], exp[p]), (p, fmt)
            assert np.array_equal(net.upscale_frames_host(rgba, W, H), rgba_exp)
            assert np.array_equal(net.upscale_image_host(rgba[1], W, H), rgba_exp[1])


@pytest.mark.gpu
def test_graph_capture_after_a_siting_call():
    """after one call with a siting pair, a torch.cuda.graph capture of that call replays to the
    same bytes on new input contents"""
    import torch
    s = torch.cuda.Stream()
    with pkg.Context(0, stream=s.cuda_stream) as c:
        h, w, H, W, n = 270, 480, 540, 960, 3
        rng = np.random.default_rng(7)
        net, _ = make_net(c, "915_64_32")
        for fmt, (s_in, s_out) in (("nv12", ("left", "left")), ("i420", ("topleft", "center"))):
            li = pkg.yuv420_layout(fmt, w, h, chroma_siting=s_in)
            lo = pkg.yuv420_layout(fmt, W, H, chroma_siting=s_out)
            sets = [yuv_frames(rng, n, h, w) for _ in range(3)]
            exps = [net.upscale_yuv420_frames_host(f, w, h, W, H, chroma_siting=s_in,
                                                   out_chroma_siting=s_out) for f in sets]
            from test_upscale_yuv420_device import pack, unpack
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
            assert np.array_equal(unpack(res.cpu().numpy(), lo, W, H, n), exps[0]), fmt
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s):
                call()
            for k in (1, 2):
                with torch.cuda.stream(s):
                    t_in.copy_(srcs[k])
                    g.replay()
                    res = t_out.clone()
                s.synchronize()
                assert np.array_equal(unpack(res.cpu().numpy(), lo, W, H, n), exps[k]), (fmt, k)
            del g
            c.release(m_in)
            c.release(m_out)


@pytest.mark.gpu
@pytest.mark.parametrize("net_name", ["915_64_32", "955_64_32"])
def test_launch_count_does_not_depend_on_the_siting(ctx, net_name):
    """a repeated call launches as many kernels at every siting pair as at centre/centre (whose
    count the header's formula gives), I420, NV12 and the host entry"""
    net, _ = make_net(ctx, net_name)
    h, w, H, W, n = 540, 960, 1080, 1920, 10
    if not net.fused_supported():
        h, w, H, W, n = 90, 70, 180, 140, 3
    frames = yuv_frames(np.random.default_rng(3), n, h, w)

    def launches(f):
        f()
        b = ctx.launch_count()
        f()
        return ctx.launch_count() - b

    for fmt in ("i420", "nv12"):
        counts = {}
        for p in [("center", "center")] + PAIRS:
            li = pkg.yuv420_layout(fmt, w, h, chroma_siting=p[0])
            lo = pkg.yuv420_layout(fmt, W, H, chroma_siting=p[1])
            m_in, m_out = ctx.alloc(needed(li, w, h, n)), ctx.alloc(needed(lo, W, H, n))
            counts[p] = launches(lambda: net.upscale_yuv420_frames(m_in, w, h, n, m_out, W, H,
                                                                   "lanczos", fmt, li, lo))
            ctx.block()
            ctx.release(m_in)
            ctx.release(m_out)
        assert len(set(counts.values())) == 1, (fmt, counts)
    counts = {p: launches(lambda: host_sited(ctx, net, frames, w, h, W, H, "lanczos", *p))
              for p in [("center", "center")] + PAIRS}
    assert len(set(counts.values())) == 1, counts


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["i420", "nv12"])
def test_sitings_outside_the_enum_are_rejected(ctx, fmt):
    """-1 and 3 in either layout or either host argument: SRCNN_EINVAL, before any launch, the
    output untouched"""
    net, _ = make_net(ctx, "915_64_32")
    L, pnet = ctx.L, pkg.C.byref(net.c)
    w, h, W, H, n = 10, 10, 20, 20, 2
    li, lo = pkg.yuv420_layout(fmt, w, h), pkg.yuv420_layout(fmt, W, H)
    m_in = ctx.upload(np.zeros(needed(li, w, h, n), np.uint8), np.uint8)
    out_bytes = needed(lo, W, H, n)
    m_out = ctx.upload(np.full(out_bytes, 7, np.uint8), np.uint8)
    src = np.zeros((n, w * h * 3 // 2), np.uint8)
    dst = np.full((n, W * H * 3 // 2), 7, np.uint8)

    def dev(si, so):
        a, b = pkg.CYuv420Layout.from_buffer_copy(li), pkg.CYuv420Layout.from_buffer_copy(lo)
        a.chroma_siting, b.chroma_siting = si, so
        return L.srcnn_upscale_yuv420_frames(ctx.h, pnet, m_in, pkg.C.byref(a), w, h, n, m_out,
                                             pkg.C.byref(b), W, H, 1)

    def host(si, so):
        return L.srcnn_upscale_yuv420_frames_host_sited(ctx.h, pnet, pkg._np_ptr(src), w, h, n, W,
                                                        H, 1, si, so, pkg._np_ptr(dst))

    before = ctx.launch_count()
    got = [f(si, so) for f in (dev, host) for bad in (-1, 3) for si, so in ((bad, 0), (0, bad), (bad, bad))]
    assert got == [EINVAL] * len(got), got
    assert ctx.launch_count() == before
    assert (ctx.read(m_out, (out_bytes,), np.uint8) == 7).all() and (dst == 7).all()
    with pytest.raises(ValueError):
        pkg.yuv420_layout(fmt, w, h, chroma_siting="bottom")
    with pytest.raises(ValueError):
        net.upscale_yuv420_frames_host(src, w, h, W, H, chroma_siting="mpeg2")
    ctx.release(m_in)
    ctx.release(m_out)


@pytest.mark.gpu
@pytest.mark.parametrize("net_name", ["915_64_32", "955_64_32"])
def test_cnn_cli_y4m_chroma_siting(ctx, tmp_path, net_name):
    """a 70-frame left-sited video: `--chroma-siting keep` copies the header (W and H scaled) and
    gives the sited host entry's frames; `--chroma-siting 420jpeg` converts the chroma to centre
    and names it in the C and XYSCSS= tags"""
    from helpers import make_params
    from test_host_cpp import CNN, HOST, run, write_config, write_params
    pkg.build()
    subprocess.check_call(["make", "-C", HOST, "-s"])
    cfg = NETS[net_name]
    rng = np.random.default_rng(53)
    params = make_params(rng, *cfg)
    pfile, cfile = str(tmp_path / "params.json"), str(tmp_path / "config.json")
    write_params(pfile, params)
    write_config(cfile, cfg, pfile)
    h, w = 22, 18
    frames = yuv_frames(rng, 70, h, w)
    src, dst = tmp_path / "in.y4m", tmp_path / "out.y4m"
    write_y4m(src, b"YUV4MPEG2 W18 H22 F25:1 Ip A1:1 C420mpeg2 XYSCSS=420MPEG2", frames)
    net = pkg.Net(ctx, *cfg, params)
    for opt, header, out_siting in (
            ("keep", b"YUV4MPEG2 W36 H44 F25:1 Ip A1:1 C420mpeg2 XYSCSS=420MPEG2", "left"),
            ("420jpeg", b"YUV4MPEG2 W36 H44 F25:1 Ip A1:1 C420jpeg XYSCSS=420JPEG", "center")):
        r = run([CNN, "-c", cfile, "-i", str(src), "-o", str(dst), "--scale", "2",
                 "--chroma-siting", opt])
        assert r.returncode == 0, r.stdout
        got_header, got = read_y4m(dst)
        assert got_header == header, got_header
        exp = net.upscale_yuv420_frames_host(frames, w, h, 2 * w, 2 * h, "lanczos",
                                             chroma_siting="left", out_chroma_siting=out_siting)
        assert got.shape == exp.shape and np.array_equal(got, exp), opt
    # a header without a C tag gains one when the siting changes
    write_y4m(src, b"YUV4MPEG2 W18 H22 F25:1", frames[:3])
    r = run([CNN, "-c", cfile, "-i", str(src), "-o", str(dst), "--scale", "2", "--chroma-siting",
             "420paldv"])
    assert r.returncode == 0, r.stdout
    got_header, got = read_y4m(dst)
    assert got_header == b"YUV4MPEG2 W36 H44 F25:1 C420paldv", got_header
    exp = net.upscale_yuv420_frames_host(frames[:3], w, h, 2 * w, 2 * h, "lanczos",
                                         chroma_siting="center", out_chroma_siting="topleft")
    assert np.array_equal(got, exp)

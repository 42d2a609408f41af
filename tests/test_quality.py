"""Enlargement quality: srcnn_image_quality (Context.image_quality), srcnn_evaluate_frames_host
(Net.evaluate_frames_host) and `cnn eval`.

The definition is oracle/quality.py (float64, from the formulas).  The CPU tests check that
restatement on cases with known answers; the GPU tests check the kernel and the entries against
it, and that a frame's result is the same bits whatever shares its launch."""
import math
import os
import re
import subprocess
import sys

import numpy as np
import pytest
from scipy.signal import correlate2d

import _pkg
from oracle import quality as Q
from oracle import resample as R
from test_upscale import FILTERS, NETS, make_net, photo, rgba_of

pkg = _pkg.load()
TESTS = os.path.dirname(os.path.abspath(__file__))
SWITCHED = [k for k in ("SRCNN_FUSED_IMPL", "SRCNN_C5_IMPL", "SRCNN_B3_IMPL", "SRCNN_GW_IMPL",
                        "SRCNN_D1_IMPL") if os.environ.get(k)]


def direct_ssim(x, y):
    """SSIM of two float64 regions by an explicit loop over the window positions"""
    x, y = np.asarray(x, np.float64), np.asarray(y, np.float64)
    g = np.exp(-((np.arange(11) - 5.0) ** 2) / (2 * 1.5 ** 2))
    win = np.outer(g, g)
    win /= win.sum()
    vals = []
    for i in range(x.shape[0] - 10):
        for j in range(x.shape[1] - 10):
            a, b = x[i:i + 11, j:j + 11], y[i:i + 11, j:j + 11]
            ma, mb = (win * a).sum(), (win * b).sum()
            va = (win * a * a).sum() - ma * ma
            vb = (win * b * b).sum() - mb * mb
            cab = (win * a * b).sum() - ma * mb
            vals.append(((2 * ma * mb + Q.C1) * (2 * cab + Q.C2)) /
                        ((ma * ma + mb * mb + Q.C1) * (va + vb + Q.C2)))
    return float(np.mean(vals))


# ----------------------------------------------------------------------------- CPU: the oracle

def test_oracle_identical_images():
    rng = np.random.default_rng(1)
    img = rgba_of(photo(rng, 40, 33), rng)
    for border in (0, 3, 11):
        mse, ssim = Q.quality(img, img, border)
        assert mse == 0.0 and abs(ssim - 1.0) < 1e-15
        assert Q.psnr(mse) == math.inf


def test_oracle_constant_offset():
    """y = x + delta: mse = delta^2; with sigma_x = sigma_y = sigma_xy the SSIM of a window is
    (2 mx (mx + delta) + C1) / (mx^2 + (mx + delta)^2 + C1)"""
    rng = np.random.default_rng(2)
    delta = np.float32(1 / 64)
    # values on a 1/1024 grid: x + delta and x - y are exact in float32
    x = (rng.integers(0, 900, (30, 41)) / 1024).astype(np.float32)
    y = x + delta
    assert Q.mse_of(y, x) == float(delta) ** 2
    mx = correlate2d(x.astype(np.float64), Q.window(), mode="valid")
    d = float(delta)
    exp = np.mean((2 * mx * (mx + d) + Q.C1) / (mx * mx + (mx + d) ** 2 + Q.C1))
    assert abs(Q.ssim_map(x, y).mean() - exp) < 1e-12
    # a constant image: one closed form for every window
    c = np.full((20, 20), 0.25, np.float32)
    exp_c = (2 * 0.25 * (0.25 + d) + Q.C1) / (0.25 ** 2 + (0.25 + d) ** 2 + Q.C1)
    assert np.allclose(Q.ssim_map(c, c + delta), exp_c, rtol=0, atol=1e-13)


def test_oracle_minimum_region_has_one_window():
    rng = np.random.default_rng(3)
    a, b = rng.uniform(0, 1, (2, 11, 11))
    assert Q.ssim_map(a, b).shape == (1, 1)
    img = rng.integers(0, 256, (2, 23, 23, 4), dtype=np.uint8)
    x, y = Q.region(Q.luma(img[0]), 6), Q.region(Q.luma(img[1]), 6)
    assert x.shape == (11, 11) and Q.ssim_map(x, y).shape == (1, 1)


def test_oracle_matches_direct_window_loop():
    rng = np.random.default_rng(4)
    for h, w in ((11, 11), (17, 25), (30, 14)):
        a = Q.luma(rng.integers(0, 256, (h, w, 3), dtype=np.uint8))
        b = Q.luma(rgba_of(photo(rng, h, w)))
        assert abs(Q.ssim_map(a, b).mean() - direct_ssim(a, b)) < 1e-12


def test_oracle_luma_is_luma_of():
    """luma's float32 arithmetic against the same expression in float64 rounded step by step"""
    p = np.arange(256, dtype=np.uint8)
    img = np.stack([p, p[::-1], np.roll(p, 77)], -1)[None]
    r, g, b = (img[..., i].astype(np.float64) for i in range(3))
    f = np.float32
    exp = (((r * f(0.299)).astype(f) + (g * f(0.587)).astype(f)).astype(f) +
           (b * f(0.114)).astype(f)).astype(f)
    exp = (exp.astype(np.float64) / 255.0).astype(f)
    assert np.array_equal(Q.luma(img), exp)


# ----------------------------------------------------------------------------- CPU: CLI

def cli_built():
    from test_host_cpp import HOST
    pkg.build()
    subprocess.check_call(["make", "-C", HOST, "-s"])


def test_cli_eval_argument_errors(tmp_path):
    """`eval` with `train`, a bad --scale and a missing OUT_DIR fail before any device work"""
    from test_host_cpp import CNN, run
    cli_built()
    cfg = os.path.join(TESTS, "golden", "ref_config", "config.json")
    (tmp_path / "in").mkdir()
    (tmp_path / "file").write_text("x")
    base = [CNN, "eval", "-c", cfg, "-i", str(tmp_path / "in")]
    r = run([CNN, "train", "eval", "-c", cfg, "-i", str(tmp_path / "in"), "-o", str(tmp_path / "p.json")])
    assert r.returncode != 0 and "eval and train exclude each other" in r.stdout, r.stdout
    for bad in ("0", "1.5", "x"):
        r = run(base + ["-o", str(tmp_path), "--scale", bad])
        assert r.returncode != 0 and "--scale must be a whole number" in r.stdout, (bad, r.stdout)
    for out in (tmp_path / "missing", tmp_path / "file"):
        r = run(base + ["-o", str(out)])
        assert r.returncode != 0 and "does not exist or is not a directory" in r.stdout, r.stdout
        assert "Evaluation mode" not in r.stdout   # stopped before the mode started


# ----------------------------------------------------------------------------- GPU: kernel

@pytest.fixture(scope="module")
def ctx():
    with pkg.Context(0) as c:
        yield c


def content(rng, kind, S, h, w):
    """S RGBA8 (result, reference) frame pairs of one kind, every frame different"""
    if kind == "random":
        return (rng.integers(0, 256, (S, h, w, 4), dtype=np.uint8),
                rng.integers(0, 256, (S, h, w, 4), dtype=np.uint8))
    ref = np.stack([rgba_of(photo(rng, h, w), rng) for _ in range(S)])
    if kind == "identical":
        return ref.copy(), ref
    noise = rng.integers(-6, 7, ref.shape)
    return np.clip(ref.astype(int) + noise, 0, 255).astype(np.uint8), ref


def device_quality(ctx, res, ref, border, bpp):
    S, h, w, _ = ref.shape
    mr = ctx.upload(np.ascontiguousarray(res[..., :bpp]), np.uint8)
    mf = ctx.upload(ref, np.uint8)
    try:
        return ctx.image_quality(mr, mf, w, h, S, border, bpp)
    finally:
        ctx.release(mr)
        ctx.release(mf)


def check_against_oracle(got, res, ref, border):
    for s in range(ref.shape[0]):
        mse, ssim = Q.quality(res[s], ref[s], border)
        if mse == 0.0:
            assert got[s, 0] == 0.0
        else:
            assert abs(got[s, 0] - mse) <= 1e-9 * mse, (s, got[s, 0], mse)
        assert abs(got[s, 1] - ssim) <= 1e-6, (s, got[s, 1], ssim)


# (h, w, border): the 11x11 + 2b minimum, odd sizes, a region narrower than one tile, 1080p
QUALITY_CASES = {"min_b6": (23, 23, 6), "min_b0": (11, 11, 0), "odd_37x29_b3": (29, 37, 3),
                 "narrow_20x60_b2": (60, 20, 2), "odd_101x67_b8": (67, 101, 8),
                 "1080p_b6": (1080, 1920, 6)}


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["random", "smooth", "identical"])
@pytest.mark.parametrize("case", list(QUALITY_CASES))
def test_image_quality_matches_oracle(ctx, case, kind):
    h, w, border = QUALITY_CASES[case]
    rng = np.random.default_rng(list(QUALITY_CASES).index(case) * 3 + len(kind))
    S = 1 if case.startswith("1080p") else 7
    res, ref = content(rng, kind, S, h, w)
    for bpp in (3, 4):
        got = device_quality(ctx, res, ref, border, bpp)
        assert got.shape == (S, 2) and got.dtype == np.float64
        if kind == "identical":
            assert (got[:, 0] == 0.0).all() and np.abs(got[:, 1] - 1.0).max() <= 1e-6, got
        check_against_oracle(got, res, ref, border)
        # bit-identical on a second call, and each frame alone as inside the set
        assert np.array_equal(device_quality(ctx, res, ref, border, bpp), got)
        for s in (0, S - 1):
            assert np.array_equal(device_quality(ctx, res[s:s + 1], ref[s:s + 1], border, bpp),
                                  got[s:s + 1])


@pytest.mark.gpu
def test_image_quality_rejects_bad_arguments(ctx):
    res = ctx.alloc(2 * 30 * 30 * 4)
    ref = ctx.alloc(2 * 30 * 30 * 4)
    out = ctx.alloc(32)
    L, h = ctx.L, ctx.h
    bad = [L.srcnn_image_quality(h, res, bpp, ref, w, hh, S, b, out)
           for bpp, w, hh, S, b in ((2, 30, 30, 2, 0), (1, 30, 30, 2, 0), (3, 30, 30, 2, 10),
                                    (3, 30, 30, 2, -1), (3, 10, 30, 2, 0), (3, 30, 30, 0, 0),
                                    (4, 0, 30, 1, 0), (3, 30, 30, 70000, 0))]
    assert bad == [-1] * len(bad), bad
    # a 12x12 region is accepted; buffers too small are not
    assert L.srcnn_image_quality(h, res, 3, ref, 30, 30, 2, 9, out) == 0
    assert L.srcnn_image_quality(h, res, 4, ref, 30, 30, 3, 0, out) != 0
    for m in (res, ref, out):
        ctx.release(m)


# ----------------------------------------------------------------------------- GPU: evaluate

def eval_set(rng, n, h, w, W, H):
    """n small RGBA8 frames and their W x H RGBA8 references (the reference is a photo at the
    large size, the small frame a subsampled copy of it)"""
    refs = np.stack([rgba_of(photo(rng, H, W) // (1 + i % 3) + 5 * i, rng) for i in range(n)])
    ys, xs = (np.arange(h) * H) // h, (np.arange(w) * W) // w
    small = np.ascontiguousarray(refs[:, ys][:, :, xs])
    return small, refs


def resample_frames(ctx, small, W, H, filt):
    n, h, w, _ = small.shape
    mi, mo = ctx.alloc(h * w * 4), ctx.alloc(W * H * 4)
    out = []
    for f in small:
        ctx.write(mi, f)
        ctx.resample(mi, w, h, mo, W, H, filt)
        out.append(ctx.read(mo, (H, W, 4), np.uint8))
    ctx.release(mi)
    ctx.release(mo)
    return np.stack(out)


# (h, w, H, W, n)
EVAL_CASES = {"40x40_n3": (20, 20, 40, 40, 3), "odd_n5": (33, 27, 99, 54, 5)}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(EVAL_CASES))
@pytest.mark.parametrize("net_name", list(NETS))
def test_evaluate_frames(ctx, net_name, case):
    net, _ = make_net(ctx, net_name)
    h, w, H, W, n = EVAL_CASES[case]
    border = net.padding // 2
    rng = np.random.default_rng(list(EVAL_CASES).index(case) + 300)
    small, refs = eval_set(rng, n, h, w, W, H)
    for filt in FILTERS:
        rgb, met = net.evaluate_frames_host(small, refs, W, H, filt)
        assert rgb.shape == (n, H, W, 3) and met.shape == (n, 4)
        assert np.array_equal(rgb, net.upscale_frames_host(small, W, H, filt))
        # the network's metrics: the quality kernel on those bytes, and the oracle
        assert np.array_equal(met[:, :2], device_quality(ctx, rgb, refs, border, 3))
        check_against_oracle(met[:, :2], rgb, refs, border)
        # the baseline: the plain enlargement
        base = resample_frames(ctx, small, W, H, filt)
        assert np.array_equal(met[:, 2:], device_quality(ctx, base, refs, border, 4))
        check_against_oracle(met[:, 2:], base, refs, border)
        # an explicit border
        _, met2 = net.evaluate_frames_host(small, refs, W, H, filt, border=2)
        check_against_oracle(met2[:, :2], rgb, refs, 2)
        assert np.array_equal(net.evaluate_frames_host(small, refs, W, H, filt)[1], met)


@pytest.mark.gpu
def test_evaluate_frames_1080p(ctx):
    """several frame groups at the default group size, the last one partial"""
    net, _ = make_net(ctx, "915_64_32")
    rng = np.random.default_rng(77)
    small, refs = eval_set(rng, 7, 540, 960, 1920, 1080)
    rgb, met = net.evaluate_frames_host(small, refs, 1920, 1080)
    assert np.array_equal(rgb, net.upscale_frames_host(small, 1920, 1080))
    for i in (0, 6):
        check_against_oracle(met[i:i + 1, :2], rgb[i:i + 1], refs[i:i + 1], 6)
    assert np.array_equal(met[:, :2], device_quality(ctx, rgb, refs, 6, 3))


GROUP_CODE = r"""
import sys
import numpy as np
sys.path[:0] = [%r, %r]
import _pkg
from test_upscale import make_net
from test_quality import eval_set
pkg = _pkg.load()
out = []
with pkg.Context(0) as ctx:
    for name in ("915_64_32", "915_128_64"):
        net, _ = make_net(ctx, name)
        small, refs = eval_set(np.random.default_rng(5), 7, 45, 38, 114, 90)
        for filt in ("lanczos", "bicubic"):
            out.append(net.evaluate_frames_host(small, refs, 114, 90, filt)[1])
np.save(sys.argv[1], np.stack(out))
print("OK")
"""


@pytest.mark.gpu
def test_evaluate_groups_bit_identical(tmp_path):
    """groups of 1 and 2 (SRCNN_FRAMES_GROUP is read once per process) and the default group
    give the same metrics, bit for bit"""
    code = GROUP_CODE % (os.path.dirname(TESTS), TESTS)
    got = {}
    for group in ("1", "2", None):
        env = {k: v for k, v in os.environ.items() if k != "SRCNN_FRAMES_GROUP"}
        if group:
            env["SRCNN_FRAMES_GROUP"] = group
        path = str(tmp_path / ("m%s.npy" % group))
        r = subprocess.run([sys.executable, "-c", code, path], env=env, stdout=subprocess.PIPE,
                           stderr=subprocess.STDOUT, text=True)
        assert r.returncode == 0 and "OK" in r.stdout, r.stdout
        got[group] = np.load(path)
    assert np.array_equal(got["1"], got["2"]) and np.array_equal(got["1"], got[None])


def check_eval_launch_count(net_name):
    """launches of a repeated call == the header's formula"""
    from test_upscale_frames import forward_launches
    with pkg.Context(0) as c:
        net, _ = make_net(c, net_name)
        for (h, w, H, W, n) in ((20, 20, 40, 40, 3), (540, 960, 1080, 1920, 6)):
            small, refs = eval_set(np.random.default_rng(n), n, h, w, W, H)
            F = forward_launches(c, net, W, H)
            net.evaluate_frames_host(small, refs, W, H)
            before = c.launch_count()
            net.evaluate_frames_host(small, refs, W, H)
            launches = c.launch_count() - before
            if net.fused_supported():
                pad = net.padding
                frame = w * h * 4 + W * H * 11 + (W - pad) * (H - pad) * 4 + W * H * 4
                env = int(os.environ.get("SRCNN_FRAMES_GROUP", "0") or 0)
                group = min(env if env > 0 else max(1, (128 << 20) // frame), n, 65535)
                expect = -(-n // group) * (5 + F + 4)
            else:
                expect = n * (4 + F + 1 + 4)
            assert launches == expect, (W, H, launches, expect)


START_GROUP = os.environ.get("SRCNN_FRAMES_GROUP")


@pytest.mark.gpu
@pytest.mark.skipif(bool(SWITCHED), reason="launch counts assume the default kernel selection")
@pytest.mark.parametrize("net_name", ["915_64_32", "915_128_64", "955_64_32"])
def test_evaluate_launch_count(net_name):
    env = {k: v for k, v in os.environ.items() if k != "SRCNN_FRAMES_GROUP"}
    if START_GROUP is not None:
        env["SRCNN_FRAMES_GROUP"] = START_GROUP
    code = ("import sys; sys.path[:0] = [%r, %r]\nfrom test_quality import check_eval_launch_count\n"
            "check_eval_launch_count(%r)\nprint('OK')" % (os.path.dirname(TESTS), TESTS, net_name))
    r = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("net_name", ["915_64_32", "955_64_32"])
def test_evaluate_state_between_calls(ctx, net_name):
    """frames and evaluate calls interleaved on one context give their own results each time"""
    net, _ = make_net(ctx, net_name)
    rng = np.random.default_rng(9)
    small, refs = eval_set(rng, 4, 30, 25, 60, 50)
    first = net.evaluate_frames_host(small, refs, 60, 50)
    frames = net.upscale_frames_host(small, 60, 50)
    for _ in range(2):
        rgb, met = net.evaluate_frames_host(small, refs, 60, 50)
        assert np.array_equal(rgb, first[0]) and np.array_equal(met, first[1])
        assert np.array_equal(net.upscale_frames_host(small, 60, 50), frames)
        assert np.array_equal(net.evaluate_frames_host(small[1:3], refs[1:3], 60, 50)[1], met[1:3])


@pytest.mark.gpu
def test_evaluate_rejects_bad_arguments(ctx):
    """each bad argument fails with SRCNN_EINVAL, and the output buffers stay untouched"""
    net, _ = make_net(ctx, "915_64_32")
    img = np.zeros((2, 10, 10, 4), np.uint8)
    ref = np.zeros((2, 40, 40, 4), np.uint8)
    out = np.full(2 * 40 * 40 * 3, 7, np.uint8)
    met = np.full(8, 7.0)
    L, h, pnet = ctx.L, ctx.h, pkg.C.byref(net.c)
    P = pkg._np_ptr

    def call(W=40, H=40, f=1, n=2, src=P(img), r=P(ref), b=-1, dst=P(out), m=P(met), c=h, nt=pnet):
        return L.srcnn_evaluate_frames_host(c, nt, src, 10, 10, n, W, H, f, r, b, dst, m)

    bad = [call(W, H, f) for W, H, f in ((9, 20, 1), (20, 9, 1), (12, 12, 0), (0, 20, 1),
                                        (70000, 70000, 1), (20, 20, 5), (20, 20, -1))]
    bad += [call(n=0), call(n=-3), call(src=None), call(dst=None), call(c=None), call(nt=None),
            call(r=None), call(m=None), call(b=15), call(b=40), call(W=22, H=40)]
    assert bad == [-1] * len(bad), bad
    assert (out == 7).all() and (met == 7.0).all()
    # the smallest region accepted: 11x11 inside the default border of 6
    assert call(W=23, H=23) == 0
    with pytest.raises(pkg.SrcnnError):
        pkg._check(call(b=15))
    with pytest.raises(ValueError):
        net.evaluate_frames_host(img, ref, 40, 40, "nearest")


# ----------------------------------------------------------------------------- GPU: CLI

LINE = re.compile(r"^(\S+): network PSNR (\S+) dB SSIM (\S+) \| baseline PSNR (\S+) dB SSIM (\S+) "
                  r"\| gain (\S+) dB$", re.M)
MEAN = re.compile(r"^mean over (\d+) pairs: network PSNR (\S+) dB SSIM (\S+) \| baseline PSNR "
                  r"(\S+) dB SSIM (\S+) \| gain (\S+) dB$", re.M)


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [1, 2])
def test_cnn_cli_eval(tmp_path, scale):
    """`cnn eval -i SAMPLES [--scale N] -o OUT`: every printed value is the oracle's on the images
    `cnn -i DIR --scale N` writes, to the printed precision; the -o images are those images; a
    pair of the wrong size is reported and skipped"""
    from helpers import make_params
    from test_host_cpp import CNN, read_ppm, run, write_config, write_params, write_ppm
    cli_built()
    cfg = NETS["915_64_32"]
    rng = np.random.default_rng(51 + scale)
    pfile, cfile = str(tmp_path / "params.json"), str(tmp_path / "config.json")
    write_params(pfile, make_params(rng, *cfg))
    write_config(cfile, cfg, pfile)
    samples, smalls = tmp_path / "samples", tmp_path / "smalls"
    samples.mkdir()
    smalls.mkdir()
    # two sizes, names interleaved; "c_bad" has a reference of the wrong size
    sizes = {"a0": (30, 26), "a1": (25, 35), "a2": (30, 26), "a3": (30, 26), "c_bad": (24, 24)}
    refs = {}
    for name, (h, w) in sizes.items():
        H, W = h * scale, w * scale
        large = photo(rng, H + (3 if name == "c_bad" else 0), W)
        ys, xs = (np.arange(h) * H) // h, (np.arange(w) * W) // w
        small = np.clip(large[ys][:, xs].astype(int) + rng.integers(-4, 5, (h, w, 3)), 0, 255)
        write_ppm(samples / (name + "_large.ppm"), large)
        write_ppm(samples / (name + "_small.ppm"), small)
        write_ppm(smalls / (name + "_small.ppm"), small)
        refs[name] = rgba_of(large)
    flags = ["--scale", str(scale)] + (["--resample", "bicubic"] if scale == 2 else [])
    out = tmp_path / "out"
    out.mkdir()
    r = run([CNN, "eval", "-c", cfile, "-i", str(samples), "-o", str(out)] + flags)
    assert r.returncode == 0, r.stdout
    assert "'c_bad': reference is" in r.stdout and "Skipping sample" in r.stdout, r.stdout
    lines = {m.group(1): [float(v) for v in m.groups()[1:]] for m in LINE.finditer(r.stdout)}
    good = ["a0", "a1", "a2", "a3"]
    assert sorted(lines) == good, r.stdout
    # the directory mode's outputs of the small images
    dirout = tmp_path / "dirout"
    dirout.mkdir()
    rd = run([CNN, "-c", cfile, "-i", str(smalls), "-o", str(dirout)] + flags)
    assert rd.returncode == 0, rd.stdout
    assert sorted(os.listdir(out)) == [g + ".ppm" for g in good]
    border = (9 + 1 + 5 - 3) // 2
    filt = "bicubic" if scale == 2 else "lanczos"
    means = np.zeros(5)
    for name in good:
        got = read_ppm(out / (name + ".ppm"))
        exp = read_ppm(dirout / (name + "_small.ppm"))
        assert np.array_equal(got, exp), name
        small = read_ppm(samples / (name + "_small.ppm"))
        base = R.resize(small, got.shape[1], got.shape[0], filt)
        mse_n, ssim_n = Q.quality(got, refs[name], border)
        mse_b, ssim_b = Q.quality(base, refs[name], border)
        vals = [Q.psnr(mse_n), ssim_n, Q.psnr(mse_b), ssim_b, Q.psnr(mse_n) - Q.psnr(mse_b)]
        for v, printed, digits in zip(vals, lines[name], (4, 6, 4, 6, 4)):
            assert abs(v - printed) <= 0.51 * 10 ** -digits + 1e-9, (name, v, printed)
        means += vals
    m = MEAN.search(r.stdout)
    assert m and int(m.group(1)) == 4, r.stdout
    for v, printed, digits in zip(means / 4, [float(x) for x in m.groups()[1:]], (4, 6, 4, 6, 4)):
        assert abs(v - printed) <= 0.51 * 10 ** -digits + 1e-9, (v, printed)
    # dry: the same lines, nothing written
    dry = tmp_path / "dry"
    dry.mkdir()
    r2 = run([CNN, "eval", "dry", "-c", cfile, "-i", str(samples), "-o", str(dry)] + flags)
    assert r2.returncode == 0 and os.listdir(dry) == [], r2.stdout
    assert {m.group(1): [float(v) for v in m.groups()[1:]] for m in LINE.finditer(r2.stdout)} == lines

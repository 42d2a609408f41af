"""Image enlargement: the Pillow-exact resampling kernel (srcnn_resample), the pipelined image
entry (srcnn_upscale_image_host) and `cnn --scale`.

The definition is Pillow's Image.resize (oracle/resample.py restates it; tests/golden/
pil_resample.npz holds Pillow's own output).  The image entry must give, byte for byte, what the
existing device-layer calls give for the same work on the same context."""
import os

import numpy as np
import pytest

import _pkg
from conftest import load_npz
from oracle import resample as R

pkg = _pkg.load()

FILTERS = ("bicubic", "lanczos")


def golden_cases():
    g = load_npz("pil_resample.npz")
    for k in sorted(g):
        if k.endswith("_in"):
            continue
        name, filt = k.rsplit("_", 1)
        yield name, filt, g[name + "_in"], g[k]


def rgba_of(rgb, rng=None):
    """RGBA8 with an arbitrary alpha (the resampling ignores it) or 255"""
    h, w, _ = rgb.shape
    a = (rng.integers(0, 256, (h, w, 1), dtype=np.uint8) if rng is not None
         else np.full((h, w, 1), 255, np.uint8))
    return np.ascontiguousarray(np.concatenate([rgb, a], -1))


def photo(rng, h, w):
    """smooth colour gradients plus noise: a photo-like image whose luma varies"""
    yy, xx = np.mgrid[0:h, 0:w]
    rgb = np.stack([127 + 100 * np.sin(xx / 9.0), 127 + 100 * np.cos(yy / 7.0),
                    127 + 60 * np.sin((xx + yy) / 5.0)], -1) + rng.normal(0, 8, (h, w, 3))
    return np.clip(rgb, 0, 255).astype(np.uint8)


# ----------------------------------------------------------------------------- CPU

def test_restatement_matches_pillow_goldens():
    n = 0
    for name, filt, src, exp in golden_cases():
        got = R.resize(src, exp.shape[1], exp.shape[0], filt)
        assert got.dtype == np.uint8 and np.array_equal(got, exp), (name, filt)
        n += 1
    assert n == 20


def test_restatement_matches_live_pillow():
    Image = pytest.importorskip("PIL.Image")
    rng = np.random.default_rng(4242)
    for _ in range(24):
        h, w = (int(v) for v in rng.integers(1, 24, 2))
        H, W = h * int(rng.integers(1, 4)) + int(rng.integers(0, 5)), w + int(rng.integers(0, 40))
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        for filt, f in (("bicubic", Image.BICUBIC), ("lanczos", Image.LANCZOS)):
            exp = np.asarray(Image.fromarray(img, "RGB").resize((W, H), f))
            assert np.array_equal(R.resize(img, W, H, filt), exp), (h, w, H, W, filt)


def test_cli_scale_argument_errors(tmp_path):
    """bad --scale / --resample values and --scale with train stop before any device work"""
    import subprocess
    from test_host_cpp import CNN, HOST, run
    pkg.build()
    subprocess.check_call(["make", "-C", HOST, "-s"])
    cfg = os.path.join(os.path.dirname(__file__), "golden", "ref_config", "config.json")
    base = [CNN, "-c", cfg, "-i", "x.ppm", "-o", str(tmp_path / "o.ppm")]
    for bad in ("2.5", "0", "-2", "two", ""):
        r = run(base + ["--scale", bad])
        assert r.returncode != 0 and "--scale must be a whole number" in r.stdout, (bad, r.stdout)
    r = run(base + ["--scale", "2", "--resample", "nearest"])
    assert r.returncode != 0 and "--resample must be lanczos or bicubic" in r.stdout
    r = run([CNN, "train", "-c", cfg, "-i", str(tmp_path), "-o", str(tmp_path / "p.json"),
             "--scale", "2"])
    assert r.returncode != 0 and "--scale applies to the forward mode only" in r.stdout


# ----------------------------------------------------------------------------- GPU

@pytest.fixture(scope="module")
def ctx():
    with pkg.Context(0) as c:
        yield c


def resample_dev(ctx, rgba, W, H, filt, with_luma=True):
    h, w, _ = rgba.shape
    mi, mo = ctx.upload(rgba, np.uint8), ctx.alloc(W * H * 4)
    ml = ctx.alloc(4 * W * H) if with_luma else pkg.NULL_MEM
    ctx.resample(mi, w, h, mo, W, H, filt, ml)
    out = ctx.read(mo, (H, W, 4), np.uint8)
    luma = ctx.read(ml, (H, W)) if with_luma else None
    for m in (mi, mo) + ((ml,) if with_luma else ()):
        ctx.release(m)
    return out, luma


@pytest.mark.gpu
def test_resample_matches_pillow_goldens(ctx):
    rng = np.random.default_rng(1)
    for name, filt, src, exp in golden_cases():
        out, _ = resample_dev(ctx, rgba_of(src, rng), exp.shape[1], exp.shape[0], filt)
        assert np.array_equal(out[..., :3], exp), (name, filt)
        assert (out[..., 3] == 255).all()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2048, 2048, 4096, 4096), (1023, 1365, 3069, 4095),
                                   (7, 1, 21, 3), (4, 4, 16, 16)])
def test_resample_matches_restatement(ctx, shape):
    h, w, H, W = shape
    rng = np.random.default_rng(h * 7 + w)
    src = photo(rng, h, w)
    for filt in FILTERS:
        out, luma = resample_dev(ctx, rgba_of(src, rng), W, H, filt)
        assert np.array_equal(out[..., :3], R.resize(src, W, H, filt)), filt
        # the luma is extract_luma(normalize = 1) of the kernel's own output, bit for bit
        m, ml = ctx.upload(out, np.uint8), ctx.alloc(4 * W * H)
        ctx.extract_luma(m, ml, W, H, True)
        assert np.array_equal(luma.view(np.uint32), ctx.read(ml, (H, W)).view(np.uint32)), filt
        ctx.release(m)
        ctx.release(ml)


@pytest.mark.gpu
def test_resample_without_luma_writes_none(ctx):
    rng = np.random.default_rng(3)
    src = rgba_of(photo(rng, 30, 20))
    mi, mo, ml = ctx.upload(src, np.uint8), ctx.alloc(60 * 90 * 4), ctx.alloc(4 * 60 * 90)
    ctx.fill_float(ml, -7.0)
    ctx.resample(mi, 20, 30, mo, 60, 90, "lanczos")
    assert (ctx.read(ml, (90, 60)) == -7.0).all()
    assert np.array_equal(ctx.read(mo, (90, 60, 4), np.uint8)[..., :3],
                          R.resize(src[..., :3], 60, 90, "lanczos"))


@pytest.mark.gpu
def test_resample_rejects_bad_arguments(ctx):
    mi, mo = ctx.alloc(16 * 16 * 4), ctx.alloc(64 * 64 * 4)
    for w, h, W, H, f in ((8, 8, 4, 16, "lanczos"), (8, 8, 16, 4, "bicubic"), (0, 8, 16, 16, "lanczos"),
                          (8, 8, 16, -1, "lanczos")):
        with pytest.raises(pkg.SrcnnError):
            ctx.resample(mi, w, h, mo, W, H, f)
    with pytest.raises(pkg.SrcnnError):
        pkg._check(ctx.L.srcnn_resample(ctx.h, mi, 8, 8, mo, pkg.NULL_MEM, 16, 16, 7))
    with pytest.raises(pkg.SrcnnError):
        ctx.resample(mi, 16, 16, mo, 128, 128, "bicubic")   # output buffer too small


NETS = {"915_64_32": (64, 32, 9, 1, 5), "915_128_64": (128, 64, 9, 1, 5),
        "915_32_16": (32, 16, 9, 1, 5), "955_64_32": (64, 32, 9, 5, 5)}
# (h, w, H, W): one sub-band; network-output heights 255 / 256 (either side of the sub-band
# threshold; H = that + the network's padding); 2048^2 -> 4096^2; x3 to 3840x513
SIZES = {"40x40": (20, 20, 40, 40), "h3_255": (90, 70, 255, 140), "h3_256": (90, 70, 256, 140),
         "4096": (2048, 2048, 4096, 4096), "x3_3840x513": (171, 1280, 513, 3840)}


def size_for(net, size):
    h, w, H, W = SIZES[size]
    return h, w, H + (net.padding if size.startswith("h3_") else 0), W


def make_net(ctx, name, seed=5):
    from helpers import make_params
    cfg = NETS[name]
    params = make_params(np.random.default_rng(seed), *cfg)
    return pkg.Net(ctx, *cfg, params), params


def existing_calls(ctx, net, rgba, W, H, filt):
    """the same work through the existing device-layer calls: resample, extract_luma, sum of
    squares read to the host, sub_from_all(sum / n), forward, swap_luma, read.
    Returns (rgb, launches of the forward call)."""
    h, w, _ = rgba.shape
    (w1, h1), (w2, h2), (w3, h3) = net.out_dims(W, H)
    n = W * H
    mi, mb, ml, ms = ctx.upload(rgba, np.uint8), ctx.alloc(n * 4), ctx.alloc(4 * n), ctx.alloc(4)
    ctx.resample(mi, w, h, mb, W, H, filt)
    ctx.extract_luma(mb, ml, W, H, True)
    ctx.sum(ml, n, True, ms)
    s = ctx.read(ms, (1,))[0]
    ctx.sub_from_all(ml, np.float32(s) / np.float32(n), n)
    mo, mr = ctx.alloc(4 * w3 * h3), ctx.alloc(3 * n)
    scratch = [] if net.fused_supported() else [ctx.alloc(4 * w1 * h1 * net.n1),
                                                ctx.alloc(4 * w2 * h2 * net.n2)]
    before = ctx.launch_count()
    net.forward_fused(ml, mo, W, H, 1, *scratch)
    fwd_launches = ctx.launch_count() - before
    ctx.swap_luma(mb, mo, mr, W, H, w3, h3)
    rgb = ctx.read(mr, (H, W, 3), np.uint8)
    for m in [mi, mb, ml, ms, mo, mr] + scratch:
        ctx.release(m)
    return rgb, fwd_launches


def n_subbands(h3):
    s = int(os.environ.get("SRCNN_E2E_SUBBANDS", "16"))
    return 1 if h3 < 256 else min(max(s, 2), 32, max(2, h3 // 64))


@pytest.mark.gpu
@pytest.mark.parametrize("size", list(SIZES))
@pytest.mark.parametrize("net_name", list(NETS))
def test_upscale_matches_existing_calls(ctx, net_name, size):
    net, _ = make_net(ctx, net_name)
    h, w, H, W = size_for(net, size)
    rng = np.random.default_rng(list(SIZES).index(size))
    rgba = rgba_of(photo(rng, h, w), rng)
    for filt in FILTERS:
        got = net.upscale_image_host(rgba, W, H, filt)
        exp, fwd = existing_calls(ctx, net, rgba, W, H, filt)
        assert got.shape == (H, W, 3)
        assert np.array_equal(got, exp), (filt, int(np.abs(got.astype(int) - exp).max()))
        # launches per call follow the documented formula (a hidden fallback would show here)
        before = ctx.launch_count()
        again = net.upscale_image_host(rgba, W, H, filt)
        launches = ctx.launch_count() - before
        assert np.array_equal(again, exp), filt
        h3 = H - net.padding
        expect = 4 + n_subbands(h3) * (fwd + 1) if net.fused_supported() else 4 + fwd + 1
        assert launches == expect, (filt, launches, expect)


@pytest.mark.gpu
@pytest.mark.parametrize("size", ["40x40", "h3_256"])
@pytest.mark.parametrize("net_name", ["915_64_32", "955_64_32"])
def test_upscale_matches_oracle_chain(ctx, port, net_name, size):
    """restated resample -> extract_luma -> subtract_mean (Q1) -> 3 layers -> swap_luma of the
    plain-C oracle; the bound of test_cnn_cli_forward_image"""
    from oracle.loader import NetState
    net, params = make_net(ctx, net_name, seed=9)
    h, w, H, W = size_for(net, size)
    rng = np.random.default_rng(11)
    rgb = photo(rng, h, w)
    pad = net.padding
    for filt in FILTERS:
        got = net.upscale_image_host(rgba_of(rgb, rng), W, H, filt)
        big = rgba_of(R.resize(rgb, W, H, filt))
        luma = port.extract_luma(big, True)
        port.subtract_mean(luma.reshape(-1), with_event=True)
        _, _, o3 = port.net_forward(NetState(*NETS[net_name], params), luma, W, H, 1)
        exp = port.swap_luma(big, o3[0], W - pad, H - pad)
        diff = np.abs(got.astype(int) - exp.astype(int))
        assert diff.max() <= 1 and (diff > 0).mean() < 1e-3, (filt, diff.max(), (diff > 0).mean())


@pytest.mark.gpu
@pytest.mark.parametrize("net_name", ["915_64_32", "955_64_32"])
def test_upscale_state_between_calls(ctx, net_name):
    net, params = make_net(ctx, net_name)
    h, w, H, W = size_for(net, "h3_256")
    rng = np.random.default_rng(21)
    rgba = rgba_of(photo(rng, h, w))
    first = net.upscale_image_host(rgba, W, H)
    assert np.array_equal(net.upscale_image_host(rgba, W, H), first)     # replay
    # new weights through srcnn_write: the next call uses them
    new = {k: (v * np.float32(1.25)).astype(np.float32) for k, v in params.items()}
    for l in range(3):
        ctx.write(net.c.w[l], new["w%d" % (l + 1)])
        ctx.write(net.c.b[l], new["b%d" % (l + 1)])
    got = net.upscale_image_host(rgba, W, H)
    exp, _ = existing_calls(ctx, net, rgba, W, H, "lanczos")
    assert np.array_equal(got, exp) and not np.array_equal(got, first)
    # pinned and pageable host buffers give the same bytes
    pin_in, pin_out = pkg.PinnedBuffer(rgba.shape, np.uint8), pkg.PinnedBuffer((H, W, 3), np.uint8)
    try:
        pin_in.array[...] = rgba
        for _ in range(2):
            net.upscale_image_host(pin_in.array, W, H, out=pin_out.array)
            assert np.array_equal(pin_out.array, exp)
    finally:
        pin_in.free()
        pin_out.free()


@pytest.mark.gpu
def test_upscale_rejects_bad_sizes(ctx):
    """too small or too large outputs, downscaling and unknown filters fail with an error code
    before anything is read or written"""
    net, _ = make_net(ctx, "915_64_32")
    img, out = np.zeros((10, 10, 4), np.uint8), np.zeros(16, np.uint8)
    for W, H, f in ((9, 20, 1), (20, 9, 1), (12, 12, 0), (0, 20, 1), (70000, 70000, 1),
                    (20, 20, 5), (20, 20, -1)):
        with pytest.raises(pkg.SrcnnError):
            pkg._check(ctx.L.srcnn_upscale_image_host(ctx.h, pkg.C.byref(net.c), pkg._np_ptr(img),
                                                      10, 10, W, H, f, pkg._np_ptr(out)))
    with pytest.raises(ValueError):
        net.upscale_image_host(img, 20, 20, "nearest")


@pytest.mark.gpu
@pytest.mark.parametrize("filt", FILTERS)
@pytest.mark.parametrize("net_name", ["915_64_32", "955_64_32"])
def test_cnn_cli_scale(tmp_path, net_name, filt):
    """`cnn --scale N` == `cnn` on the restated N-times enlargement of the same image"""
    import subprocess
    from test_host_cpp import CNN, HOST, read_ppm, run, write_config, write_params, write_ppm
    from helpers import make_params
    pkg.build()
    subprocess.check_call(["make", "-C", HOST, "-s"])
    cfg = NETS[net_name]
    rng = np.random.default_rng(31)
    pfile, cfile = str(tmp_path / "params.json"), str(tmp_path / "config.json")
    write_params(pfile, make_params(rng, *cfg))
    write_config(cfile, cfg, pfile)
    for (h, w), s in (((48, 64), 2), ((37, 29), 3)):
        small = photo(rng, h, w)
        write_ppm(tmp_path / "small.ppm", small)
        write_ppm(tmp_path / "big.ppm", R.resize(small, s * w, s * h, filt))
        r = run([CNN, "-c", cfile, "-i", str(tmp_path / "small.ppm"), "-o",
                 str(tmp_path / "out.ppm"), "--scale", str(s), "--resample", filt])
        assert r.returncode == 0, r.stdout
        assert ("Scale: %dx, resample: %s" % (s, filt)) in r.stdout
        r = run([CNN, "-c", cfile, "-i", str(tmp_path / "big.ppm"), "-o", str(tmp_path / "ref.ppm")])
        assert r.returncode == 0, r.stdout
        got, ref = read_ppm(tmp_path / "out.ppm"), read_ppm(tmp_path / "ref.ppm")
        assert got.shape == (s * h, s * w, 3)
        assert np.array_equal(got, ref), (s, int(np.abs(got.astype(int) - ref).max()))

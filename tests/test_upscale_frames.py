"""Many frames per call: srcnn_upscale_frames_host (Net.upscale_frames_host) and `cnn -i DIR`.

Frame i of the frames entry must be, byte for byte, what srcnn_upscale_image_host returns for
frame i alone on the same context.  Every frame of a set has its own content (and so its own Q1
mean), so that a frame or ring-slot mix-up shows."""
import os
import subprocess
import sys

import numpy as np
import pytest

import _pkg
from test_upscale import FILTERS, NETS, make_net, photo, rgba_of

pkg = _pkg.load()

SWITCHED = [k for k in ("SRCNN_FUSED_IMPL", "SRCNN_C5_IMPL", "SRCNN_B3_IMPL", "SRCNN_GW_IMPL",
                        "SRCNN_D1_IMPL") if os.environ.get(k)]

# (h, w, H, W, n_frames); H of the h3_* cases is + the network's padding (either side of the
# image entry's sub-band threshold); "1080p" gives the default group size at least 3 groups and
# a partial last one (see default_group)
CASES = {"40x40_n1": (20, 20, 40, 40, 1), "40x40_n2": (20, 20, 40, 40, 2),
         "h3_255_n2": (90, 70, 255, 140, 2), "h3_256_n2": (90, 70, 256, 140, 2),
         "same_size_n2": (53, 61, 53, 61, 2), "1080p_n10": (540, 960, 1080, 1920, 10)}


def frames_of(rng, n, h, w):
    """n different photo-like RGBA8 frames (arbitrary alpha)"""
    return np.stack([rgba_of(photo(rng, h, w) // (1 + i % 3) + 7 * i, rng) for i in range(n)])


def default_group(net, w, h, W, H, n):
    """the group size the header documents: ~128 MB of device staging per group"""
    env = int(os.environ.get("SRCNN_FRAMES_GROUP", "0") or 0)
    if not net.fused_supported():
        return 1
    pad = net.padding
    frame = w * h * 4 + W * H * 11 + (W - pad) * (H - pad) * 4
    return min(env if env > 0 else max(1, (128 << 20) // frame), n, 65535)


def forward_launches(ctx, net, W, H):
    """launches of one srcnn_forward_fused call with the packed operand image cached"""
    (w1, h1), (w2, h2), (w3, h3) = net.out_dims(W, H)
    mi, mo = ctx.alloc(4 * W * H), ctx.alloc(4 * w3 * h3)
    scratch = [] if net.fused_supported() else [ctx.alloc(4 * w1 * h1 * net.n1),
                                                ctx.alloc(4 * w2 * h2 * net.n2)]
    net.forward_fused(mi, mo, W, H, 1, *scratch)
    before = ctx.launch_count()
    net.forward_fused(mi, mo, W, H, 1, *scratch)
    n = ctx.launch_count() - before
    for m in [mi, mo] + scratch:
        ctx.release(m)
    return n


def per_frame(net, frames, W, H, filt):
    return np.stack([net.upscale_image_host(f, W, H, filt) for f in frames])


def size_for(net, case):
    h, w, H, W, n = CASES[case]
    return h, w, H + (net.padding if case.startswith("h3_") else 0), W, n


@pytest.fixture(scope="module")
def ctx():
    with pkg.Context(0) as c:
        yield c


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("net_name", list(NETS))
def test_frames_match_image_entry(ctx, net_name, case):
    net, _ = make_net(ctx, net_name)
    h, w, H, W, n = size_for(net, case)
    rng = np.random.default_rng(list(CASES).index(case) + 100)
    frames = frames_of(rng, n, h, w)
    if case.startswith("1080p") and net.fused_supported():
        g = default_group(net, w, h, W, H, n)
        if not os.environ.get("SRCNN_FRAMES_GROUP"):
            assert -(-n // g) >= 3 and n % g != 0, g
    for filt in FILTERS:
        got = net.upscale_frames_host(frames, W, H, filt)
        exp = per_frame(net, frames, W, H, filt)
        assert got.shape == (n, H, W, 3)
        for i in range(n):
            assert np.array_equal(got[i], exp[i]), (filt, i, int(np.abs(got[i].astype(int) - exp[i]).max()))


@pytest.mark.gpu
@pytest.mark.parametrize("group", [1, 2])
def test_ring_wrap_around(group):
    """7 frames through groups of 1 and 2 (SRCNN_FRAMES_GROUP is read once per process): every
    ring slot is reused"""
    code = r"""
import sys
import numpy as np
sys.path.insert(0, %r)
sys.path.insert(0, %r)
import _pkg
from test_upscale import make_net
from test_upscale_frames import frames_of, per_frame
pkg = _pkg.load()
with pkg.Context(0) as ctx:
    for name in ("915_64_32", "915_128_64"):
        net, _ = make_net(ctx, name)
        frames = frames_of(np.random.default_rng(5), 7, 45, 38)
        for filt in ("lanczos", "bicubic"):
            got = net.upscale_frames_host(frames, 90, 114, filt)
            exp = per_frame(net, frames, 90, 114, filt)
            assert np.array_equal(got, exp), (name, filt)
print("OK")
""" % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, SRCNN_FRAMES_GROUP=str(group))
    r = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout


def check_launch_count(net_name):
    """launches of a repeated call == the documented formula"""
    with pkg.Context(0) as c:
        net, _ = make_net(c, net_name)
        for (h, w, H, W, n) in ((20, 20, 40, 40, 3), (540, 960, 1080, 1920, 6)):
            frames = frames_of(np.random.default_rng(n), n, h, w)
            F = forward_launches(c, net, W, H)
            net.upscale_frames_host(frames, W, H)
            before = c.launch_count()
            net.upscale_frames_host(frames, W, H)
            launches = c.launch_count() - before
            if net.fused_supported():
                n_groups = -(-n // default_group(net, w, h, W, H, n))
                expect = n_groups * (5 + F)
            else:
                expect = n * (4 + F + 1)
            assert launches == expect, (W, H, launches, expect)


# SRCNN_FRAMES_GROUP as the test process started (other tests set it in-process, after the
# library has read it once), for the subprocess below
START_GROUP = os.environ.get("SRCNN_FRAMES_GROUP")


@pytest.mark.gpu
@pytest.mark.skipif(bool(SWITCHED), reason="launch counts assume the default kernel selection")
@pytest.mark.parametrize("net_name", ["915_64_32", "915_128_64", "955_64_32"])
def test_launch_count(net_name):
    """in a process of its own, so that the group size the library reads once per process is the
    one default_group computes"""
    env = {k: v for k, v in os.environ.items() if k != "SRCNN_FRAMES_GROUP"}
    if START_GROUP is not None:
        env["SRCNN_FRAMES_GROUP"] = START_GROUP
    tests = os.path.dirname(os.path.abspath(__file__))
    code = ("import sys; sys.path[:0] = [%r, %r]\nfrom test_upscale_frames import check_launch_count\n"
            "check_launch_count(%r)\nprint('OK')" % (os.path.dirname(tests), tests, net_name))
    r = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("net_name", ["915_64_32", "955_64_32"])
def test_frames_state_between_calls(ctx, net_name):
    net, params = make_net(ctx, net_name)
    h, w, H, W = 90, 70, 256 + net.padding, 140
    rng = np.random.default_rng(21)
    frames = frames_of(rng, 5, h, w)
    first = net.upscale_frames_host(frames, W, H)
    assert np.array_equal(net.upscale_frames_host(frames, W, H), first)     # repeat
    # new weights through srcnn_write: the next call uses them
    new = {k: (v * np.float32(1.25)).astype(np.float32) for k, v in params.items()}
    for l in range(3):
        ctx.write(net.c.w[l], new["w%d" % (l + 1)])
        ctx.write(net.c.b[l], new["b%d" % (l + 1)])
    got = net.upscale_frames_host(frames, W, H)
    exp = per_frame(net, frames, W, H, "lanczos")
    assert np.array_equal(got, exp) and not np.array_equal(got, first)
    # pinned and pageable host buffers give the same bytes
    pin_in, pin_out = pkg.PinnedBuffer(frames.shape, np.uint8), pkg.PinnedBuffer((5, H, W, 3), np.uint8)
    try:
        pin_in.array[...] = frames
        for _ in range(2):
            net.upscale_frames_host(pin_in.array, W, H, out=pin_out.array)
            assert np.array_equal(pin_out.array, exp)
    finally:
        pin_in.free()
        pin_out.free()
    # image and frames calls interleaved on one context, other sizes too: each matches its own
    # reference
    small = frames_of(rng, 3, 20, 20)
    small_exp = per_frame(net, small, 40, 40, "bicubic")
    for _ in range(2):
        assert np.array_equal(net.upscale_image_host(frames[2], W, H), exp[2])
        assert np.array_equal(net.upscale_frames_host(small, 40, 40, "bicubic"), small_exp)
        assert np.array_equal(net.upscale_image_host(small[1], 40, 40, "bicubic"), small_exp[1])
        assert np.array_equal(net.upscale_frames_host(frames, W, H), exp)


@pytest.mark.gpu
def test_frames_rejects_bad_arguments(ctx):
    """each bad argument fails with SRCNN_EINVAL, and the output buffer stays untouched"""
    net, _ = make_net(ctx, "915_64_32")
    img = np.zeros((2, 10, 10, 4), np.uint8)
    out = np.full(2 * 40 * 40 * 3, 7, np.uint8)
    L, h, pnet = ctx.L, ctx.h, pkg.C.byref(net.c)

    def call(W, H, f, n=2, src=pkg._np_ptr(img), dst=pkg._np_ptr(out), c=h, nt=pnet):
        return L.srcnn_upscale_frames_host(c, nt, src, 10, 10, n, W, H, f, dst)

    bad = [call(W, H, f) for W, H, f in ((9, 20, 1), (20, 9, 1), (12, 12, 0), (0, 20, 1),
                                        (70000, 70000, 1), (20, 20, 5), (20, 20, -1))]
    bad += [call(20, 20, 1, n=0), call(20, 20, 1, n=-3), call(20, 20, 1, src=None),
            call(20, 20, 1, dst=None), call(20, 20, 1, c=None), call(20, 20, 1, nt=None)]
    assert bad == [-1] * len(bad), bad
    assert (out == 7).all()
    with pytest.raises(pkg.SrcnnError):
        pkg._check(call(20, 9, 1))
    with pytest.raises(ValueError):
        net.upscale_frames_host(img, 20, 20, "nearest")


# ----------------------------------------------------------------------------- CLI

def write_pgm(path, gray):
    h, w = gray.shape
    with open(path, "wb") as fh:
        fh.write(b"P5\n%d %d\n255\n" % (w, h))
        fh.write(np.ascontiguousarray(gray, np.uint8).tobytes())


def test_cli_directory_needs_output_directory(tmp_path):
    """-i DIR with an -o that is missing or a file fails before any device work"""
    from test_host_cpp import CNN, HOST, run
    pkg.build()
    subprocess.check_call(["make", "-C", HOST, "-s"])
    cfg = os.path.join(os.path.dirname(__file__), "golden", "ref_config", "config.json")
    (tmp_path / "in").mkdir()
    (tmp_path / "file").write_text("x")
    for out in (tmp_path / "missing", tmp_path / "file"):
        r = run([CNN, "-c", cfg, "-i", str(tmp_path / "in"), "-o", str(out)])
        assert r.returncode != 0 and "does not exist or is not a directory" in r.stdout, r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("net_name", ["915_64_32", "955_64_32"])
def test_cnn_cli_directory(tmp_path, net_name):
    """`cnn -i DIR -o OUT_DIR [--scale 2]`: every result is byte-equal to `cnn` on that file
    alone with the same flags; `dry` writes nothing; a non-image file is skipped"""
    from helpers import make_params
    from test_host_cpp import CNN, HOST, read_ppm, run, write_config, write_params, write_ppm
    pkg.build()
    subprocess.check_call(["make", "-C", HOST, "-s"])
    cfg = NETS[net_name]
    rng = np.random.default_rng(41)
    pfile, cfile = str(tmp_path / "params.json"), str(tmp_path / "config.json")
    write_params(pfile, make_params(rng, *cfg))
    write_config(cfile, cfg, pfile)
    src = tmp_path / "frames"
    src.mkdir()
    # two sizes, names interleaved (a batch ends at every size change), one grey image
    sizes = {"a0": (40, 52), "a1": (37, 29), "a2": (40, 52), "a3": (40, 52), "a4": (37, 29)}
    for stem, (h, w) in sizes.items():
        write_ppm(src / (stem + ".ppm"), photo(rng, h, w))
    write_pgm(src / "a5.pgm", photo(rng, 40, 52)[..., 1])
    (src / "notes.txt").write_text("not an image")
    stems = list(sizes) + ["a5"]
    for flags in (["--scale", "2", "--resample", "bicubic"], []):
        out = tmp_path / ("out%d" % len(flags))
        out.mkdir()
        r = run([CNN, "-c", cfile, "-i", str(src), "-o", str(out)] + flags)
        assert r.returncode == 0, r.stdout
        assert "Input directory: " in r.stdout and "'notes.txt' is not a .ppm/.pgm image" in r.stdout
        assert sorted(os.listdir(out)) == [s + ".ppm" for s in stems]
        for s in stems:
            f = src / (s + (".pgm" if s == "a5" else ".ppm"))
            r = run([CNN, "-c", cfile, "-i", str(f), "-o", str(tmp_path / "ref.ppm")] + flags)
            assert r.returncode == 0, r.stdout
            got, ref = read_ppm(out / (s + ".ppm")), read_ppm(tmp_path / "ref.ppm")
            assert got.shape == ref.shape and np.array_equal(got, ref), (flags, s)
        dry = tmp_path / "dry"
        dry.mkdir()
        r = run([CNN, "dry", "-c", cfile, "-i", str(src), "-o", str(dry)] + flags)
        assert r.returncode == 0, r.stdout
        assert os.listdir(dry) == [] and "Saving result image" not in r.stdout
        dry.rmdir()

"""Launches per call of the pipelined host-buffer inference entries: srcnn_infer_rows_host (its
sub-band pipeline, captured and replayed as a CUDA graph), srcnn_infer_rows_host_async and
srcnn_infer_frames_host (its ring of frame groups).

Each sub-band or frame group is one fused forward, so a call launches what that many
srcnn_forward_fused calls launch.  The launches of one forward are measured, not assumed, so the
counts hold under every kernel switch."""
import os
import subprocess
import sys

import numpy as np
import pytest

import _pkg
from helpers import luma_image, make_params
from test_upscale import n_subbands
from test_upscale_frames import forward_launches

pkg = _pkg.load()

NETS = {"915_64_32": (64, 32), "915_128_64": (128, 64)}
# (w, h): 188 output rows (one sub-band) and 688 output rows (the multi-stream pipeline)
ROWS_SIZES = {"h3_188": (120, 200), "h3_688": (150, 700)}


@pytest.fixture(scope="module")
def ctx():
    with pkg.Context(0) as c:
        yield c


def make_net(ctx, name, seed=7):
    n1, n2 = NETS[name]
    return pkg.Net(ctx, n1, n2, 9, 1, 5, make_params(np.random.default_rng(seed), n1, n2, 9, 1, 5))


def launches(ctx, fn):
    before = ctx.launch_count()
    fn()
    return ctx.launch_count() - before


@pytest.mark.gpu
@pytest.mark.parametrize("size", list(ROWS_SIZES))
@pytest.mark.parametrize("net_name", list(NETS))
def test_rows_host_launches(ctx, net_name, size):
    """one fused forward per sub-band, on the capturing call and on a replay"""
    net = make_net(ctx, net_name)
    w, h = ROWS_SIZES[size]
    (_, _), (_, _), (w3, h3) = net.out_dims(w, h)
    F = forward_launches(ctx, net, w, h)
    hin, hout = pkg.PinnedBuffer((h, w)), pkg.PinnedBuffer((h3, w3))
    hin.array[:] = luma_image(np.random.default_rng(h), h, w)
    expect = n_subbands(h3) * F
    for call in ("capture", "replay"):
        n = launches(ctx, lambda: net.infer_rows_host(hin.array, w, h, 0, h3, hout.array))
        assert n == expect, (call, n, expect)


@pytest.mark.gpu
@pytest.mark.parametrize("size", list(ROWS_SIZES))
@pytest.mark.parametrize("net_name", list(NETS))
def test_rows_host_async_launches(ctx, net_name, size):
    """two asynchronous calls (one per lane) launch what two blocking calls launch and give the
    blocking call's bytes"""
    net = make_net(ctx, net_name)
    w, h = ROWS_SIZES[size]
    (_, _), (_, _), (w3, h3) = net.out_dims(w, h)
    F = forward_launches(ctx, net, w, h)
    hin = pkg.PinnedBuffer((h, w))
    hin.array[:] = luma_image(np.random.default_rng(h + 1), h, w)
    ref = pkg.PinnedBuffer((h3, w3))
    net.infer_rows_host(hin.array, w, h, 0, h3, ref.array)
    outs = [pkg.PinnedBuffer((h3, w3)) for _ in range(2)]
    for call in ("capture", "replay"):
        for o in outs:
            o.array[:] = -1.0

        def two_async():
            for o in outs:
                net.infer_rows_host(hin.array, w, h, 0, h3, o.array, block=False)
            ctx.block()

        n = launches(ctx, two_async)
        assert n == 2 * n_subbands(h3) * F, (call, n, n_subbands(h3), F)
        for o in outs:
            assert np.array_equal(o.array, ref.array), call


def check_frames_launches(net_name, group):
    """launches of srcnn_infer_frames_host with SRCNN_FRAMES_GROUP=group: one fused forward per
    frame group, the last one partial"""
    n_frames, w, h = 2 * group + 1, 64, 48
    with pkg.Context(0) as c:
        net = make_net(c, net_name)
        (_, _), (_, _), (w3, h3) = net.out_dims(w, h)
        F = forward_launches(c, net, w, h)
        hin, hout = pkg.PinnedBuffer((n_frames, h, w)), pkg.PinnedBuffer((n_frames, h3, w3))
        hin.array[:] = np.stack([luma_image(np.random.default_rng(i), h, w) for i in range(n_frames)])
        for call in range(2):
            n = launches(c, lambda: net.infer_frames_host(hin.array, w, h, hout.array))
            assert n == -(-n_frames // group) * F, (call, n, F)


@pytest.mark.gpu
@pytest.mark.parametrize("net_name", list(NETS))
def test_frames_host_launches(net_name):
    """in a process of its own: the library reads SRCNN_FRAMES_GROUP once per process"""
    group = 3
    tests = os.path.dirname(os.path.abspath(__file__))
    code = ("import sys; sys.path[:0] = [%r, %r]\nfrom test_host_pipelines import check_frames_launches\n"
            "check_frames_launches(%r, %d)\nprint('OK')" % (os.path.dirname(tests), tests, net_name, group))
    env = dict(os.environ, SRCNN_FRAMES_GROUP=str(group))
    r = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout

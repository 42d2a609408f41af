"""The tensor-core kernels of a training chunk (the fused 9-1-5 training forward, the 9-5-5
layer-1-only forward, conv5_tc forward / deltas, bwd3_tc, wgrad1_fused_tc, wgrad2_tc,
wgrad5_tc) outside the regime of test_gpu_parity.py: parameters and inputs over many orders of
magnitude, the edges of their FP16-split operand domains, sample geometries that straddle the
128-column strips, wrap the accumulator rings and sit on either side of every width and
sample-count limit, and state that a chunk leaves behind in the context.

Every comparison is relative to the compared tensor's own scale, so that it means the same at
1e-6 as at 1e3:
    activations, deltas: |got - exp| <= 1e-4 |exp| + 1e-5 max|exp|
    gradients:           |got - exp| <= 1e-4 |exp| + 2e-6 max|exp|
and a tensor of zeros must violate it (unless the case requires the tensor to be exactly zero).
The launch count of each chunk is part of the case: a kernel that silently stops taking its
shape turns the case into a test of the FP32 kernels, and changes the count.
    python -m pytest tests/test_train_tc_edges.py -m gpu
"""
import os
import zlib

import numpy as np
import pytest

import _pkg
from helpers import make_params, patches
from oracle.loader import NetState

pytestmark = pytest.mark.gpu
pkg = _pkg.load()

# Under an A/B switch of the library (README "Environment switches") the same numeric cases run
# on the fallback kernels; only the launch-count assertions are skipped then.
SWITCHED = [k for k in ("SRCNN_FUSED_IMPL", "SRCNN_C5_IMPL", "SRCNN_B3_IMPL", "SRCNN_GW_IMPL",
                        "SRCNN_D1_IMPL") if os.environ.get(k)]

N915 = (64, 32, 9, 1, 5)
N955 = (64, 32, 9, 5, 5)
ACT = (1e-4, 1e-5)    # activations and deltas: (relative, floor relative to max|exp|)
GRAD = (1e-4, 2e-6)   # gradients
GRAD_KEYS = ("w1", "b1", "w2", "b2", "w3", "b3")


@pytest.fixture(scope="module")
def ctx():
    c = pkg.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module", autouse=True)
def _threads(port):
    port.set_num_threads(len(os.sched_getaffinity(0)))


def _rng(*key):
    return np.random.default_rng(zlib.crc32(repr(key).encode()))


def assert_close(name, got, exp, tol, exact_zero=False, mask=None):
    """|got - exp| <= rel |exp| + floor max|exp| over `mask` (all entries by default); the
    bound must not hold for zeros in place of `got` unless the case requires exp == 0."""
    got = np.asarray(got, np.float64).reshape(-1)
    exp = np.asarray(exp, np.float64).reshape(-1)
    assert np.isfinite(got).all(), "%s: %d non-finite entries" % (name, (~np.isfinite(got)).sum())
    if mask is not None:
        got, exp = got[mask.reshape(-1)], exp[mask.reshape(-1)]
    if exact_zero:
        assert not exp.any(), "%s: the oracle's tensor is not zero (case set-up)" % name
        assert not got.any(), "%s: %d non-zero entries, max |x| %.3g" % (
            name, np.count_nonzero(got), np.abs(got).max())
        return
    rel, floor = tol
    scale = float(np.abs(exp).max())
    bound = rel * np.abs(exp) + floor * scale
    err = np.abs(got - exp)
    bad = err > bound
    if bad.any():
        i = int(np.argmax(err - bound))
        raise AssertionError("%s: %d of %d entries out of bound; worst [%d] got %.9g exp %.9g "
                             "(|err| %.3g, bound %.3g, max|exp| %.3g)"
                             % (name, bad.sum(), bad.size, i, got[i], exp[i], err[i], bound[i], scale))
    assert (np.abs(exp) > bound).any(), "%s: zeros would pass (max|exp| %.3g)" % (name, scale)


class Chunk:
    """One srcnn_train_chunk on fresh parameters and what the oracle says about it."""

    def __init__(self, ctx, port, cfg, params, x, gt, w, h, S, oracle=True):
        self.cfg, self.params, self.w, self.h, self.S = cfg, params, w, h, S
        self.net = net = pkg.Net(ctx, *cfg, params)
        on = NetState(*cfg, params)
        (w1, h1), (w2, h2), (w3, h3) = net.out_dims(w, h)
        shapes = {"out1": (S, h1, w1, cfg[0]), "out2": (S, h2, w2, cfg[1]), "out3": (S, h3, w3)}
        mi, mg = ctx.upload(x), ctx.upload(gt)
        self.work = ctx.alloc(net.train_workspace_bytes(w, h, S))
        n0 = ctx.launch_count()
        net.train_chunk(mi, mg, w, h, S, self.work)
        self.launches = ctx.launch_count() - n0
        # sub-buffers out1, out2, out3, d1, d2, d3, each 256-byte aligned (srcnn_train_chunk)
        self.offset, self.got, off = {}, {}, 0
        for name in ("out1", "out2", "out3", "d1", "d2", "d3"):
            shape = shapes["out" + name[-1]]
            self.offset[name] = off
            self.got[name] = ctx.read(self.work, shape, offset=off)
            off += (int(np.prod(shape)) * 4 + 255) // 256 * 256
        self.grads = net.grads()
        ctx.release(mi)
        ctx.release(mg)
        if not oracle:
            return
        self.exp = dict(zip(("out1", "out2", "out3"), port.net_forward(on, x, w, h, S)))
        # The backward pass switches on [activation > 0] (ReLU derivative, and quirk Q2 on the
        # linear output): the oracle's backward runs on the activations the GPU produced.
        d = port.net_backward(on, x, gt, w, h, S, self.got["out1"], self.got["out2"], self.got["out3"])
        self.exp.update(zip(("d1", "d2", "d3"), d))
        self.egrads = {}
        for l in range(3):
            self.egrads["w%d" % (l + 1)], self.egrads["b%d" % (l + 1)] = on.gw[l], on.gb[l]
        self.d1_written = net.train_materializes_d1()

    def check(self, zero=(), masks=None, grad_tol=GRAD):
        """Everything against the oracle; `zero`: tensors / gradients ("gw1", "gb2", ...) the
        case requires to be exactly zero; `masks`: entries a tensor is checked on."""
        masks = masks or {}
        for name in ("out1", "out2", "out3", "d1", "d2", "d3"):
            if name == "d1" and not self.d1_written:
                continue   # lives inside the layer-1 gradient kernel: checked through gW1 / gB1
            assert_close(name, self.got[name], self.exp[name], ACT, name in zero, masks.get(name))
        for k in GRAD_KEYS:
            assert_close("g" + k, self.grads[k], self.egrads[k], grad_tol, "g" + k in zero)

    def release(self, ctx):
        ctx.release(self.work)


def assert_launches(chunk, expected):
    if SWITCHED:
        return
    assert chunk.launches == expected, (
        "%d launches, the case expects %d: a kernel of the chunk took another path"
        % (chunk.launches, expected))


# ------------------------------------------------------------------ A. value range
# 9-1-5 64/32 at S = 170 and 9-5-5 at S = 200, samples 33x33: every tensor-core kernel of the
# chunk runs (the training forward, bwd3_tc, wgrad1_fused_tc, wgrad2_tc / the layer-1-only
# forward, conv5_tc forward and deltas, bwd3_tc, wgrad5_tc).  launches: the chunk's count.
RANGE_NETS = [pytest.param(N915, 170, 10, id="915"), pytest.param(N955, 200, 16, id="955")]


def _range_case(ctx, port, cfg, S, launches, tag, params=None, x=None, gt=None, zero=(),
                grad_tol=GRAD):
    w = h = 33
    rng = _rng(tag, cfg)
    p0 = make_params(rng, *cfg)
    x0, gt0 = patches(rng, S, w, h)
    c = Chunk(ctx, port, cfg, p0 if params is None else params(p0, rng),
              x0 if x is None else x(x0, rng), gt0 if gt is None else gt(gt0, rng), w, h, S)
    c.check(zero, grad_tol=grad_tol)
    assert_launches(c, launches)
    c.release(ctx)
    return c


@pytest.mark.parametrize("cfg,S,launches", RANGE_NETS)
def test_reference_initial_scale(ctx, port, cfg, S, launches):
    """`cnn train` starts from N(0, 0.001) weights and zero biases (example_config.json): out3
    ~1e-6, out2 ~1e-4, the layer-1 gradient ~1e-3."""

    def params(p, rng):
        p = make_params(rng, *cfg, sd=0.001, bias_sd=0)
        p["b3"] = np.zeros_like(p["b3"])   # (make_params lifts b3 to keep the output alive)
        return p

    _range_case(ctx, port, cfg, S, launches, "sd1e-3", params=params)


@pytest.mark.parametrize("cfg,S,launches", RANGE_NETS)
def test_large_parameters(ctx, port, cfg, S, launches):
    """He-scaled parameters x30: activations up to ~1e4."""
    _range_case(ctx, port, cfg, S, launches, "x30",
                params=lambda p, rng: {k: (v * 30).astype(np.float32) for k, v in p.items()})


@pytest.mark.parametrize("cfg,S,launches", RANGE_NETS)
def test_unnormalised_luma(ctx, port, cfg, S, launches):
    """Inputs of 0..255 (extract_luma with normalize=false): outside the |x| < 64 domain of the
    9-1-5 training forward (its 3xTF32 kernel redoes the chunk, and max|out2| for bwd3_tc must
    come from that kernel); the 9-5-5 layer-1-only kernel scales from the measured maximum."""
    _range_case(ctx, port, cfg, S, launches, "255",
                x=lambda x, rng: np.round((x - x.min()) * 255).astype(np.float32),
                gt=lambda gt, rng: (gt * 255).astype(np.float32))


@pytest.mark.parametrize("pixel", [63.9, 64.0, 1000.0])
@pytest.mark.parametrize("cfg,S,launches", RANGE_NETS)
def test_input_domain_edge(ctx, port, cfg, S, launches, pixel):
    """Luma-range samples with one pixel at the edge of the FP16 domain (63.9), on it (64) and
    far outside (1000), in the last row of the last sample."""

    def x(x0, rng):
        x1 = x0.copy()
        x1[-1, -1, 20] = pixel
        return x1

    # the layer-3 gradient of the 9-1-5 chunk with the 1000 pixel sums terms of up to ~1e4 next
    # to terms of ~1: bwd3_tc's FP32 tensor-memory accumulator keeps it to 3e-6 of its largest
    # entry (measured on a B200)
    grad_tol = (1e-4, 4e-6) if pixel > 64 else GRAD
    _range_case(ctx, port, cfg, S, launches, "edge%g" % pixel, x=x, grad_tol=grad_tol)


@pytest.mark.parametrize("cfg,S,launches", RANGE_NETS)
def test_dead_output_layer(ctx, port, cfg, S, launches):
    """b3 = -10: out3 <= 0 everywhere, so d3 = (out3 - gt) [out3 > 0] = 0 (quirk Q2) and every
    delta and gradient below it is exactly zero."""

    def params(p, rng):
        p = dict(p)
        p["b3"] = np.full_like(p["b3"], -10.0)
        return p

    c = _range_case(ctx, port, cfg, S, launches, "dead3", params=params,
                    zero=("d1", "d2", "d3") + tuple("g" + k for k in GRAD_KEYS))
    assert c.exp["out3"].max() <= 0


@pytest.mark.parametrize("cfg,S,launches", RANGE_NETS)
def test_dead_layer1(ctx, port, cfg, S, launches):
    """b1 = -10: out1 = 0 everywhere (its measured maximum is 0 and the split operands take the
    scale of 0), out2 = relu(b2), and gW1, gB1, gW2 are exactly zero."""

    def params(p, rng):
        p = dict(p)
        p["b1"] = np.full_like(p["b1"], -10.0)
        return p

    c = _range_case(ctx, port, cfg, S, launches, "dead1", params=params,
                    zero=("out1", "d1", "gw1", "gb1", "gw2"))
    relu_b2 = np.maximum(c.params["b2"], 0)
    np.testing.assert_array_equal(c.got["out2"], np.broadcast_to(relu_b2, c.got["out2"].shape))


@pytest.mark.parametrize("cfg,S,launches", RANGE_NETS)
def test_ground_truth_outlier(ctx, port, cfg, S, launches):
    """One ground-truth pixel at 1e3: max|d3| (the scale of d3's split operand) follows it;
    every delta outside the outlier's footprint must still meet the bound at its own scale."""
    w = h = 33
    rng = _rng("outlier", cfg)
    params = make_params(rng, *cfg)
    x, gt = patches(rng, S, w, h)
    # a pixel of sample S / 2 where out3 > 0 (d3 = 0 where out3 <= 0: quirk Q2), 5 from the edges
    s, pad = S // 2, (sum(cfg[2:]) - 3) // 2
    _, _, o3 = port.net_forward(NetState(*cfg, params), x[s:s + 1], w, h, 1)
    inner = o3[0, 5:-5, 5:-5]
    y3, x3 = (int(v) + 5 for v in np.unravel_index(np.argmax(inner), inner.shape))
    gt[s, pad + y3, pad + x3] = 1e3
    c = Chunk(ctx, port, cfg, params, x, gt, w, h, S)
    assert c.exp["d3"][s, y3, x3] < -100, "the outlier must reach d3 (out3 > 0 there)"
    # footprint of the outlier: d3 at one pixel, d2 over the f3 x f3 window below it, d1 over
    # f2 + f3 - 1
    f2, f3 = cfg[3], cfg[4]
    masks = {}
    for name, extent in (("d3", 1), ("d2", f3), ("d1", f2 + f3 - 1)):
        m = np.ones(c.exp[name].shape[:3], bool)
        m[s, y3:y3 + extent, x3:x3 + extent] = False
        masks[name] = np.broadcast_to(m[..., None], c.exp[name].shape) if name != "d3" else m
    c.check(masks=masks)
    assert_close("d3 outlier", c.got["d3"][s, y3, x3], c.exp["d3"][s, y3, x3], ACT)
    assert_launches(c, launches)
    c.release(ctx)


# ------------------------------------------------------------------ B. geometry
GEOMETRY = [
    # net, w, h, S, launches
    # 9-5-5: w3 = 1 (out1 9 wide, lower than conv5_tc's accumulator ring)
    pytest.param(N955, 17, 17, 460, 16, id="955-w17"),
    # w1 = 100 / 101: the widest layer-2 gradient wgrad5_tc takes / the FP32 split-K kernel.  Both
    # launch a contraction and a reduce: these twins differ in path, not in count.
    pytest.param(N955, 108, 33, 41, 16, id="955-w108"),
    pytest.param(N955, 109, 33, 41, 16, id="955-w109"),
    # w1 = 128 / 129: one 128-column strip per sample, and one strip plus a column.  S = 32 also
    # ends the layer-1-only kernel's last 124-column strip on the chunk's last out3 column
    # (S w - 12 = 35 * 124): the 4 out1 columns to its right are that strip's to store
    pytest.param(N955, 136, 33, 32, 16, id="955-w136"),
    pytest.param(N955, 137, 33, 32, 16, id="955-w137"),
    # the widest sample of the layer-1-only kernel / layer 1 in FP32 with conv5_tc measuring
    # max|out1| itself
    pytest.param(N955, 512, 20, 9, 16, id="955-w512"),
    pytest.param(N955, 513, 20, 9, 13, id="955-w513"),
    # w1 = 1024 / 1025: the widest sample of conv5_tc / the FP32 layer 2 and layer-1 deltas
    pytest.param(N955, 1032, 18, 4, 13, id="955-w1032"),
    pytest.param(N955, 1033, 18, 4, 10, id="955-w1033"),
    # S w1 = 4096 exactly (conv5_tc runs; bwd3_tc with S w2 = 3584 does not: a mixed chunk), and
    # one sample less (neither runs)
    pytest.param(N955, 40, 33, 128, 16, id="955-w40-S128"),
    pytest.param(N955, 40, 33, 127, 10, id="955-w40-S127"),
    # tall: the 16 / 8-slot accumulator rings wrap many times inside one sample
    pytest.param(N955, 33, 120, 170, 16, id="955-tall"),
    # 9-1-5: out3 124 / 125 columns (one strip of the fused forward, and one more column); at
    # S = 32 the last strip ends on the chunk's last out3 column (as above)
    pytest.param(N915, 136, 33, 32, 10, id="915-w136"),
    pytest.param(N915, 137, 33, 33, 10, id="915-w137"),
    # patches whose last strip ends on the chunk's last out3 column (33 S - 12 = 18 * 124)
    pytest.param(N915, 33, 33, 68, 9, id="915-w33-S68"),
    # wide samples in the fused training forward
    pytest.param(N915, 600, 30, 8, 10, id="915-w600"),
    # bwd3_tc ow = 1024 / 1025: its widest sample / the FP32 kernel
    pytest.param(N915, 1032, 33, 4, 10, id="915-w1032"),
    pytest.param(N915, 1033, 33, 4, 11, id="915-w1033"),
    # tall: bwd3_tc at its tallest sample (64 out2 rows: its plane rings wrap 16 times), and
    # taller samples, which it leaves to the FP32 kernel
    pytest.param(N915, 33, 72, 170, 10, id="915-tall64"),
    pytest.param(N915, 33, 400, 170, 9, id="915-tall"),
]


@pytest.mark.parametrize("cfg,w,h,S,launches", GEOMETRY)
def test_chunk_geometry(ctx, port, cfg, w, h, S, launches):
    rng = _rng("geometry", cfg, w, h, S)
    params = make_params(rng, *cfg)
    x, gt = patches(rng, S, w, h)
    c = Chunk(ctx, port, cfg, params, x, gt, w, h, S)
    c.check()
    assert_launches(c, launches)
    c.release(ctx)


# ------------------------------------------------------------------ C. state between calls
def _d2_region(ctx, chunk):
    """A handle on the chunk workspace's d2 sub-buffer."""
    return ctx.wrap(ctx.mem_ptr(chunk.work) + chunk.offset["d2"], chunk.got["d2"].nbytes)


def _deltas_into_new_target(ctx, chunk, dn_handle):
    (w1, h1), _, _ = chunk.net.out_dims(chunk.w, chunk.h)
    lo = ctx.upload(chunk.got["out1"])
    target = ctx.alloc(chunk.got["out1"].nbytes)
    n0 = ctx.launch_count()
    ctx.deltas(dn_handle, lo, target, chunk.net.c.w[1], 64, 5, 32, w1, h1, chunk.S)
    launches = ctx.launch_count() - n0
    got = ctx.read(target, chunk.got["out1"].shape)
    ctx.release(lo)
    ctx.release(target)
    return got, launches


@pytest.mark.parametrize("factor", [1e3, 1e-3])
def test_deltas_after_chunk_measure_their_own_d2(ctx, port, factor):
    """A standalone srcnn_deltas whose deltas_next is the d2 buffer a 9-5-5 chunk just wrote
    (the C++ pipeline's ConfigBasedDataPipeline::backpropagate on the pools execute_batch used)
    must scale its split operand from max|d2| of the data it is given, not from the maximum the
    chunk's layer-3 backward recorded: new values written into the buffer, and a layer-2
    gradient of another tensor run in between, which overwrites the recorded maximum."""
    cfg, w, h, S = N955, 33, 33, 200
    rng = _rng("stale-d2", factor)
    params = make_params(rng, *cfg)
    x, gt = patches(rng, S, w, h)
    (w1, h1), (w2, h2), _ = pkg.Net(ctx, *cfg, params).out_dims(w, h)

    # 1. new values in the chunk's d2 buffer
    c = Chunk(ctx, port, cfg, params, x, gt, w, h, S, oracle=False)
    d2 = (c.got["d2"] * factor).astype(np.float32)
    hd2 = _d2_region(ctx, c)
    ctx.write(hd2, d2)
    got, launches = _deltas_into_new_target(ctx, c, hd2)
    exp = port.deltas(d2, c.got["out1"], params["w2"], 64, 5, 32, w1, h1, S)
    assert_close("d1 (d2 x %g written after the chunk)" % factor, got, exp, ACT)
    if not SWITCHED:
        assert launches == 2, "conv5_tc deltas: absmax of d2 + contraction (%d launches)" % launches
    ctx.release(hd2)
    c.release(ctx)

    # 2. the chunk's own d2, after a layer-2 gradient of a tensor `factor` times smaller / larger
    c = Chunk(ctx, port, cfg, params, x, gt, w, h, S, oracle=False)
    other_d = (c.got["d2"][::-1] / factor).astype(np.float32)
    other_in = np.ascontiguousarray(c.got["out1"][::-1])
    md, mi = ctx.upload(other_d), ctx.upload(other_in)
    gw, gb = ctx.zeros(params["w2"].size), ctx.zeros(32)
    ctx.backpropagate(md, mi, gw, gb, 32, 64, 5, w2, h2, S)
    hd2 = _d2_region(ctx, c)
    got, launches = _deltas_into_new_target(ctx, c, hd2)
    exp = port.deltas(c.got["d2"], c.got["out1"], params["w2"], 64, 5, 32, w1, h1, S)
    assert_close("d1 (after a layer-2 gradient of d2 / %g)" % factor, got, exp, ACT)
    if not SWITCHED:
        assert launches == 2, "conv5_tc deltas: absmax of d2 + contraction (%d launches)" % launches
    for m in (md, mi, gw, gb, hd2):
        ctx.release(m)
    c.release(ctx)


def test_conv5_weight_image_follows_the_parameters(ctx, port):
    """conv5_tc packs W2 into FP16 hi / lo images once per context and reuses them while the
    buffer is untouched.  Every way W2 can change must re-pack it: a host write, a device copy,
    a fill, the training update, and a write through a raw-pointer alias announced with
    srcnn_invalidate_params.  Checked through a standalone layer-2 forward (the first call after
    a change re-packs, the second is served from the cache) and through a training chunk."""
    cfg, w, h, S = N955, 33, 33, 200
    rng = _rng("c5-image")
    params = make_params(rng, *cfg)
    x, gt = patches(rng, S, w, h)
    net = pkg.Net(ctx, *cfg, params)
    (w1, h1), (w2, h2), _ = net.out_dims(w, h)
    S1 = 170    # standalone layer-2 forward: S1 * w1 >= 32 * 128 takes conv5_tc
    x1 = np.maximum(rng.normal(0, 1, (S1, h1, w1, 64)), 0).astype(np.float32)
    mi1, mo1 = ctx.upload(x1), ctx.alloc(4 * S1 * w2 * h2 * 32)
    mi, mg = ctx.upload(x), ctx.upload(gt)
    work = ctx.alloc(net.train_workspace_bytes(w, h, S))
    off2 = (S * h1 * w1 * 64 * 4 + 255) // 256 * 256

    def check(p, what, cached=True):
        exp1 = port.forward(x1, p["w2"], p["b2"], 64, 32, 5, False, w1, h1, S1)
        for call, repack in ((1, True), (2, not cached)):
            n0 = ctx.launch_count()
            ctx.forward_layer(mi1, mo1, net.c.w[1], net.c.b[1], 64, 32, 5, False, w1, h1, S1)
            launches = ctx.launch_count() - n0
            assert_close("out2 of the layer-2 forward (%s, call %d)" % (what, call),
                         ctx.read(mo1, exp1.shape), exp1, ACT)
            if not SWITCHED:   # absmax + contraction, + the packing kernel
                assert launches == 2 + repack, "%s, call %d: %d launches" % (what, call, launches)
        net.train_chunk(mi, mg, w, h, S, work)
        on = NetState(*cfg, p)
        _, exp2, _ = port.net_forward(on, x, w, h, S)
        assert_close("out2 of a chunk (%s)" % what, ctx.read(work, exp2.shape, offset=off2), exp2, ACT)

    check(params, "initial parameters")
    # host write
    p = dict(params, w2=(params["w2"] * 1.5).astype(np.float32))
    ctx.write(net.c.w[1], p["w2"])
    check(p, "host write")
    # device-to-device copy
    p = dict(params, w2=(params["w2"][::-1] * 0.75).astype(np.float32))
    tmp = ctx.upload(p["w2"])
    ctx.copy(tmp, net.c.w[1])
    ctx.release(tmp)
    check(p, "device copy")
    # fill
    p = dict(p, w2=np.full_like(params["w2"], 0.002))
    ctx.fill_float(net.c.w[1], 0.002)
    check(p, "fill")
    # the training update, with a learning rate that moves W2 by half its size
    g = net.grads()
    lr2 = 0.5 * float(np.abs(p["w2"]).max()) * S / float(np.abs(g["w2"]).max())
    net.update_all(S, 0.0, 0.0, np.array([0.0, lr2, 0.0], np.float32))
    p = net.params()
    assert float(np.abs(p["w2"] - 0.002).max()) > 1e-4
    check(p, "update_all")
    # a write the device layer cannot see, through an alias of the raw pointer
    alias = ctx.wrap(ctx.mem_ptr(net.c.w[1]), 4 * params["w2"].size)
    check(p, "raw pointer taken", cached=False)
    p = dict(p, w2=(params["w2"] * -0.5).astype(np.float32))
    ctx.write(alias, p["w2"])
    ctx.invalidate_params()
    check(p, "write through an alias + srcnn_invalidate_params", cached=False)
    for m in (alias, mi1, mo1, mi, mg, work):
        ctx.release(m)

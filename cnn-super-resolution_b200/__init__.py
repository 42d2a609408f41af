"""cnn-super-resolution_b200 -- B200 (sm_100a) SRCNN hot path behind the reference's interface.

The product is native: ``csrc/`` (hand-written CUDA kernels + the C-ABI of
``include/srcnn_b200.h``) and ``host/`` (C++ ``DataPipeline`` / ``ConfigBasedDataPipeline`` /
``LayerData`` / ``Config`` / the ``cnn`` CLI, which call only the C-ABI).  This Python module
is a thin ctypes binding over the same C-ABI, used by tests/ and bench.py and for the
torch.distributed plumbing of the multi-GPU paths.  It never computes anything itself and it
never imports oracle/: if ``libsrcnn_b200.so`` is missing or there is no CUDA device, it
raises.
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
LIB_PATH = os.environ.get("SRCNN_B200_LIB") or os.path.join(HERE, "libsrcnn_b200.so")
HEADER = os.path.join(ROOT, "include", "srcnn_b200.h")

NULL_MEM = 1 << 30

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]

KERNEL_IDS = ["forward", "squared_err", "last_layer_delta", "deltas", "backpropagate",
              "update_params", "sum", "sub_from_all", "extract_luma", "swap_luma",
              "forward_fused", "train_fused", "resample", "quality"]

RESAMPLE_FILTERS = {"bicubic": 0, "lanczos": 1}   # SRCNN_RESAMPLE_BICUBIC / _LANCZOS


class SrcnnError(RuntimeError):
    pass


def build(verbose=False, force=False):
    """Compile csrc/ for sm_100a into libsrcnn_b200.so (in-tree, so it travels to the GPU box)."""
    srcs = [os.path.join(HERE, "csrc", f) for f in sorted(os.listdir(os.path.join(HERE, "csrc")))]
    deps = srcs + [HEADER]
    if (not force and os.path.exists(LIB_PATH)
            and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(d) for d in deps)):
        return LIB_PATH
    cmd = ["nvcc"] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
          ["-o", LIB_PATH, os.path.join(HERE, "csrc", "srcnn.cu")]
    subprocess.check_call(cmd)
    return LIB_PATH


_lib = None

_u64 = C.c_uint64
_vp = C.c_void_p
_i = C.c_int
_f = C.c_float
_u = C.c_uint
_sz = C.c_size_t


class CNet(C.Structure):
    """struct srcnn_net of include/srcnn_b200.h"""
    _fields_ = [("n1", _i), ("n2", _i), ("f1", _i), ("f2", _i), ("f3", _i),
                ("w", _u64 * 3), ("b", _u64 * 3),
                ("grad_w", _u64 * 3), ("grad_b", _u64 * 3),
                ("prev_dw", _u64 * 3), ("prev_db", _u64 * 3)]


YUV420_FORMATS = {"i420": 0, "nv12": 1}   # SRCNN_YUV_I420 / _NV12
# SRCNN_CHROMA_CENTER / _LEFT / _TOPLEFT, by ffmpeg's chroma_location names
CHROMA_SITINGS = {"center": 0, "left": 1, "topleft": 2}


class CYuv420Layout(C.Structure):
    """struct srcnn_yuv420_layout of include/srcnn_b200.h"""
    _fields_ = [("format", _i), ("frame_stride", _sz), ("y_pitch", _sz), ("c_pitch", _sz),
                ("cb_offset", _sz), ("cr_offset", _sz), ("chroma_siting", _i), ("bit_depth", _i)]


def _siting_id(name):
    if name not in CHROMA_SITINGS:
        raise ValueError("unknown chroma siting %r (have %s)" % (name, sorted(CHROMA_SITINGS)))
    return CHROMA_SITINGS[name]


def yuv420_layout(fmt, w, h, y_pitch=None, c_pitch=None, cb_offset=None, frame_stride=None,
                  chroma_siting="center", bit_depth=8):
    """Where the planes of w x h 4:2:0 frames ("i420" or "nv12") lie in a buffer, in bytes, and
    where their chroma samples sit (CHROMA_SITINGS).  bit_depth 10 makes them I010 ("i420") or
    P010 ("nv12"), a 16-bit word a sample.  The defaults are the dense layout; otherwise the chroma
    follows Y at cb_offset (default: right after the Y plane's h rows), an I420 Cr plane follows Cb
    right after its h/2 rows, and a frame spans frame_stride bytes (default: to the end of its last
    plane's last pitched row)."""
    if fmt not in YUV420_FORMATS:
        raise ValueError("unknown 4:2:0 format %r (have %s)" % (fmt, sorted(YUV420_FORMATS)))
    if bit_depth not in (8, 10):
        raise ValueError("bit depth %r is not 8 or 10" % (bit_depth,))
    siting = _siting_id(chroma_siting)
    nv12 = fmt == "nv12"
    b = 2 if bit_depth == 10 else 1   # bytes a sample
    y_pitch = w * b if y_pitch is None else y_pitch
    c_pitch = (w if nv12 else w // 2) * b if c_pitch is None else c_pitch
    cb_offset = h * y_pitch if cb_offset is None else cb_offset
    cr_offset = 0 if nv12 else cb_offset + (h // 2) * c_pitch
    end = (cb_offset if nv12 else cr_offset) + (h // 2) * c_pitch
    return CYuv420Layout(YUV420_FORMATS[fmt], end if frame_stride is None else frame_stride,
                         y_pitch, c_pitch, cb_offset, cr_offset, siting, bit_depth)


_SIGS = {
    "srcnn_ctx_create": (_i, [_i, _i, C.POINTER(_vp)]),
    "srcnn_ctx_create_on_stream": (_i, [_i, _vp, _i, C.POINTER(_vp)]),
    "srcnn_ctx_destroy": (_i, [_vp]),
    "srcnn_last_error": (C.c_char_p, []),
    "srcnn_block": (_i, [_vp]),
    "srcnn_device_info": (_i, [_vp, C.c_char_p, _sz, C.POINTER(_i), C.POINTER(_sz)]),
    "srcnn_profile_get": (_i, [_vp, _i, C.POINTER(_u64), C.POINTER(_u64)]),
    "srcnn_launch_count": (_i, [_vp, C.POINTER(_u64)]),
    "srcnn_stream": (_i, [_vp, C.POINTER(_vp)]),
    "srcnn_alloc": (_i, [_vp, _sz, C.POINTER(_u64)]),
    "srcnn_wrap": (_i, [_vp, _vp, _sz, C.POINTER(_u64)]),
    "srcnn_release": (_i, [_vp, _u64]),
    "srcnn_mem_size": (_i, [_vp, _u64, C.POINTER(_sz)]),
    "srcnn_mem_ptr": (_i, [_vp, _u64, C.POINTER(_vp)]),
    "srcnn_mem_usage": (_i, [_vp, C.POINTER(_sz)]),
    "srcnn_write": (_i, [_vp, _u64, _sz, _sz, _vp, _i]),
    "srcnn_read": (_i, [_vp, _u64, _sz, _sz, _vp, _i]),
    "srcnn_copy": (_i, [_vp, _u64, _u64, _sz]),
    "srcnn_copy_region": (_i, [_vp, _u64, _sz, _u64, _sz, _sz]),
    "srcnn_gather": (_i, [_vp, C.POINTER(_u64), _i, _sz, _u64]),
    "srcnn_fill_float": (_i, [_vp, _u64, _f]),
    "srcnn_host_alloc": (_i, [_sz, C.POINTER(_vp)]),
    "srcnn_host_free": (_i, [_vp]),
    "srcnn_forward_layer": (_i, [_vp, _u64, _u64, _u64, _u64] + [_i] * 7),
    "srcnn_squared_error": (_i, [_vp, _u64, _u64, _u64] + [_i] * 5),
    "srcnn_last_layer_delta": (_i, [_vp, _u64, _u64, _u64] + [_i] * 5),
    "srcnn_deltas": (_i, [_vp, _u64, _u64, _u64, _u64] + [_i] * 6),
    "srcnn_backpropagate": (_i, [_vp, _u64, _u64, _u64, _u64] + [_i] * 6),
    "srcnn_update_params": (_i, [_vp] + [_u64] * 6 + [_f] * 3 + [_u] * 3),
    "srcnn_sum": (_i, [_vp, _u64, _u, _i, _u64]),
    "srcnn_sub_from_all": (_i, [_vp, _u64, _f, _u]),
    "srcnn_extract_luma": (_i, [_vp, _u64, _u64, _i, _i, _i]),
    "srcnn_swap_luma": (_i, [_vp, _u64, _u64, _u64] + [_i] * 4),
    "srcnn_resample": (_i, [_vp, _u64, _i, _i, _u64, _u64, _i, _i, _i]),
    "srcnn_upscale_image_host": (_i, [_vp, C.POINTER(CNet), _vp, _i, _i, _i, _i, _i, _vp]),
    "srcnn_upscale_frames_host": (_i, [_vp, C.POINTER(CNet), _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "srcnn_upscale_yuv420_frames_host": (_i, [_vp, C.POINTER(CNet), _vp, _i, _i, _i, _i, _i, _i,
                                              _vp]),
    "srcnn_upscale_yuv420_frames_host_sited": (_i, [_vp, C.POINTER(CNet), _vp, _i, _i, _i, _i,
                                                    _i, _i, _i, _i, _vp]),
    "srcnn_upscale_yuv420p10_frames_host": (_i, [_vp, C.POINTER(CNet), _vp, _i, _i, _i, _i, _i,
                                                 _i, _i, _i, _vp]),
    "srcnn_upscale_yuv420_frames": (_i, [_vp, C.POINTER(CNet), _u64, C.POINTER(CYuv420Layout), _i,
                                         _i, _i, _u64, C.POINTER(CYuv420Layout), _i, _i, _i]),
    "srcnn_image_quality": (_i, [_vp, _u64, _i, _u64, _i, _i, _i, _i, _u64]),
    "srcnn_evaluate_frames_host": (_i, [_vp, C.POINTER(CNet), _vp, _i, _i, _i, _i, _i, _i, _vp,
                                        _i, _vp, _vp]),
    "srcnn_forward_fused_supported": (_i, [C.POINTER(CNet)]),
    "srcnn_forward_fused": (_i, [_vp, C.POINTER(CNet), _u64, _u64, _i, _i, _i, _u64, _u64]),
    "srcnn_infer_rows_host": (_i, [_vp, C.POINTER(CNet), _vp, _i, _i, _i, _i, _vp]),
    "srcnn_infer_rows_host_async": (_i, [_vp, C.POINTER(CNet), _vp, _i, _i, _i, _i, _vp]),
    "srcnn_infer_frames_host": (_i, [_vp, C.POINTER(CNet), _vp, _i, _i, _i, _vp]),
    "srcnn_train_chunk": (_i, [_vp, C.POINTER(CNet), _u64, _u64, _i, _i, _i, _u64]),
    "srcnn_train_chunks_host": (_i, [_vp, C.POINTER(CNet), _vp, _vp, _i, _i, _i, _i, _u64]),
    "srcnn_train_chunk_buffers": (_i, [_vp, C.POINTER(CNet), _u64, _u64, _i, _i, _i,
                                       _u64, _u64, _u64, _u64, _u64, _u64]),
    "srcnn_train_workspace_bytes": (_sz, [C.POINTER(CNet), _i, _i, _i]),
    "srcnn_train_materializes_d1": (_i, [_vp, C.POINTER(CNet)]),
    "srcnn_update_all": (_i, [_vp, C.POINTER(CNet), _u, _f, _f, C.POINTER(_f)]),
    "srcnn_validate_chunk": (_i, [_vp, C.POINTER(CNet), _u64, _u64, _i, _i, _i, _u64, _u64]),
    "srcnn_invalidate_params": (_i, [_vp]),
    "srcnn_comm_unique_id": (_i, [_vp]),
    "srcnn_comm_init": (_i, [_vp, _i, _i, _vp]),
    "srcnn_comm_destroy": (_i, [_vp]),
    "srcnn_comm_info": (_i, [_vp, C.POINTER(_i), C.POINTER(_i)]),
    "srcnn_allreduce_sum": (_i, [_vp, _u64, _sz, _sz]),
    "srcnn_allreduce_grads": (_i, [_vp, C.POINTER(CNet)]),
    "srcnn_broadcast": (_i, [_vp, _u64, _sz, _i]),
}


def exported_symbols():
    """Every entry point declared in include/srcnn_b200.h (checked by the CPU test-suite)."""
    return sorted(_SIGS)


def lib():
    """Load libsrcnn_b200.so.  Raises if it has not been built -- there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SrcnnError("%s is missing: run `python -c 'import __graft_entry__ as g; "
                             "g.build()'` (nvcc, sm_100a) first; there is no CPU fallback"
                             % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        raise SrcnnError("srcnn error %d: %s" % (rc, lib().srcnn_last_error().decode()))


def _filter_id(name):
    if name not in RESAMPLE_FILTERS:
        raise ValueError("unknown resample filter %r (have %s)" % (name, sorted(RESAMPLE_FILTERS)))
    return RESAMPLE_FILTERS[name]


def _np_ptr(a):
    return C.c_void_p(a.ctypes.data)


class PinnedBuffer:
    """Page-locked host staging buffer (srcnn_host_alloc) exposed as a numpy array."""

    def __init__(self, shape, dtype=np.float32):
        self.shape = tuple(shape)
        self.dtype = np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        p = _vp()
        _check(lib().srcnn_host_alloc(self.nbytes, C.byref(p)))
        self.ptr = p.value
        buf = (C.c_char * self.nbytes).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=self.dtype).reshape(self.shape)

    def free(self):
        if self.ptr:
            self.array = None
            lib().srcnn_host_free(_vp(self.ptr))
            self.ptr = None


class Context:
    """One device + one in-order stream + a handle table.
    Mirrors opencl::Context (reference: src/opencl/Context.hpp:72-299)."""

    def __init__(self, device=0, profile=False, stream=None):
        L = lib()
        h = _vp()
        if stream is None:
            _check(L.srcnn_ctx_create(device, int(profile), C.byref(h)))
        else:
            _check(L.srcnn_ctx_create_on_stream(device, _vp(stream), int(profile), C.byref(h)))
        self.h = h
        self.L = L
        self.device = device

    # -- lifetime / info --
    def close(self):
        if self.h:
            self.L.srcnn_ctx_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def block(self):
        _check(self.L.srcnn_block(self.h))

    def device_info(self):
        name = C.create_string_buffer(256)
        sm, mem = _i(), _sz()
        _check(self.L.srcnn_device_info(self.h, name, 256, C.byref(sm), C.byref(mem)))
        return name.value.decode(), sm.value, mem.value

    def launch_count(self):
        n = _u64()
        _check(self.L.srcnn_launch_count(self.h, C.byref(n)))
        return n.value

    def profile(self):
        out = {}
        for i, name in enumerate(KERNEL_IDS):
            ns, n = _u64(), _u64()
            _check(self.L.srcnn_profile_get(self.h, i, C.byref(ns), C.byref(n)))
            out[name] = (ns.value, n.value)
        return out

    def stream(self):
        p = _vp()
        _check(self.L.srcnn_stream(self.h, C.byref(p)))
        return p.value

    # -- multi-GPU (NCCL communicator owned by the context) --
    @staticmethod
    def comm_unique_id():
        """128-byte NCCL id created on rank 0; hand it to the other ranks."""
        buf = (C.c_ubyte * 128)()
        _check(lib().srcnn_comm_unique_id(C.cast(buf, _vp)))
        return bytes(buf)

    def comm_init(self, rank, world, unique_id):
        buf = (C.c_ubyte * 128).from_buffer_copy(bytes(unique_id))
        _check(self.L.srcnn_comm_init(self.h, rank, world, C.cast(buf, _vp)))

    def comm_destroy(self):
        _check(self.L.srcnn_comm_destroy(self.h))

    def comm_info(self):
        r, w = _i(), _i()
        _check(self.L.srcnn_comm_info(self.h, C.byref(r), C.byref(w)))
        return r.value, w.value

    def allreduce_sum(self, mem, count, offset=0):
        _check(self.L.srcnn_allreduce_sum(self.h, mem, offset, count))

    def broadcast(self, mem, count, root=0):
        _check(self.L.srcnn_broadcast(self.h, mem, count, root))

    def invalidate_params(self):
        _check(self.L.srcnn_invalidate_params(self.h))

    # -- memory --
    def alloc(self, nbytes):
        m = _u64()
        _check(self.L.srcnn_alloc(self.h, int(nbytes), C.byref(m)))
        return m.value

    def wrap(self, device_ptr, nbytes):
        m = _u64()
        _check(self.L.srcnn_wrap(self.h, _vp(device_ptr), int(nbytes), C.byref(m)))
        return m.value

    def release(self, mem):
        _check(self.L.srcnn_release(self.h, mem))

    def mem_size(self, mem):
        s = _sz()
        _check(self.L.srcnn_mem_size(self.h, mem, C.byref(s)))
        return s.value

    def mem_ptr(self, mem):
        p = _vp()
        _check(self.L.srcnn_mem_ptr(self.h, mem, C.byref(p)))
        return p.value

    def mem_usage(self):
        s = _sz()
        _check(self.L.srcnn_mem_usage(self.h, C.byref(s)))
        return s.value

    def write(self, mem, array, offset=0, block=True):
        a = np.ascontiguousarray(array)
        _check(self.L.srcnn_write(self.h, mem, offset, a.nbytes, _np_ptr(a), int(block)))

    def read(self, mem, shape, dtype=np.float32, offset=0):
        out = np.empty(shape, dtype)
        _check(self.L.srcnn_read(self.h, mem, offset, out.nbytes, _np_ptr(out), 1))
        return out

    def upload(self, array, dtype=np.float32):
        a = np.ascontiguousarray(array, dtype)
        m = self.alloc(max(a.nbytes, 4))
        if a.nbytes:
            self.write(m, a)
        return m

    def zeros(self, nfloats):
        m = self.alloc(4 * max(int(nfloats), 1))
        self.fill_float(m, 0.0)
        return m

    def copy(self, src, dst, dst_offset=0):
        _check(self.L.srcnn_copy(self.h, src, dst, dst_offset))

    def copy_region(self, src, src_offset, dst, dst_offset, nbytes):
        _check(self.L.srcnn_copy_region(self.h, src, src_offset, dst, dst_offset, nbytes))

    def gather(self, handles, nbytes_each, dst):
        """copies the equally-sized buffers `handles` into consecutive slots of dst (one launch)"""
        arr = (_u64 * len(handles))(*handles)
        _check(self.L.srcnn_gather(self.h, arr, len(handles), int(nbytes_each), dst))

    def fill_float(self, mem, value):
        _check(self.L.srcnn_fill_float(self.h, mem, float(value)))

    # -- kernels (one per reference .cl entry point) --
    def forward_layer(self, inp, out, W, B, k, n, f, skip_relu, in_w, in_h, S=1):
        _check(self.L.srcnn_forward_layer(self.h, inp, out, W, B, k, n, f, int(skip_relu),
                                          in_w, in_h, S))

    def squared_error(self, gt, algo, target, gt_w, gt_h, algo_w, algo_h, S=1):
        _check(self.L.srcnn_squared_error(self.h, gt, algo, target, gt_w, gt_h, algo_w, algo_h, S))

    def last_layer_delta(self, gt, algo, target, gt_w, gt_h, algo_w, algo_h, S=1):
        _check(self.L.srcnn_last_layer_delta(self.h, gt, algo, target, gt_w, gt_h, algo_w,
                                             algo_h, S))

    def deltas(self, deltas_next, layer_output, target, W, n_curr, f_next, n_next, out_w, out_h,
               S=1):
        _check(self.L.srcnn_deltas(self.h, deltas_next, layer_output, target, W, n_curr, f_next,
                                   n_next, out_w, out_h, S))

    def backpropagate(self, deltas, layer_input, grad_w, grad_b, n, k, f, out_w, out_h, S=1):
        _check(self.L.srcnn_backpropagate(self.h, deltas, layer_input, grad_w, grad_b, n, k, f,
                                          out_w, out_h, S))

    def update_params(self, w, b, gw, gb, pdw, pdb, momentum, decay, lr, batch, wsize, bsize):
        _check(self.L.srcnn_update_params(self.h, w, b, gw, gb, pdw, pdb, momentum, decay, lr,
                                          batch, wsize, bsize))

    def sum(self, data, length, squared, target):
        _check(self.L.srcnn_sum(self.h, data, length, int(squared), target))

    def sub_from_all(self, data, value, length):
        _check(self.L.srcnn_sub_from_all(self.h, data, value, length))

    def extract_luma(self, rgba, target, w, h, normalize=True):
        _check(self.L.srcnn_extract_luma(self.h, rgba, target, w, h, int(normalize)))

    def swap_luma(self, rgba, new_luma, target, gt_w, gt_h, luma_w, luma_h):
        _check(self.L.srcnn_swap_luma(self.h, rgba, new_luma, target, gt_w, gt_h, luma_w, luma_h))

    def resample(self, rgba_in, w, h, rgba_out, out_w, out_h, resample="lanczos",
                 luma_out=NULL_MEM):
        """Pillow-exact enlargement of a w x h RGBA8 image to out_w x out_h RGBA8 (alpha 255),
        with its normalized luma in luma_out unless that is NULL_MEM."""
        _check(self.L.srcnn_resample(self.h, rgba_in, w, h, rgba_out, luma_out, out_w, out_h,
                                     _filter_id(resample)))

    def image_quality(self, result_mem, reference_mem, w, h, S, border, result_bpp=3):
        """{mse, ssim} of S w x h result frames (RGB8, or RGBA8 with result_bpp=4) against S RGBA8
        reference frames on the device, over [border, w-border) x [border, h-border) of the
        normalized luma: float64 [S, 2].  PSNR = 10 log10(1 / mse)."""
        out = self.alloc(16 * S)
        try:
            _check(self.L.srcnn_image_quality(self.h, result_mem, result_bpp, reference_mem, w, h,
                                              S, border, out))
            return self.read(out, (S, 2), np.float64)
        finally:
            self.release(out)


class Net:
    """Device-resident parameters, gradient accumulators and momentum state of the three
    layers (reference: GpuAllocationPool / LayerAllocationPool, src/DataPipeline.hpp:11-29,
    src/ConfigBasedDataPipeline.hpp:33-39) plus the fused entry points."""

    def __init__(self, ctx, n1, n2, f1, f2, f3, params, grad_flat=None):
        self.ctx = ctx
        self.n1, self.n2, self.f1, self.f2, self.f3 = n1, n2, f1, f2, f3
        c = CNet()
        c.n1, c.n2, c.f1, c.f2, c.f3 = n1, n2, f1, f2, f3
        self.sizes = []
        for l, (k, n, f) in enumerate(self.shapes()):
            ws, bs = f * f * k * n, n
            w = np.ascontiguousarray(params["w%d" % (l + 1)], np.float32).reshape(-1)
            b = np.ascontiguousarray(params["b%d" % (l + 1)], np.float32).reshape(-1)
            assert w.size == ws and b.size == bs, (l, w.size, ws, b.size, bs)
            c.w[l], c.b[l] = ctx.upload(w), ctx.upload(b)
            c.prev_dw[l], c.prev_db[l] = ctx.zeros(ws), ctx.zeros(bs)
            self.sizes.append((ws, bs))
        # the six gradient tensors live in ONE contiguous buffer so that data-parallel
        # training needs a single all-reduce (SURVEY 8e); grad_flat may be caller memory
        # (a torch tensor) registered with Context.wrap.
        self.grad_count = sum(ws + bs for ws, bs in self.sizes)
        if grad_flat is None:
            self.grad_flat = ctx.zeros(self.grad_count)
        else:
            self.grad_flat = grad_flat
        base = ctx.mem_ptr(self.grad_flat)
        off = 0
        for l, (ws, bs) in enumerate(self.sizes):
            c.grad_w[l] = ctx.wrap(base + 4 * off, 4 * ws)
            off += ws
            c.grad_b[l] = ctx.wrap(base + 4 * off, 4 * bs)
            off += bs
        self.c = c

    def shapes(self):
        return [(1, self.n1, self.f1), (self.n1, self.n2, self.f2), (self.n2, 1, self.f3)]

    def out_dims(self, w, h):
        w1, h1 = w - self.f1 + 1, h - self.f1 + 1
        w2, h2 = w1 - self.f2 + 1, h1 - self.f2 + 1
        return (w1, h1), (w2, h2), (w2 - self.f3 + 1, h2 - self.f3 + 1)

    @property
    def padding(self):
        """Config::total_padding (reference: src/Config.cpp:44)"""
        return self.f1 + self.f2 + self.f3 - 3

    def fused_supported(self):
        return bool(self.ctx.L.srcnn_forward_fused_supported(C.byref(self.c)))

    def forward_fused(self, inp, out, w, h, S=1, scratch1=NULL_MEM, scratch2=NULL_MEM):
        _check(self.ctx.L.srcnn_forward_fused(self.ctx.h, C.byref(self.c), inp, out, w, h, S,
                                              scratch1, scratch2))

    def infer_rows_host(self, host_in, w, h, row0, row1, host_out, block=True):
        """host_in: full [h][w] float32 image; host_out: array whose first row is output row row0.
        block=False queues the call (two can be in flight); Context.block() completes them."""
        assert host_in.dtype == np.float32 and host_out.dtype == np.float32
        fn = self.ctx.L.srcnn_infer_rows_host if block else self.ctx.L.srcnn_infer_rows_host_async
        _check(fn(self.ctx.h, C.byref(self.c), _np_ptr(host_in), w, h, row0, row1,
                  _np_ptr(host_out)))

    def upscale_image_host(self, rgba, out_w, out_h, resample="lanczos", out=None):
        """rgba: uint8 [h][w][4] (alpha ignored) -> uint8 [out_h][out_w][3]: the image enlarged
        with Pillow's filter, then the `cnn` forward mode on it (luma through the network,
        swapped back into the enlarged image).  `out` may be a preallocated (pinned) array."""
        assert rgba.dtype == np.uint8 and rgba.ndim == 3 and rgba.shape[2] == 4
        rgba = np.ascontiguousarray(rgba)
        if out is None:
            out = np.empty((out_h, out_w, 3), np.uint8)
        assert out.dtype == np.uint8 and out.shape == (out_h, out_w, 3) and out.flags.c_contiguous
        _check(self.ctx.L.srcnn_upscale_image_host(self.ctx.h, C.byref(self.c), _np_ptr(rgba),
                                                   rgba.shape[1], rgba.shape[0], out_w, out_h,
                                                   _filter_id(resample), _np_ptr(out)))
        return out

    def upscale_frames_host(self, rgba, out_w, out_h, resample="lanczos", out=None):
        """rgba: uint8 [n][h][w][4] frames (alpha ignored) -> uint8 [n][out_h][out_w][3]: frame i
        is what upscale_image_host returns for rgba[i]; upload, device work and download of
        consecutive frame groups overlap.  `out` may be a preallocated (pinned) array."""
        assert rgba.dtype == np.uint8 and rgba.ndim == 4 and rgba.shape[3] == 4
        rgba = np.ascontiguousarray(rgba)
        n = rgba.shape[0]
        if out is None:
            out = np.empty((n, out_h, out_w, 3), np.uint8)
        assert out.dtype == np.uint8 and out.shape == (n, out_h, out_w, 3) and out.flags.c_contiguous
        _check(self.ctx.L.srcnn_upscale_frames_host(self.ctx.h, C.byref(self.c), _np_ptr(rgba),
                                                    rgba.shape[2], rgba.shape[1], n, out_w, out_h,
                                                    _filter_id(resample), _np_ptr(out)))
        return out

    def upscale_yuv420_frames_host(self, frames, w, h, out_w, out_h, resample="lanczos", out=None,
                                   chroma_siting="center", out_chroma_siting=None):
        """frames: uint8 [n][w*h*3//2] planar Y'CbCr 4:2:0 (I420: Y, then Cb, then Cr; w and h
        even) -> uint8 [n][out_w*out_h*3//2] I420: Y enlarged with Pillow's filter and its interior
        replaced by the network's luma, Cb and Cr enlarged with the same filter from chroma sited
        at `chroma_siting` to chroma sited at `out_chroma_siting` (CHROMA_SITINGS; None: the
        input's).  `out` may be a preallocated (pinned) array."""
        s_in = _siting_id(chroma_siting)
        s_out = s_in if out_chroma_siting is None else _siting_id(out_chroma_siting)
        n = frames.shape[0]
        assert frames.dtype == np.uint8 and frames.ndim == 2 and frames.shape[1] == w * h * 3 // 2
        frames = np.ascontiguousarray(frames)
        if out is None:
            out = np.empty((n, out_w * out_h * 3 // 2), np.uint8)
        assert out.dtype == np.uint8 and out.shape == (n, out_w * out_h * 3 // 2)
        assert out.flags.c_contiguous
        if s_in == s_out == CHROMA_SITINGS["center"]:
            _check(self.ctx.L.srcnn_upscale_yuv420_frames_host(
                self.ctx.h, C.byref(self.c), _np_ptr(frames), w, h, n, out_w, out_h,
                _filter_id(resample), _np_ptr(out)))
        else:
            _check(self.ctx.L.srcnn_upscale_yuv420_frames_host_sited(
                self.ctx.h, C.byref(self.c), _np_ptr(frames), w, h, n, out_w, out_h,
                _filter_id(resample), s_in, s_out, _np_ptr(out)))
        return out

    def upscale_yuv420p10_frames_host(self, frames, w, h, out_w, out_h, resample="lanczos",
                                      out=None, chroma_siting="center", out_chroma_siting=None):
        """upscale_yuv420_frames_host for 10-bit frames: uint16 [n][w*h*3//2] I010 (the samples of
        I420 frames, each a value in its low 10 bits; the other bits are ignored) -> uint16
        [n][out_w*out_h*3//2] I010 with the upper bits 0: every plane enlarged with Pillow's 16-bit
        filter ("I;16") and capped at 1023, and the interior of Y replaced by the network's luma
        (it reads v / 1023 and writes clamp(out * 1023) truncated).  `out` may be a preallocated
        (pinned) array."""
        s_in = _siting_id(chroma_siting)
        s_out = s_in if out_chroma_siting is None else _siting_id(out_chroma_siting)
        n = frames.shape[0]
        assert frames.dtype == np.uint16 and frames.ndim == 2 and frames.shape[1] == w * h * 3 // 2
        frames = np.ascontiguousarray(frames)
        if out is None:
            out = np.empty((n, out_w * out_h * 3 // 2), np.uint16)
        assert out.dtype == np.uint16 and out.shape == (n, out_w * out_h * 3 // 2)
        assert out.flags.c_contiguous
        _check(self.ctx.L.srcnn_upscale_yuv420p10_frames_host(
            self.ctx.h, C.byref(self.c), _np_ptr(frames), w, h, n, out_w, out_h,
            _filter_id(resample), s_in, s_out, _np_ptr(out)))
        return out

    def upscale_yuv420_frames(self, in_mem, w, h, n_frames, out_mem, out_w, out_h,
                              resample="lanczos", fmt="i420", in_layout=None, out_layout=None,
                              bit_depth=8):
        """upscale_yuv420_frames_host on device memory handles (Context.alloc, or Context.wrap of
        e.g. a torch CUDA tensor's data_ptr()): n_frames frames of w x h in in_mem -> out_w x out_h
        in out_mem, both in `fmt` ("i420" or "nv12") and laid out as in_layout / out_layout
        (yuv420_layout, which also carries the chroma siting and the bit depth; default: dense,
        centre-sited, `bit_depth` bits: 10 is I010 or P010).  Enqueued on the context stream;
        returns at once, without a copy or a host synchronisation."""
        li = yuv420_layout(fmt, w, h, bit_depth=bit_depth) if in_layout is None else in_layout
        lo = yuv420_layout(fmt, out_w, out_h, bit_depth=bit_depth) if out_layout is None else out_layout
        _check(self.ctx.L.srcnn_upscale_yuv420_frames(self.ctx.h, C.byref(self.c), in_mem,
                                                      C.byref(li), w, h, n_frames, out_mem,
                                                      C.byref(lo), out_w, out_h,
                                                      _filter_id(resample)))

    def evaluate_frames_host(self, rgba, reference, out_w, out_h, resample="lanczos", border=None,
                             out=None):
        """upscale_frames_host plus the quality of every frame against its reference (uint8
        [n][out_h][out_w][4] RGBA8): returns (rgb [n][out_h][out_w][3], metrics float64 [n][4]),
        metrics[i] = {mse, ssim} of the network's result, then {mse, ssim} of the plain
        enlargement, over the region `border` pixels in from each edge (None: (f1+f2+f3-3)/2)."""
        assert rgba.dtype == np.uint8 and rgba.ndim == 4 and rgba.shape[3] == 4
        n = rgba.shape[0]
        assert reference.dtype == np.uint8 and reference.shape == (n, out_h, out_w, 4)
        rgba, reference = np.ascontiguousarray(rgba), np.ascontiguousarray(reference)
        if out is None:
            out = np.empty((n, out_h, out_w, 3), np.uint8)
        assert out.dtype == np.uint8 and out.shape == (n, out_h, out_w, 3) and out.flags.c_contiguous
        metrics = np.empty((n, 4), np.float64)
        _check(self.ctx.L.srcnn_evaluate_frames_host(
            self.ctx.h, C.byref(self.c), _np_ptr(rgba), rgba.shape[2], rgba.shape[1], n, out_w,
            out_h, _filter_id(resample), _np_ptr(reference), -1 if border is None else int(border),
            _np_ptr(out), _np_ptr(metrics)))
        return out, metrics

    def infer_frames_host(self, host_in, w, h, host_out):
        """host_in: [n][h][w] float32 frames; host_out: [n][h3][w3].  Upload / forward / download
        of consecutive frame groups overlap."""
        assert host_in.dtype == np.float32 and host_out.dtype == np.float32
        assert host_in.flags.c_contiguous and host_out.flags.c_contiguous
        _check(self.ctx.L.srcnn_infer_frames_host(self.ctx.h, C.byref(self.c), _np_ptr(host_in), w,
                                                  h, int(host_in.shape[0]), _np_ptr(host_out)))

    def train_workspace_bytes(self, w, h, S):
        return self.ctx.L.srcnn_train_workspace_bytes(C.byref(self.c), w, h, S)

    def train_materializes_d1(self):
        """False when the chunk entries keep the layer-1 deltas inside the gradient kernel."""
        return bool(self.ctx.L.srcnn_train_materializes_d1(self.ctx.h, C.byref(self.c)))

    def train_chunk(self, inp, gt, w, h, S, work):
        _check(self.ctx.L.srcnn_train_chunk(self.ctx.h, C.byref(self.c), inp, gt, w, h, S, work))

    def train_chunks_host(self, host_in, host_gt, w, h, chunk, work):
        """Forward + backward over HOST sample arrays [n][h][w] (pinned for overlap), uploads
        pipelined with the training of the previous chunk; gradients accumulate."""
        assert host_in.dtype == np.float32 and host_gt.dtype == np.float32
        assert host_in.shape == host_gt.shape and host_in.flags.c_contiguous
        _check(self.ctx.L.srcnn_train_chunks_host(self.ctx.h, C.byref(self.c), _np_ptr(host_in),
                                                  _np_ptr(host_gt), w, h, int(host_in.shape[0]),
                                                  chunk, work))

    def update_all(self, batch_size, momentum, decay, lr3):
        lr = (C.c_float * 3)(*[float(v) for v in lr3])
        _check(self.ctx.L.srcnn_update_all(self.ctx.h, C.byref(self.c), batch_size, momentum,
                                           decay, lr))

    def validate_chunk(self, inp, gt, w, h, S, work, target):
        _check(self.ctx.L.srcnn_validate_chunk(self.ctx.h, C.byref(self.c), inp, gt, w, h, S,
                                               work, target))

    def allreduce_grads(self):
        """Sum the six gradient accumulators over the ranks of the context's communicator."""
        _check(self.ctx.L.srcnn_allreduce_grads(self.ctx.h, C.byref(self.c)))

    def params(self):
        out = {}
        for l, (ws, bs) in enumerate(self.sizes):
            out["w%d" % (l + 1)] = self.ctx.read(self.c.w[l], (ws,))
            out["b%d" % (l + 1)] = self.ctx.read(self.c.b[l], (bs,))
        return out

    def grads(self):
        flat = self.ctx.read(self.grad_flat, (self.grad_count,))
        out, off = {}, 0
        for l, (ws, bs) in enumerate(self.sizes):
            out["w%d" % (l + 1)] = flat[off:off + ws]
            off += ws
            out["b%d" % (l + 1)] = flat[off:off + bs]
            off += bs
        return out


# ----------------------------------------------------------------------------- sharding
def row_bands(out_h, world_size):
    """Row-band partition of the OUTPUT rows of one image across ranks (SURVEY 8e): rank g gets
    [g*ceil(out_h/N), ...).  Each band needs `halo` = f1+f2+f3-3 extra INPUT rows, no exchange."""
    per = -(-out_h // world_size)
    bands = []
    for g in range(world_size):
        r0 = min(g * per, out_h)
        r1 = min(r0 + per, out_h)
        bands.append((r0, r1))
    return bands


def patch_shards(n_patches, world_size):
    """Contiguous even split of the training patches across ranks (data parallel)."""
    base, rem = divmod(n_patches, world_size)
    out, start = [], 0
    for g in range(world_size):
        cnt = base + (1 if g < rem else 0)
        out.append((start, start + cnt))
        start += cnt
    return out

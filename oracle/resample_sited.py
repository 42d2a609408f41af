"""numpy restatement of Pillow's 8-bit resampling of a box with a fractional start
(libImaging/Resample.c precompute_coeffs with `in0`), and of 4:2:0 chroma siting on top of it:
the definition the chroma tables of csrc/resample.cuh reproduce byte for byte.

Per axis: output i takes the taps around center = in0 + (i + 0.5) * scale, then the taps, weights,
normalisation and 22-bit rounding of oracle/resample.py.  With in0 = 0.0 and scale = n_in / n_out
that is oracle/resample.py's enlargement, bit for bit.

Chroma siting: a chroma sample sits at s inside its 2x2 luma cell, per axis in chroma samples
(0.5 centred, 0.25 co-sited with the even luma column or row).  An axis from n_in samples sited at
s_in to n_out sited at s_out starts its box at
    in0 = (s_out - 0.5) * scale + (0.5 - s_in),    scale = n_in / n_out,
computed in double in that order.  Pillow's Python API cannot state this itself: for left siting
the box starts outside the image, which Image.resize refuses.
"""
import numpy as np

from oracle.resample import FILT, PB

# name -> (s_x, s_y); the names are ffmpeg's chroma_location ones
SITINGS = {"center": (0.5, 0.5), "left": (0.25, 0.5), "topleft": (0.25, 0.25)}


def coeffs(n_in, n_out, name, in0=0.0, scale=None):   # upscaling: filterscale = 1
    f, support = FILT[name]
    scale = n_in / n_out if scale is None else scale
    bounds, kk = [], []
    for i in range(n_out):
        center = in0 + (i + 0.5) * scale
        xmin = max(int(center - support + 0.5), 0)
        n = min(int(center + support + 0.5), n_in) - xmin
        k = [f(j + xmin - center + 0.5) for j in range(n)]
        ww = sum(k)
        k = [v / ww if ww != 0.0 else v for v in k]
        kk.append([int(-0.5 + v * (1 << PB)) if v < 0 else int(0.5 + v * (1 << PB)) for v in k])
        bounds.append(xmin)
    return bounds, kk


def pass_(img, n_out, name, axis, in0=0.0, scale=None):   # img uint8, axis 1 = horizontal
    src = np.moveaxis(img, axis, 0).astype(np.int64)
    bounds, kk = coeffs(src.shape[0], n_out, name, in0, scale)
    out = np.empty((n_out,) + src.shape[1:], np.uint8)
    for i in range(n_out):
        acc = np.full(src.shape[1:], 1 << (PB - 1), np.int64)
        for j, c in enumerate(kk[i]):
            acc += src[bounds[i] + j] * c
        out[i] = np.clip(acc >> PB, 0, 255)
    return np.moveaxis(out, 0, axis)


def resize_box(img, W, H, name, x0=0.0, y0=0.0, sx=None, sy=None):
    """Pillow's resize((W, H), box=(x0, y0, x0 + sx * W, y0 + sy * H)): horizontal first, 8-bit
    intermediate; an axis is not resampled when its size does not change and its start is 0.0"""
    h, w = img.shape[:2]
    t = img if (W == w and x0 == 0.0) else pass_(img, W, name, 1, x0, sx)
    return t if (H == h and y0 == 0.0) else pass_(t, H, name, 0, y0, sy)


def chroma_in0(n_in, n_out, s_in, s_out):
    scale = n_in / n_out
    return (s_out - 0.5) * scale + (0.5 - s_in)


def resize_sited(plane, W, H, name, siting_in, siting_out):
    """a chroma plane [h][w] sited at `siting_in` enlarged to [H][W] sited at `siting_out`"""
    h, w = plane.shape
    (sx_in, sy_in), (sx_out, sy_out) = SITINGS[siting_in], SITINGS[siting_out]
    return resize_box(plane, W, H, name, chroma_in0(w, W, sx_in, sx_out),
                      chroma_in0(h, H, sy_in, sy_out))

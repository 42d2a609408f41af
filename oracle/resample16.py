"""numpy restatement of Pillow's 16-bit resampling (its "I;16" mode: libImaging/Resample.c
ImagingResampleHorizontal_16bpc / ImagingResampleVertical_16bpc) of a box with a fractional start,
and of the 10-bit 4:2:0 planes on top of it: the definition the 10-bit instantiations of
csrc/resample.cuh reproduce word for word.

Per axis the taps and the normalised weights are those of oracle/resample_sited.py, kept as doubles
(Pillow's 16-bit path does not round them to 22 bits).  Each output is
    ss = 0.0;  ss += v[j] * k[j]   (in tap order, in double, no fused multiply-add)
rounded half away from zero (Pillow's ROUND_UP) and clipped to [0, 65535].  The horizontal pass
runs first into that 16-bit intermediate; an axis is not resampled when its size does not change and
its box starts at 0.0.  A 10-bit plane (values in [0, 1023]) is resampled on its values and the
result capped at 1023; the cap is not applied to the intermediate.
"""
import numpy as np

from oracle.resample import FILT
from oracle.resample_sited import SITINGS, chroma_in0


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
        kk.append([v / ww if ww != 0.0 else v for v in k])
        bounds.append(xmin)
    return bounds, kk


def round_up(ss):
    """Pillow's ROUND_UP: (int)(x + 0.5) for x >= 0, (int)(x - 0.5) below, in double"""
    return np.where(ss >= 0.0, np.trunc(ss + 0.5), np.trunc(ss - 0.5)).astype(np.int64)


def pass_(img, n_out, name, axis, in0=0.0, scale=None):   # axis 1 = horizontal
    src = np.moveaxis(img, axis, 0).astype(np.float64)
    bounds, kk = coeffs(src.shape[0], n_out, name, in0, scale)
    out = np.empty((n_out,) + src.shape[1:], np.uint16)
    for i in range(n_out):
        ss = np.zeros(src.shape[1:], np.float64)
        for j, c in enumerate(kk[i]):
            ss = ss + src[bounds[i] + j] * c
        out[i] = np.clip(round_up(ss), 0, 65535)
    return np.moveaxis(out, 0, axis)


def resize_box(img, W, H, name, x0=0.0, y0=0.0, sx=None, sy=None):
    """Pillow's Image.fromarray(img, "I;16").resize((W, H), box=(x0, y0, x0 + sx * W, y0 + sy * H))
    on a uint16 [h][w] plane; an axis is copied when the box spans it exactly"""
    h, w = img.shape
    copy_x = W == w and x0 == 0.0 and sx in (None, 1.0)
    copy_y = H == h and y0 == 0.0 and sy in (None, 1.0)
    t = img.astype(np.uint16) if copy_x else pass_(img, W, name, 1, x0, sx)
    return t if copy_y else pass_(t, H, name, 0, y0, sy)


def resize10(plane, W, H, name):
    """a 10-bit plane [h][w] (values in [0, 1023]) enlarged to [H][W], capped at 1023"""
    return np.minimum(resize_box(plane, W, H, name), 1023).astype(np.uint16)


def resize10_sited(plane, W, H, name, siting_in, siting_out):
    """a 10-bit chroma plane [h][w] sited at `siting_in` enlarged to [H][W] sited at `siting_out`"""
    h, w = plane.shape
    (sx_in, sy_in), (sx_out, sy_out) = SITINGS[siting_in], SITINGS[siting_out]
    t = resize_box(plane, W, H, name, chroma_in0(w, W, sx_in, sx_out),
                   chroma_in0(h, H, sy_in, sy_out))
    return np.minimum(t, 1023).astype(np.uint16)

"""numpy restatement of Pillow's 8-bit RGB resampling (libImaging/Resample.c) for UPSCALING,
the definition the CUDA kernel of csrc/resample.cuh reproduces byte for byte.

Per axis: scale = in/out, filterscale = 1; the taps of output i are the input samples
[xmin, xmin + n) around center = (i + 0.5) * scale, weighted by the filter in double and
normalised by their sum, then rounded to int32 with 22 fraction bits.  The horizontal pass runs
first into an 8-bit intermediate; an axis whose size does not change is not resampled.
"""
import math

import numpy as np

PB = 22                                        # Pillow's PRECISION_BITS for 8-bit images


def bicubic(x, a=-0.5):
    x = abs(x)
    if x < 1.0:
        return ((a + 2.0) * x - (a + 3.0)) * x * x + 1
    if x < 2.0:
        return (((x - 5) * x + 8) * x - 4) * a
    return 0.0


def sinc(x):
    return 1.0 if x == 0.0 else math.sin(x * math.pi) / (x * math.pi)


def lanczos(x):
    return sinc(x) * sinc(x / 3) if -3.0 <= x < 3.0 else 0.0


FILT = {"bicubic": (bicubic, 2.0), "lanczos": (lanczos, 3.0)}


def coeffs(n_in, n_out, name):                 # upscaling: filterscale = 1
    f, support = FILT[name]
    scale, bounds, kk = n_in / n_out, [], []
    for i in range(n_out):
        center = (i + 0.5) * scale
        xmin = max(int(center - support + 0.5), 0)
        n = min(int(center + support + 0.5), n_in) - xmin
        k = [f(j + xmin - center + 0.5) for j in range(n)]
        ww = sum(k)
        k = [v / ww if ww != 0.0 else v for v in k]
        kk.append([int(-0.5 + v * (1 << PB)) if v < 0 else int(0.5 + v * (1 << PB)) for v in k])
        bounds.append(xmin)
    return bounds, kk


def pass_(img, n_out, name, axis):             # img uint8 [h][w][3]; axis 1 = horizontal
    src = np.moveaxis(img, axis, 0).astype(np.int64)
    bounds, kk = coeffs(src.shape[0], n_out, name)
    out = np.empty((n_out,) + src.shape[1:], np.uint8)
    for i in range(n_out):
        acc = np.full(src.shape[1:], 1 << (PB - 1), np.int64)
        for j, c in enumerate(kk[i]):
            acc += src[bounds[i] + j] * c
        out[i] = np.clip(acc >> PB, 0, 255)
    return np.moveaxis(out, 0, axis)


def resize(img, W, H, name):                   # horizontal first, 8-bit intermediate
    t = pass_(img, W, name, 1) if W != img.shape[1] else img
    return pass_(t, H, name, 0) if H != img.shape[0] else t

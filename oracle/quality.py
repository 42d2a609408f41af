"""float64 restatement of the enlargement-quality metrics srcnn_image_quality computes
(csrc/quality.cuh), written from their definitions:

  luma   generic::luma_of(p, normalize = 1): ((R*.299 + G*.587) + B*.114) / 255, every operation
         rounded to float32 in that order (numpy's float32 ufuncs round each operation and never
         fuse a multiply and an add);
  region [border, w - border) x [border, h - border);
  mse    the mean over the region of d^2, d = Y_result - Y_ref taken in float32, d^2 and the mean
         in float64; PSNR = 10 log10(1 / mse), +inf for mse = 0;
  ssim   Wang et al. 2004 (`ssim_index`): an 11x11 Gaussian window of sigma 1.5 normalised to sum
         1, "valid" windows only (wholly inside the region), C1 = 0.01^2, C2 = 0.03^2, population
         statistics (sigma_x^2 = E[x^2] - mu_x^2 ...), the mean of the SSIM map.
"""
import math

import numpy as np
from scipy.signal import correlate2d

C1, C2 = 0.01 ** 2, 0.03 ** 2
WIN = 11


def luma(img):
    """uint8 [..., h, w, >= 3] (RGB8 or RGBA8; alpha ignored) -> float32 normalized luma"""
    p = img[..., :3].astype(np.float32)
    y = p[..., 0] * np.float32(0.299) + p[..., 1] * np.float32(0.587)
    y = y + p[..., 2] * np.float32(0.114)
    return y / np.float32(255.0)


def window():
    """the 11x11 Gaussian window, sigma 1.5, sum 1 (fspecial('gaussian', 11, 1.5))"""
    x = np.arange(WIN, dtype=np.float64) - WIN // 2
    g = np.exp(-(x[:, None] ** 2 + x[None, :] ** 2) / (2.0 * 1.5 ** 2))
    return g / g.sum()


def region(y, border):
    h, w = y.shape
    return y[border:h - border, border:w - border]


def mse_of(x, y):
    """x, y: float32 luma of the region"""
    d = (np.asarray(x, np.float32) - np.asarray(y, np.float32)).astype(np.float64)
    return float(np.mean(d * d))


def ssim_map(x, y):
    """the SSIM of every valid 11x11 window of two luma regions (float64)"""
    x, y = np.asarray(x, np.float64), np.asarray(y, np.float64)
    win = window()

    def f(a):
        return correlate2d(a, win, mode="valid")

    mx, my = f(x), f(y)
    vx, vy, cxy = f(x * x) - mx * mx, f(y * y) - my * my, f(x * y) - mx * my
    return ((2 * mx * my + C1) * (2 * cxy + C2)) / ((mx * mx + my * my + C1) * (vx + vy + C2))


def quality(result, reference, border):
    """(mse, ssim) of one uint8 result image (RGB8 / RGBA8) against its RGBA8 reference"""
    x, y = region(luma(result), border), region(luma(reference), border)
    return mse_of(x, y), float(ssim_map(x, y).mean())


def psnr(mse):
    return math.inf if mse == 0 else 10.0 * math.log10(1.0 / mse)

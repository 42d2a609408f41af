"""Writes tests/golden/pil_resample.npz: Pillow's BICUBIC and LANCZOS enlargements of small RGB
images, the ground truth of oracle/resample.py and of the CUDA resampling kernel.

    python tests/golden/make_resample_golden.py     (needs Pillow)

Each case `<name>` stores `<name>_in` (uint8 [h][w][3]) and `<name>_<filter>` (uint8 [H][W][3]).
"""
import os

import numpy as np
from PIL import Image

HERE = os.path.dirname(os.path.abspath(__file__))
FILTERS = {"bicubic": Image.BICUBIC, "lanczos": Image.LANCZOS}


def cases():
    rng = np.random.default_rng(20261020)
    yy, xx = np.mgrid[0:12, 0:12]
    checker = np.repeat((((yy + xx) & 1) * 255).astype(np.uint8)[..., None], 3, axis=2)
    yield "random_x2", rng.integers(0, 256, (9, 11, 3), dtype=np.uint8), 22, 18
    yield "random_x3", rng.integers(0, 256, (7, 6, 3), dtype=np.uint8), 18, 21
    yield "random_x4", rng.integers(0, 256, (5, 8, 3), dtype=np.uint8), 32, 20
    yield "checker_x2", checker, 24, 24
    yield "checker_x3", checker[:7, :9], 27, 21
    yield "zeros_x2", np.zeros((6, 5, 3), np.uint8), 10, 12
    yield "full_x3", np.full((4, 6, 3), 255, np.uint8), 18, 12
    yield "random_5to13", rng.integers(0, 256, (5, 5, 3), dtype=np.uint8), 13, 13
    yield "row_1to4", rng.integers(0, 256, (1, 6, 3), dtype=np.uint8), 24, 4
    yield "height_only", rng.integers(0, 256, (6, 9, 3), dtype=np.uint8), 9, 17


def main():
    out = {}
    for name, img, W, H in cases():
        out[name + "_in"] = img
        for fname, f in FILTERS.items():
            out["%s_%s" % (name, fname)] = np.asarray(Image.fromarray(img, "RGB").resize((W, H), f))
    np.savez_compressed(os.path.join(HERE, "pil_resample.npz"), **out)


if __name__ == "__main__":
    main()

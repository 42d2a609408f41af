"""Writes tests/golden/pil_box_resample.npz: Pillow's BICUBIC and LANCZOS enlargements of small
"L" images from boxes with fractional starts, the ground truth of oracle/resample_sited.py (the
chroma-siting tables of the CUDA resampler are that restatement's).

    python tests/golden/make_box_resample_golden.py     (needs Pillow)

Each case `<name>` stores `<name>_in` (uint8 [h][w]), `<name>_box` (float64 [x0, y0, x1, y1]),
`<name>_size` (int64 [W, H]) and `<name>_<filter>` (uint8 [H][W]): Image.fromarray(in, "L")
.resize((W, H), filter, box=box).  Pillow refuses a box that extends past the image, so each box
ends inside it.  Pillow holds the box, and an axis's extent, in single precision and divides in
double: x0 = float32(box[0]), scale = (double)(float32(box[2]) - x0) / W.
"""
import os

import numpy as np
from PIL import Image

HERE = os.path.dirname(os.path.abspath(__file__))
FILTERS = {"bicubic": Image.BICUBIC, "lanczos": Image.LANCZOS}
STARTS = (0.0625, 0.125, 0.3, 1.7)
# (name, n_in, n_out) of an axis: x2, x3, a ratio that is not whole, and a size that does not change
AXES = (("x2", 10, 20), ("x3", 7, 21), ("9to13", 9, 13), ("12to12", 12, 12))


def box_axis(n, start):
    """a box on an axis of n samples starting at `start` and ending inside the image"""
    return start, (n - 0.5 if start < n - 1 else float(n))


def cases():
    rng = np.random.default_rng(20261022)
    for ax, n, N in AXES:
        for k, s in enumerate(STARTS):
            tag = "%s_%d" % (ax, k)
            # the horizontal axis alone (the vertical neither resized nor offset)
            img = rng.integers(0, 256, (5, n), dtype=np.uint8)
            x0, x1 = box_axis(n, s)
            yield "h_" + tag, img, (x0, 0.0, x1, 5.0), (N, 5)
            # the vertical axis alone
            img = rng.integers(0, 256, (n, 6), dtype=np.uint8)
            y0, y1 = box_axis(n, s)
            yield "v_" + tag, img, (0.0, y0, 6.0, y1), (6, N)
            # both axes, the vertical with the next start
            img = rng.integers(0, 256, (n, n), dtype=np.uint8)
            y0, y1 = box_axis(n, STARTS[(k + 1) % len(STARTS)])
            yield "hv_" + tag, img, (x0, y0, x1, y1), (N, N)


def main():
    out = {}
    for name, img, box, size in cases():
        out[name + "_in"] = img
        out[name + "_box"] = np.array(box, np.float64)
        out[name + "_size"] = np.array(size, np.int64)
        for fname, f in FILTERS.items():
            out["%s_%s" % (name, fname)] = np.asarray(Image.fromarray(img, "L").resize(size, f, box=box))
    np.savez_compressed(os.path.join(HERE, "pil_box_resample.npz"), **out)


if __name__ == "__main__":
    main()

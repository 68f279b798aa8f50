"""Generates tests/golden/cv2_golden.npz from the REAL cv2 (4.13.0): the cv2 results that tests/test_canny_oracle.py compares the
oracles with beyond canny_golden.npz and gauss_golden.npz, so those comparisons run where cv2 is not installed too.

    python tests/golden/make_cv2_golden.py

Stored: Canny cases in the layout of canny_golden.npz (seeded inputs, bit-packed edges, CRC32s of input and gray image); the CRC32 of
cv2's gray conversion of one seeded 512x512 random image; CRC32s of input and cv2.GaussianBlur(src, (5, 5), 0) for random arrays
drawn in order from one seeded generator."""
import os
import sys
import zlib

import cv2
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle.canny_oracle import synthetic_image  # noqa: E402

KINDS = ["shapes", "noise", "smooth"]
CANNY = [(11, 200, 300, "shapes"), (12, 77, 131, "noise"), (13, 128, 128, "smooth")]   # (seed, h, w, kind)
THRESHOLDS = [(100, 200), (10, 20), (300, 50)]
GRAY_SEED = 0                                                                         # rng.integers(0, 256, (512, 512, 3))
BLUR_SEED, BLUR_SHAPES = 3, [(64, 64), (37, 53, 3), (4, 6), (300, 200, 3)]

if __name__ == "__main__":
    out = {}
    i = 0
    for seed, h, w, kind in CANNY:
        img = synthetic_image(seed, h, w, kind)
        gray = cv2.cvtColor(img, cv2.COLOR_RGB2GRAY)
        for lo, hi in THRESHOLDS:
            out[f"case{i}_meta"] = np.array([seed, h, w, KINDS.index(kind), lo, hi, zlib.crc32(img.tobytes())], np.int64)
            out[f"case{i}_gray_crc"] = np.array([zlib.crc32(gray.tobytes())], np.int64)
            out[f"case{i}_edges"] = np.packbits(cv2.Canny(gray, lo, hi) > 0)
            i += 1
    img = np.random.default_rng(GRAY_SEED).integers(0, 256, size=(512, 512, 3), dtype=np.uint8)
    out["gray_sample"] = np.array([GRAY_SEED, zlib.crc32(img.tobytes()), zlib.crc32(cv2.cvtColor(img, cv2.COLOR_RGB2GRAY).tobytes())], np.int64)
    rng = np.random.default_rng(BLUR_SEED)
    out["blur_seed"] = np.array([BLUR_SEED], np.int64)
    for j, shape in enumerate(BLUR_SHAPES):
        a = rng.integers(0, 256, shape, dtype=np.uint8)
        out[f"blur{j}_shape"] = np.array(shape, np.int64)
        out[f"blur{j}_crc"] = np.array([zlib.crc32(a.tobytes()), zlib.crc32(cv2.GaussianBlur(a, (5, 5), 0).tobytes())], np.int64)
    np.savez_compressed(os.path.join(os.path.dirname(os.path.abspath(__file__)), "cv2_golden.npz"), **out)

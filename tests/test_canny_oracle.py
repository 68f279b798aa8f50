"""CPU: the Canny oracle (numpy + plain C) against the committed cv2 golden vectors, and those against live cv2 where it is installed."""
import os
import zlib

import numpy as np

from oracle import c_oracle
from oracle.canny_oracle import canny_gray, preprocess_image, rgb_to_gray
from tests.util import GOLDEN, canny_golden_cases


def _cv2():
    try:
        import cv2
    except ImportError:
        return None
    return cv2


def _cv2_golden():
    return np.load(os.path.join(GOLDEN, "cv2_golden.npz"))


def test_numpy_oracle_matches_golden():
    n = 0
    for img, lo, hi, edges, gray_crc in canny_golden_cases():
        gray = rgb_to_gray(img)
        assert zlib.crc32(gray.tobytes()) == gray_crc
        assert np.array_equal(canny_gray(gray, lo, hi), edges)
        if img.shape[0] * img.shape[1] <= 256 * 256:   # the pure-Python flood fill only on small cases
            assert np.array_equal(canny_gray(gray, lo, hi, fast=False), edges)
        n += 1
    assert n >= 10


def test_c_oracle_matches_golden():
    for img, lo, hi, edges, _ in canny_golden_cases():
        out = c_oracle.canny_u8(img[None], lo, hi)
        assert np.array_equal(out[0], edges)
        out3 = c_oracle.canny_u8(img[None], lo, hi, replicate3=True)
        assert np.array_equal(out3[0], np.stack([edges] * 3, axis=2))


def test_oracle_matches_live_cv2():
    """Three more images at three threshold pairs (incl. low > high) against cv2's edges stored in cv2_golden.npz, and the stored
    edges against live cv2."""
    cv2 = _cv2()
    n = 0
    for img, lo, hi, ref, gray_crc in canny_golden_cases("cv2_golden.npz"):
        gray = rgb_to_gray(img)
        assert zlib.crc32(gray.tobytes()) == gray_crc
        if cv2 is not None:
            assert np.array_equal(cv2.cvtColor(img, cv2.COLOR_RGB2GRAY), gray)
            assert np.array_equal(cv2.Canny(gray, lo, hi), ref)
        assert np.array_equal(canny_gray(gray, lo, hi), ref)
        assert np.array_equal(c_oracle.canny_u8(gray[None], lo, hi)[0], ref)
        if (lo, hi) == (100, 200):
            assert np.array_equal(preprocess_image(img)[..., 1], ref)
        n += 1
    assert n == 9


def test_gray_formula_exhaustive_sample():
    seed, img_crc, gray_crc = [int(v) for v in _cv2_golden()["gray_sample"]]
    rng = np.random.default_rng(seed)
    img = rng.integers(0, 256, size=(512, 512, 3), dtype=np.uint8)
    assert zlib.crc32(img.tobytes()) == img_crc, "numpy's generator drifted from the committed fixture"
    assert zlib.crc32(rgb_to_gray(img).tobytes()) == gray_crc
    cv2 = _cv2()
    if cv2 is not None:
        assert np.array_equal(cv2.cvtColor(img, cv2.COLOR_RGB2GRAY), rgb_to_gray(img))


def test_empty_and_flat_inputs():
    flat = np.full((1, 40, 50, 3), 77, np.uint8)
    assert c_oracle.canny_u8(flat).sum() == 0
    assert c_oracle.canny_u8(np.zeros((0, 8, 8, 3), np.uint8)).shape == (0, 8, 8)


def test_gaussian_oracle_matches_golden_and_live_cv2():
    """The optional Gaussian pre-stage: plain-C restatement of cv2.GaussianBlur(img, (5, 5), 0) against the committed cv2 CRCs
    (incl. 1-, 2- and 3-pixel-wide images where BORDER_REFLECT_101 wraps more than once), on random arrays against the CRCs of
    cv2_golden.npz, and against cv2 itself where it is installed."""
    from tests.util import gauss_golden_cases
    n = 0
    for src, blur_crc, edges_crc in gauss_golden_cases():
        blur = c_oracle.gaussian_blur5_u8(src[None])[0]
        assert zlib.crc32(blur.tobytes()) == blur_crc, src.shape
        if edges_crc is not None:
            assert zlib.crc32(c_oracle.canny_u8(blur[None], 100, 200)[0].tobytes()) == edges_crc
        n += 1
    assert n >= 10
    cv2 = _cv2()
    z = _cv2_golden()
    rng = np.random.default_rng(int(z["blur_seed"][0]))
    n = 0
    while f"blur{n}_shape" in z:
        shape = tuple(int(s) for s in z[f"blur{n}_shape"])
        img_crc, blur_crc = [int(v) for v in z[f"blur{n}_crc"]]
        a = rng.integers(0, 256, shape, dtype=np.uint8)
        assert zlib.crc32(a.tobytes()) == img_crc, "numpy's generator drifted from the committed fixture"
        blur = c_oracle.gaussian_blur5_u8(a[None])[0]
        assert zlib.crc32(blur.tobytes()) == blur_crc, shape
        if cv2 is not None:
            assert np.array_equal(blur, cv2.GaussianBlur(a, (5, 5), 0))
        n += 1
    assert n == 4

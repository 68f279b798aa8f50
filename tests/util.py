"""Shared helpers for the test-suite."""
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
KINDS = ["shapes", "noise", "smooth"]


def canny_golden_cases(name="canny_golden.npz"):
    """Yields (img_u8 [h,w,3], low, high, edges_u8 [h,w], crc32 of the gray image) from a committed cv2 fixture."""
    import zlib
    from oracle.canny_oracle import synthetic_image
    z = np.load(os.path.join(GOLDEN, name))
    i = 0
    while f"case{i}_meta" in z:
        seed, h, w, kind, lo, hi, crc = [int(v) for v in z[f"case{i}_meta"]]
        img = synthetic_image(seed, h, w, KINDS[kind])
        assert zlib.crc32(img.tobytes()) == crc, "synthetic_image() drifted from the committed fixture"
        edges = np.unpackbits(z[f"case{i}_edges"])[: h * w].reshape(h, w).astype(np.uint8) * 255
        yield img, lo, hi, edges, int(z[f"case{i}_gray_crc"][0])
        i += 1


def rel_err(a, b):
    """max |a-b| / max |b| on torch tensors."""
    a = a.float()
    b = b.float()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-12))


def gauss_golden_cases():
    """Yields (src_u8 [h,w] or [h,w,3], crc32 of cv2.GaussianBlur(src, (5,5), 0), crc32 of the blurred Canny or None)."""
    import zlib
    from oracle.canny_oracle import rgb_to_gray, synthetic_image
    z = np.load(os.path.join(GOLDEN, "gauss_golden.npz"))
    i = 0
    while f"case{i}_meta" in z:
        seed, h, w, kind, gray, crc, blur_crc = [int(v) for v in z[f"case{i}_meta"]]
        img = synthetic_image(seed, h, w, KINDS[kind])
        assert zlib.crc32(img.tobytes()) == crc, "synthetic_image() drifted from the committed fixture"
        src = rgb_to_gray(img) if gray else img
        edges_crc = int(z[f"case{i}_edges_crc"][0]) if f"case{i}_edges_crc" in z else None
        yield src, blur_crc, edges_crc
        i += 1


def guarded(rows, cols, ld, dev, lead=64, tail=64, dtype=None):
    """A [rows, cols] view (fp16 unless dtype is given) with row stride ld, starting lead elements into a sentinel-filled buffer;
    returns (view, checker): checker() is True while the lead and tail bands and the row padding still hold the sentinel."""
    import torch
    dtype = dtype or torch.float16
    s = float(torch.tensor(1234.0, dtype=dtype))          # the sentinel as the type holds it (bf16: 1232)
    buf = torch.full((lead + rows * ld + tail,), s, dtype=dtype, device=dev)
    view = buf[lead:lead + rows * ld].view(rows, ld)[:, :cols]

    def untouched():
        pad = buf[lead:lead + rows * ld].view(rows, ld)[:, cols:]
        return bool((buf[:lead] == s).all()) and bool((buf[lead + rows * ld:] == s).all()) and bool((pad == s).all())
    return view, untouched

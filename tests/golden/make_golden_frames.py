"""Generates tests/golden/frames_cases.npz: the reference's own test-time input transform -- BaseTransform
(data/augmentations.py:601-615, imported unmodified from the reference tree, with cv2) followed by the dataset's BGR -> RGB
swap and permute (data/ava.py:330-338) -- on the seeded frames of oracle.frames.source_frames for every case of
oracle.frames.GOLDEN_CASES.  Only outputs are stored (rows 0, 8, 16, ... and the last row of each output frame).
Only runnable where the reference tree is present; the file it writes is committed.

    python tests/golden/make_golden_frames.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import frames as ofr  # noqa: E402
from oracle import refload  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def gen_frames():
    assert refload.available(), "reference tree not present"
    if refload.REF not in sys.path:
        sys.path.insert(0, refload.REF)
    import cv2
    from data.augmentations import BaseTransform
    out = {"cv2_version": np.asarray([int(v) for v in cv2.__version__.split(".")[:3]])}
    for name, T, H0, W0, size, scale, mean, stds, noise, seed in ofr.GOLDEN_CASES:
        images = ofr.source_frames(T, H0, W0, seed, noise)
        res, _, _ = BaseTransform(size, mean, stds, scale)(images.copy())
        res = np.ascontiguousarray(res[:, :, :, (2, 1, 0)].transpose(0, 3, 1, 2))      # BGR -> RGB, [T, C, H, W]
        rows = np.unique(np.r_[np.arange(0, size[1], ofr.GOLDEN_ROW_STRIDE), size[1] - 1])
        out[name + "_rows"] = rows
        out[name + "_out"] = np.ascontiguousarray(res[:, :, rows, :]).astype(np.float32)
    np.savez_compressed(os.path.join(OUT, "frames_cases.npz"), **out)
    print("frames cases ok")


if __name__ == "__main__":
    gen_frames()

"""numpy restatement of the reference's test-time input transform, without cv2 and without the reference tree.

BaseTransform(size, mean, stds, scale) (data/augmentations.py:601-615) on one clip of uint8 BGR frames [T, H0, W0, 3], then
the BGR -> RGB swap and permute of data/ava.py:330-338 -> [T, 3, H, W] fp32.  Every step is fp32, in the reference's
order:
  ConvertFromInts (:75-84)  scale 0: u,  1: u / 255,  2: u * 2 / 255 - 1
  Resize (:162-169)         cv2.resize(frame, (W, H)) INTER_LINEAR on float32: cv2's coefficients
                            f = (d + 0.5) * src / dst - 0.5 in double, i = floor(f), w1 = float32(f - i), w0 = 1 - w1
                            in fp32, clamped at both borders (i, w1 = 0, 0 left; src - 1, 0 right);
                            horizontal blend first, rounded to fp32, then the vertical blend
  SubtractMeans / DivideStds (v - mean[c]) / std[c], c the BGR channel
cv2 evaluates the blends with SIMD multiply-adds, so it differs from this in the last 1-2 ulp; the goldens pin the
tolerance (tests/test_frames.py).
"""
import numpy as np


# Cases of tests/golden/frames_cases.npz (tests/golden/make_golden_frames.py runs the reference on them):
# (name, T, H0, W0, size (W, H), scale, BGR mean, BGR stds, noise, seed)
GOLDEN_CASES = [
    ("c4_i3d", 2, 360, 640, (224, 224), 2, (0, 0, 0), (1, 1, 1), 24.0, 500),           # non-integer downscale, the I3D setting
    ("c4_norm", 1, 360, 640, (224, 224), 1, (0.406, 0.456, 0.485), (0.225, 0.224, 0.229), 24.0, 501),
    ("ava_context", 1, 360, 480, (400, 400), 0, (104.0, 117.0, 123.0), (57.0, 58.0, 59.0), 24.0, 502),   # mixed up/down
    ("down2x", 1, 448, 448, (224, 224), 2, (0, 0, 0), (1, 1, 1), 24.0, 503),              # exactly 2x: still linear, not area
    ("upscale", 1, 100, 90, (224, 224), 1, (0.1, 0.2, 0.3), (0.5, 0.25, 2.0), 24.0, 504),
    ("identity", 1, 224, 224, (224, 224), 2, (0, 0, 0), (1, 1, 1), 24.0, 505),
    ("odd_source", 2, 255, 341, (224, 224), 2, (0.25, -0.5, 0.125), (1.5, 0.75, 3.0), 24.0, 506),
    ("non_square", 1, 240, 427, (400, 320), 1, (0, 0, 0), (1, 1, 1), 24.0, 507),         # BaseTransform's default size (W, H)
    ("extremes", 1, 120, 200, (96, 160), 2, (0, 0, 0), (1, 1, 1), 4000.0, 508),          # nearly all pixels 0 or 255
]
GOLDEN_ROW_STRIDE = 8   # outputs keep rows 0, 8, 16, ... and the last row (every column): the file stays under 2 MB


def source_frames(T, H0, W0, seed, noise=24.0):
    """Seeded uint8 BGR frames [T, H0, W0, 3] shared by the golden generator and the tests: smooth gradients plus Gaussian
    noise of deviation `noise` (clipped), with the extreme values 0 and 255 present in every frame."""
    rng = np.random.default_rng(seed)
    y = np.arange(H0, dtype=np.float64)[:, None, None]
    x = np.arange(W0, dtype=np.float64)[None, :, None]
    c = np.arange(3, dtype=np.float64)[None, None, :]
    out = np.empty((T, H0, W0, 3), dtype=np.uint8)
    for t in range(T):
        base = 127.5 + 127.5 * np.sin(0.05 * (x + 3 * t) + 0.07 * y + 2.1 * c)
        v = base + rng.normal(0.0, noise, size=(H0, W0, 3))
        f = np.clip(np.rint(v), 0, 255).astype(np.uint8)
        f[0, 0] = 0
        f[-1, -1] = 255
        out[t] = f
    return out


def convert_from_ints(u, scale):
    f = u.astype(np.float32)
    if scale == 0:
        return f
    if scale == 1:
        return f / np.float32(255)
    if scale == 2:
        return f * np.float32(2) / np.float32(255) - np.float32(1)
    raise ValueError("scale must be 0, 1 or 2")


def resize_taps(src, dst):
    """cv2 INTER_LINEAR coefficients of one axis: (i0, i1, w0, w1) per output position."""
    d = np.arange(dst, dtype=np.float64)
    f = (d + 0.5) * (float(src) / float(dst)) - 0.5
    i = np.floor(f).astype(np.int64)
    f = (f - i).astype(np.float32)
    lo = i < 0
    i[lo], f[lo] = 0, 0
    hi = i >= src - 1
    i[hi], f[hi] = src - 1, 0
    return i, np.minimum(i + 1, src - 1), (np.float32(1) - f).astype(np.float32), f.astype(np.float32)


def resize_linear(img, W, H):
    """cv2.resize(img, (W, H)) on float32 [H0, W0, C]."""
    H0, W0 = img.shape[:2]
    x0, x1, a0, a1 = resize_taps(W0, W)
    y0, y1, b0, b1 = resize_taps(H0, H)
    hz = img[:, x0] * a0[None, :, None] + img[:, x1] * a1[None, :, None]   # [H0, W, C] fp32
    return (hz[y0] * b0[:, None, None] + hz[y1] * b1[:, None, None]).astype(np.float32)


def base_transform(images, size, mean=(0, 0, 0), stds=(1, 1, 1), scale=1):
    """images uint8 [T, H0, W0, 3] BGR; size (W, H) -> fp32 [T, 3, H, W] RGB."""
    W, H = size
    f = convert_from_ints(np.asarray(images), scale)
    out = np.stack([resize_linear(f[t], W, H) for t in range(f.shape[0])])
    out = (out - np.asarray(mean, dtype=np.float32)) / np.asarray(stds, dtype=np.float32)
    return np.ascontiguousarray(out[..., ::-1].transpose(0, 3, 1, 2)).astype(np.float32)

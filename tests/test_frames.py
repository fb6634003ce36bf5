"""CPU: the input transform from decoded frames (csrc/frames.cu, step_b200/frames.py).  The numpy oracle against the
reference's own BaseTransform (tests/golden/frames_cases.npz), argument checks of the C entries without a GPU, and the
host side of the Python layer."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import frames as ofr

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "frames_cases.npz")
STEP_E_ARG = 10001


def tolerance(ref, scale, stds):
    """cv2 blends with multiply-adds, so the resized value (range 255 at scale 0, else 1) may differ in its last 1-2 ulp;
    SubtractMeans / DivideStds carry that difference over scaled by 1 / std."""
    rng = 255.0 if scale == 0 else 1.0
    return 3e-7 * max(1.0, float(np.abs(ref).max()), rng / min(abs(s) for s in stds))


@pytest.mark.parametrize("case", ofr.GOLDEN_CASES, ids=[c[0] for c in ofr.GOLDEN_CASES])
def test_oracle_matches_reference_base_transform(case):
    name, T, H0, W0, size, scale, mean, stds, noise, seed = case
    g = np.load(GOLDEN)
    ref = g[name + "_out"]
    out = ofr.base_transform(ofr.source_frames(T, H0, W0, seed, noise), size, mean, stds, scale)
    assert out.shape == (T, 3, size[1], size[0]) and out.dtype == np.float32
    got = out[:, :, g[name + "_rows"]]
    assert np.abs(got - ref).max() <= tolerance(ref, scale, stds), name


def test_golden_cases_cover_the_contract():
    names = {c[0]: c for c in ofr.GOLDEN_CASES}
    assert {c[5] for c in ofr.GOLDEN_CASES} == {0, 1, 2}
    assert any(len(set(c[6])) == 3 and 0 not in c[6] and len(set(c[7])) == 3 for c in ofr.GOLDEN_CASES)
    assert any(c[4][0] != c[4][1] for c in ofr.GOLDEN_CASES)           # non-square (width, height)
    assert any(c[2] % 2 == 1 or c[3] % 2 == 1 for c in ofr.GOLDEN_CASES)
    assert names["identity"][2:4] == names["identity"][4][::-1]
    f = ofr.source_frames(1, 20, 30, 0)
    assert f.min() == 0 and f.max() == 255


def test_resize_identity_and_borders():
    img = ofr.source_frames(1, 17, 23, 3)[0].astype(np.float32)
    assert np.array_equal(ofr.resize_linear(img, 23, 17), img)      # same size copies through
    i0, i1, w0, w1 = ofr.resize_taps(10, 40)                        # upscale: both borders clamp to one sample
    assert i0[0] == 0 and w1[0] == 0 and i0[-1] == 9 and i1[-1] == 9 and w1[-1] == 0


def _lib():
    from step_b200 import _lib as L
    lib = L.lib()
    lib.step_last_error.restype = ctypes.c_char_p
    return lib


GOOD = dict(N=2, T=4, Hmax=360, Wmax=640, H=224, W=224, scale=2, mean=(0.0, 0.0, 0.0), stds=(1.0, 1.0, 1.0))


@pytest.mark.parametrize("entry", ["step_frames_to_clip_f32", "step_frames_to_s2d_f16"])
@pytest.mark.parametrize("bad,needle", [
    (dict(scale=3), b"scale must be 0, 1 or 2"),
    (dict(scale=-1), b"scale must be 0, 1 or 2"),
    (dict(stds=(1.0, 0.0, 1.0)), b"std non-zero"),
    (dict(mean=(0.0, float("nan"), 0.0)), b"must be finite"),
    (dict(null="frames"), b"null pointer"),
    (dict(null="sizes"), b"null pointer"),
    (dict(null="out"), b"null pointer"),
    (dict(Hmax=50000, Wmax=50000), b"exceeds 2^31 bytes"),
    (dict(N=0), b"bad extent"),
    (dict(W=-2), b"bad extent"),
])
def test_entries_reject_bad_arguments(entry, bad, needle):
    lib = _lib()
    buf = (ctypes.c_char * 4096)()
    p = ctypes.cast(buf, ctypes.c_void_p).value
    a = dict(GOOD, **{k: v for k, v in bad.items() if k != "null"})
    ptrs = {k: (None if bad.get("null") == k else p) for k in ("frames", "sizes", "out")}
    rc = getattr(lib, entry)(ptrs["frames"], ptrs["sizes"], a["N"], a["T"], a["Hmax"], a["Wmax"], a["H"], a["W"], a["scale"],
                             *a["mean"], *a["stds"], ptrs["out"], None)
    assert rc == STEP_E_ARG
    assert needle in lib.step_last_error()


@pytest.mark.parametrize("T,H,W", [(3, 224, 224), (4, 223, 224), (4, 224, 225)])
def test_s2d_entry_needs_even_extent(T, H, W):
    lib = _lib()
    buf = (ctypes.c_char * 4096)()
    p = ctypes.cast(buf, ctypes.c_void_p).value
    rc = lib.step_frames_to_s2d_f16(p, p, 1, T, 360, 640, H, W, 2, 0.0, 0.0, 0.0, 1.0, 1.0, 1.0, p, None)
    assert rc == STEP_E_ARG and b"must be even" in lib.step_last_error()


def test_s2d_entry_needs_32_byte_aligned_output():
    lib = _lib()
    buf = (ctypes.c_char * 4096)()
    p = ctypes.cast(buf, ctypes.c_void_p).value
    out = (p + 31) // 32 * 32 + 16
    rc = lib.step_frames_to_s2d_f16(p, p, 1, 2, 8, 8, 4, 4, 2, 0.0, 0.0, 0.0, 1.0, 1.0, 1.0, out, None)
    assert rc == STEP_E_ARG and b"32-byte aligned" in lib.step_last_error()


def test_pack_frames_places_clips_and_sizes():
    from step_b200.frames import pack_frames
    a = ofr.source_frames(3, 5, 7, 1)
    b = torch.from_numpy(ofr.source_frames(3, 9, 4, 2))
    frames, sizes = pack_frames([a, b], pin_memory=False)
    assert frames.dtype == torch.uint8 and frames.shape == (2, 3, 9, 7, 3)
    assert sizes.dtype == torch.int32 and sizes.tolist() == [[5, 7], [9, 4]]
    assert np.array_equal(frames[0, :, :5, :7].numpy(), a) and np.array_equal(frames[1, :, :9, :4].numpy(), b.numpy())
    assert not frames[0, :, 5:].any() and not frames[0, :, :, 7:].any() and not frames[1, :, :, 4:].any()
    frames, sizes = pack_frames([a], max_hw=(6, 8), pin_memory=False)
    assert frames.shape == (1, 3, 6, 8, 3) and sizes.tolist() == [[5, 7]]
    with pytest.raises(ValueError):
        pack_frames([b], max_hw=(8, 8), pin_memory=False)
    with pytest.raises(ValueError):
        pack_frames([a, ofr.source_frames(2, 5, 7, 1)], pin_memory=False)      # T differs
    with pytest.raises(ValueError):
        pack_frames([a.astype(np.float32)], pin_memory=False)


def test_check_sizes_rejects_out_of_slot_sizes():
    from step_b200.frames import check_sizes
    assert check_sizes([[360, 640], [1, 1]], 2, 360, 640).tolist() == [[360, 640], [1, 1]]
    for bad in ([[361, 640], [1, 1]], [[360, 641], [1, 1]], [[0, 640], [1, 1]], [[360, 640]], [[1.5, 2.0], [1.0, 1.0]]):
        with pytest.raises(ValueError):
            check_sizes(bad, 2, 360, 640)


def test_frames_to_clip_raises_on_cpu_tensors():
    from step_b200.frames import frames_to_clip, pack_frames
    frames, sizes = pack_frames([ofr.source_frames(2, 8, 8, 0)], pin_memory=False)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        frames_to_clip(frames, sizes, (4, 4))

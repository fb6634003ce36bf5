"""The reference's test-time input transform on the device, from decoded uint8 frames.

In the reference the data loader turns every clip into the network's input on the host: `BaseTransform`
(data/augmentations.py:601-615: ConvertFromInts -> Resize -> SubtractMeans -> DivideStds) on the BGR frames
`cv2.imread` returned, then the BGR -> RGB swap and permute of data/ava.py:330-338.  Here the host only decodes;
everything after the uint8 frame runs in CUDA (csrc/frames.cu):

    frames, sizes = pack_frames([clip0, clip1, ...])       # per-clip uint8 [T, H0, W0, 3] BGR, sizes may differ
    x = frames_to_clip(frames.cuda(), sizes, size=(W, H), mean=..., stds=..., scale=...)   # [N, T, 3, H, W] fp32
or, inside the captured step, `StepRunner(..., frames=dict(...))` (runner.py), which goes straight to the stem's
space-to-depth input.  `size` is (width, height), as in `BaseTransform`; `mean` and `stds` are in BGR order.
"""
import numpy as np
import torch

from . import _lib as L
from .engine import Act


def pack_frames(clips, max_hw=None, pin_memory=None):
    """clips: list of uint8 arrays or tensors [T, H0, W0, 3] (one T for all, H0 x W0 per clip).
    Returns (frames [N, T, Hmax, Wmax, 3] uint8, sizes [N, 2] int32 = (H0, W0)), both in page-locked host memory when
    CUDA is available (pin_memory=None), so that copies to the device are asynchronous.  Clip n fills the top-left
    H0 x W0 of each of its frame slots.  max_hw = (Hmax, Wmax) fixes the slot size (a StepRunner's `frames["max_hw"]`);
    by default it is the largest clip's."""
    ts = [torch.as_tensor(np.ascontiguousarray(c)) if not torch.is_tensor(c) else c for c in clips]
    if not ts:
        raise ValueError("pack_frames: no clips")
    for t in ts:
        if t.dtype != torch.uint8 or t.dim() != 4 or t.shape[3] != 3:
            raise ValueError("pack_frames: expected uint8 [T, H0, W0, 3] clips, got %s %s" % (t.dtype, tuple(t.shape)))
        if t.shape[0] != ts[0].shape[0]:
            raise ValueError("pack_frames: clips differ in T (%d vs %d)" % (t.shape[0], ts[0].shape[0]))
    hmax = max(t.shape[1] for t in ts)
    wmax = max(t.shape[2] for t in ts)
    if max_hw is not None:
        if max_hw[0] < hmax or max_hw[1] < wmax:
            raise ValueError("pack_frames: a clip of %dx%d does not fit max_hw %s" % (hmax, wmax, tuple(max_hw)))
        hmax, wmax = int(max_hw[0]), int(max_hw[1])
    if pin_memory is None:
        pin_memory = torch.cuda.is_available()
    frames = torch.zeros((len(ts), ts[0].shape[0], hmax, wmax, 3), dtype=torch.uint8, pin_memory=pin_memory)
    sizes = torch.empty((len(ts), 2), dtype=torch.int32, pin_memory=pin_memory)
    for n, t in enumerate(ts):
        frames[n, :, :t.shape[1], :t.shape[2]] = t.cpu()
        sizes[n, 0], sizes[n, 1] = t.shape[1], t.shape[2]
    return frames, sizes


def check_sizes(sizes, N, Hmax, Wmax):
    """Host-side validation of a size table before it reaches the device: [N, 2] integers, 1 <= H0 <= Hmax,
    1 <= W0 <= Wmax.  Returns it as a CPU int32 tensor."""
    s = torch.as_tensor(sizes)
    if s.is_cuda:
        s = s.cpu()
    if s.shape != (N, 2) or s.is_floating_point() or s.is_complex():
        raise ValueError("frames: sizes must be an integer [%d, 2] table of (H0, W0), got %s %s" % (N, s.dtype, tuple(s.shape)))
    h, w = s[:, 0], s[:, 1]
    if bool((h < 1).any() or (h > Hmax).any() or (w < 1).any() or (w > Wmax).any()):
        raise ValueError("frames: every (H0, W0) must lie in [1, %d] x [1, %d], got %s" % (Hmax, Wmax, s.tolist()))
    return s.to(torch.int32)


def _check_frames(frames):
    L.need_cuda(frames)
    if frames.dtype != torch.uint8 or frames.dim() != 5 or frames.shape[4] != 3 or not frames.is_contiguous():
        raise ValueError("frames: expected a contiguous uint8 [N, T, Hmax, Wmax, 3] tensor, got %s %s"
                         % (frames.dtype, tuple(frames.shape)))


def launch(fn, frames, sizes_dev, size, mean, stds, scale, out):
    """Enqueue step_frames_to_clip_f32 / step_frames_to_s2d_f16 on the current stream.  sizes_dev: device int32 [N, 2],
    already validated (check_sizes)."""
    N, T, Hmax, Wmax, _ = frames.shape
    W, H = size
    L.check(fn(L.ptr(frames), L.ptr(sizes_dev), N, T, Hmax, Wmax, H, W, int(scale), *[float(v) for v in mean],
               *[float(v) for v in stds], L.ptr(out), L.stream()))
    return out


def frames_to_clip(frames, sizes, size, mean=(0, 0, 0), stds=(1, 1, 1), scale=1):
    """frames: CUDA uint8 [N, T, Hmax, Wmax, 3] BGR (pack_frames); sizes: [N, 2] (H0, W0); size: (W, H).
    Returns the CUDA fp32 clip [N, T, 3, H, W] in RGB that `BaseTransform(size, mean, stds, scale)` followed by the
    dataset's BGR -> RGB swap and permute gives for each clip."""
    _check_frames(frames)
    N, T, Hmax, Wmax, _ = frames.shape
    s = check_sizes(sizes, N, Hmax, Wmax).to(frames.device)
    W, H = size
    out = torch.empty((N, T, 3, H, W), dtype=torch.float32, device=frames.device)
    with torch.cuda.device(frames.device):
        return launch(L.lib().step_frames_to_clip_f32, frames, s, size, mean, stds, scale, out)


def frames_to_s2d(frames, sizes_dev, size, mean=(0, 0, 0), stds=(1, 1, 1), scale=1):
    """The same transform written as the fp16 stem's space-to-depth input: an Act [N, T/2, H/2, W/2, 32] equal bit for bit
    to step_clip_to_s2d_f16 of frames_to_clip's result.  sizes_dev: device int32 [N, 2], validated by the caller."""
    _check_frames(frames)
    N, T, _, _, _ = frames.shape
    W, H = size
    out = Act.empty(N, T // 2, H // 2, W // 2, 32, L.F16, frames.device)
    launch(L.lib().step_frames_to_s2d_f16, frames, sizes_dev, size, mean, stds, scale, out.buf)
    return out

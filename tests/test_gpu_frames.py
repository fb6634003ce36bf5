"""GPU: the input transform from decoded uint8 frames (csrc/frames.cu, step_b200/frames.py, StepRunner(frames=...)).

(1) frames_to_clip equals the reference's BaseTransform (goldens) and the oracle at the C4 batch with mixed source widths;
(2) the s2d form equals step_clip_to_s2d_f16 of the clip form bit for bit; (3) clips of a mixed batch are independent;
(4) a StepRunner fed frames equals one fed frames_to_clip's output bit for bit, fp16 and fp32, and replays another mix of
source sizes without a new capture."""
import os

import numpy as np
import pytest
import torch

from oracle import frames as ofr
from step_b200 import synth

pytestmark = pytest.mark.gpu

C4_WIDTHS = [480, 640, 654, 426, 360, 500, 640, 584]   # 360-pixel-high sources of different aspect ratios
DETECT = dict(conf_thresh=0.01, nms_thresh=0.4, topk=300)
NORM = dict(mean=(0.25, -0.125, 0.5), stds=(0.5, 2.0, 0.75), scale=1)


def tolerance(ref, scale, stds):
    rng = 255.0 if scale == 0 else 1.0
    return 3e-7 * max(1.0, float(np.abs(ref).max()), rng / min(abs(s) for s in stds))


def c4_clips(T=32, H0=360, widths=C4_WIDTHS, seed=0):
    return [ofr.source_frames(T, H0, w, seed + i) for i, w in enumerate(widths)]


def s2d_of_clip(x):
    from step_b200 import _lib as L
    N, T, C, H, W = x.shape
    out = torch.empty((N, T // 2, H // 2, W // 2, 32), dtype=torch.float16, device=x.device)
    L.check(L.lib().step_clip_to_s2d_f16(L.ptr(x), N, T, C, H, W, L.ptr(out), 32, L.stream()))
    return out


def to_s2d(frames, sizes, size, **norm):
    from step_b200.frames import check_sizes, frames_to_s2d
    s = check_sizes(sizes, frames.shape[0], frames.shape[2], frames.shape[3]).cuda()
    return frames_to_s2d(frames, s, size, **norm).buf


@pytest.mark.parametrize("case", ofr.GOLDEN_CASES, ids=[c[0] for c in ofr.GOLDEN_CASES])
def test_frames_to_clip_matches_reference(case):
    from step_b200.frames import frames_to_clip, pack_frames
    name, T, H0, W0, size, scale, mean, stds, noise, seed = case
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "frames_cases.npz"))
    frames, sizes = pack_frames([ofr.source_frames(T, H0, W0, seed, noise)], max_hw=(H0 + 3, W0 + 5))   # padded slot
    out = frames_to_clip(frames.cuda(), sizes, size, mean, stds, scale)
    assert out.shape == (1, T, 3, size[1], size[0])
    ref = g[name + "_out"]
    got = out[0].cpu().numpy()[:, :, g[name + "_rows"]]
    assert np.abs(got - ref).max() <= tolerance(ref, scale, stds), name


def test_frames_to_clip_matches_oracle_at_c4():
    from step_b200.frames import frames_to_clip, pack_frames
    clips = c4_clips()
    frames, sizes = pack_frames(clips)
    out = frames_to_clip(frames.cuda(), sizes, (224, 224), **NORM).cpu().numpy()
    for n, c in enumerate(clips):
        ref = ofr.base_transform(c, (224, 224), **NORM)
        assert np.abs(out[n] - ref).max() <= tolerance(ref, NORM["scale"], NORM["stds"]), n


@pytest.mark.parametrize("T,size,norm", [(32, (224, 224), dict(scale=2)), (32, (224, 224), NORM),
                                         (36, (400, 400), dict(mean=(104.0, 117.0, 123.0), stds=(57.0, 58.0, 59.0), scale=0))],
                         ids=["c4_i3d", "c4_norm", "ava_context"])
def test_s2d_bit_identical_to_clip_then_s2d(T, size, norm):
    from step_b200.frames import frames_to_clip, pack_frames
    frames, sizes = pack_frames(c4_clips(T=T, seed=40))
    frames = frames.cuda()
    ref = s2d_of_clip(frames_to_clip(frames, sizes, size, **norm))
    got = to_s2d(frames, sizes, size, **norm)
    assert got.shape == ref.shape and torch.equal(got, ref)
    assert not got[..., 24:].any()


def test_clips_of_a_mixed_batch_are_independent():
    from step_b200.frames import frames_to_clip, pack_frames
    clips = c4_clips(T=8, seed=80)
    frames, sizes = pack_frames(clips)
    batch = frames_to_clip(frames.cuda(), sizes, (224, 224), **NORM)
    batch_s2d = to_s2d(frames.cuda(), sizes, (224, 224), **NORM)
    for n, c in enumerate(clips):
        f1, s1 = pack_frames([c])
        assert torch.equal(frames_to_clip(f1.cuda(), s1, (224, 224), **NORM)[0], batch[n])
        assert torch.equal(to_s2d(f1.cuda(), s1, (224, 224), **NORM)[0], batch_s2d[n])


def build_nets(cfg):
    import step_b200
    nets = {"base_net": step_b200.BaseNet(cfg), "roi_net": step_b200.ROINet(cfg.pool_mode, cfg.pool_size)}
    nets["base_net"].load_state_dict(synth.base_net_state_dict(), strict=True)
    for i in range(cfg.max_iter):
        h = step_b200.TwoBranchNet(cfg)
        h.load_state_dict(synth.head_state_dict(100 + i, cfg), strict=True)
        nets["det_net%d" % i] = h
    return {k: v.cuda().eval() for k, v in nets.items()}


def snapshot(runner, hist):
    out = []
    for d in hist:
        out += [v.clone() for _, v in sorted(d.items()) if torch.is_tensor(v)]
    for _, d in sorted(runner.detections.items()):   # kept detections only: rows past a clip's count are never written
        cnt = d["count"].cpu()
        out += [cnt] + [d["det"][b, :int(c)].clone() for b, c in enumerate(cnt.tolist())]
    return out


@pytest.mark.parametrize("fp16", [True, False], ids=["fp16", "fp32"])
def test_runner_from_frames_equals_runner_from_clips(fp16):
    import step_b200
    from step_b200.frames import frames_to_clip, pack_frames
    cfg = synth.make_cfg(fp16=fp16, T=8, max_iter=3, NUM_CHUNKS={1: 1, 2: 1, 3: 1}, image_size=(224, 224))
    nets = build_nets(cfg)
    B, N = 8, 11
    tubes = synth.make_proposals(B, N, cfg.T, 224, 224)
    max_hw = (360, 654)
    fr = dict(max_hw=max_hw, **NORM)
    frames, sizes = pack_frames(c4_clips(seed=120), max_hw=max_hw)
    with torch.no_grad():
        by_frames = step_b200.StepRunner(cfg, nets, B, 32, 224, 224, tubes, detect=DETECT, frames=fr)
        by_clips = step_b200.StepRunner(cfg, nets, B, 32, 224, 224, tubes, detect=DETECT)
        a = snapshot(by_frames, by_frames(frames=frames, sizes=sizes))
        x = frames_to_clip(frames.cuda(), sizes, (224, 224), **NORM)
        b = snapshot(by_clips, by_clips(x))
        torch.cuda.synchronize()
        assert len(a) == len(b) and all(torch.equal(u, v) for u, v in zip(a, b))
        # another mix of source sizes, same graph: equals an eager step on the same frames
        frames2, sizes2 = pack_frames(c4_clips(H0=300, widths=[654, 200, 400, 533, 640, 360, 224, 500], seed=160),
                                      max_hw=max_hw)
        again = snapshot(by_frames, by_frames(frames=frames2, sizes=sizes2))
        eager = step_b200.StepRunner(cfg, nets, B, 32, 224, 224, tubes, detect=DETECT, frames=fr, use_graph=False)
        ref = snapshot(eager, eager(frames=frames2, sizes=sizes2))
        torch.cuda.synchronize()
    assert all(torch.equal(u, v) for u, v in zip(again, ref))
    assert not all(torch.equal(u, v) for u, v in zip(again, a))
    with pytest.raises(ValueError):
        by_frames(frames=frames2, sizes=[[361, 654]] * B)

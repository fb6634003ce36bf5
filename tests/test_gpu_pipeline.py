"""GPU: module- and pipeline-level parity against the committed golden vectors (outputs of the
unmodified reference on seeded synthetic inputs) and the oracle.

Tolerances (SURVEY.md section 8c):
  fp32 path (cfg.fp16=False, SIMT):  atol = 1e-4 * max|ref|, rtol = 1e-4   (accumulation order only)
  fp16 path (cfg.fp16=True, tcgen05, fp32 accumulate): max-abs <= 2e-2 * max|ref| at the trunk output,
      mean-relative <= 1e-2; sigmoid scores <= 5e-3 abs; boxes <= 1.5 px.
"""
import numpy as np
import pytest
import torch

from oracle import tubes as otubes
from step_b200 import synth

pytestmark = pytest.mark.gpu

PIPES = {
    "pipe_c1": dict(T=2, max_iter=1, NUM_CHUNKS={1: 1}, image_size=(112, 112)),
    "pipe_spatial": dict(T=4, max_iter=3, NUM_CHUNKS={1: 1, 2: 1, 3: 1}, image_size=(112, 112)),
    "pipe_temporal_predict": dict(T=3, max_iter=3, NUM_CHUNKS={1: 1, 2: 1, 3: 3}, temporal_mode="predict", image_size=(112, 112)),
    "pipe_temporal_extrapolate": dict(T=3, max_iter=3, NUM_CHUNKS={1: 1, 2: 1, 3: 3}, temporal_mode="extrapolate", image_size=(112, 112)),
    "pipe_temporal_mean": dict(T=3, max_iter=3, NUM_CHUNKS={1: 1, 2: 1, 3: 3}, temporal_mode="mean", image_size=(112, 112)),
}


def build(cfg, context=False):
    import step_b200
    nets = {"base_net": step_b200.BaseNet(cfg), "roi_net": step_b200.ROINet(cfg.pool_mode, cfg.pool_size)}
    nets["base_net"].load_state_dict(synth.base_net_state_dict(), strict=True)
    for i in range(cfg.max_iter):
        h = step_b200.TwoBranchNet(cfg)
        h.load_state_dict(synth.head_state_dict(100 + i, cfg), strict=True)
        nets["det_net%d" % i] = h
    if context:
        c = step_b200.ContextNet(cfg)
        c.load_state_dict(synth.context_net_state_dict(), strict=True)
        nets["context_net"] = c
    for k in nets:
        nets[k] = nets[k].cuda().eval()
        if hasattr(nets[k], "set_device"):
            nets[k].set_device("cuda:0")
    return nets


def run(name, g, fp16, context=False, **cfg_kw):
    import step_b200
    cfg = synth.make_cfg(fp16=fp16, **cfg_kw)
    nets = build(cfg, context)
    B, T_in, HW, N = int(g["B"]), int(g["T_in"]), int(g["HW"]), int(g["N"])
    x = synth.make_clips(B, T_in, HW, HW).cuda()
    tubes = synth.make_proposals(B, N, cfg.T * cfg.NUM_CHUNKS[1], HW, HW)
    with torch.no_grad():
        cf = nets["base_net"](x)
        ctx = nets["context_net"](cf) if context else None
        hist, traj = step_b200.inference(cfg, cf, ctx, nets, cfg.max_iter, tubes)
    torch.cuda.synchronize()
    return cfg, cf, ctx, hist, traj


def check(name, g, cfg, cf, hist, traj, fp16):
    HW = int(g["HW"])
    if "conv_feat" in g:
        ref = g["conv_feat"]
        got = cf.float().cpu().numpy()
        assert got.shape == ref.shape
        mx = np.abs(ref).max()
        if fp16:
            assert np.abs(got - ref).max() <= 2e-2 * mx
            assert np.abs(got - ref).mean() <= 1e-2 * np.abs(ref).mean()
        else:
            assert np.allclose(got, ref, rtol=1e-4, atol=1e-4 * mx)
    p_tol = 5e-3 if fp16 else 2e-5
    b_tol = 1.5 if fp16 else 2e-3
    for i, h in enumerate(hist):
        assert np.abs(h["pred_prob"][:, 0].float().cpu().numpy() - g["prob%d" % i]).max() <= p_tol, (name, i)
        extends = i + 1 < cfg.max_iter and cfg.NUM_CHUNKS[i + 2] == cfg.NUM_CHUNKS[i + 1] + 2
        loc = h["pred_loc"].cpu().numpy()
        v = loc if extends else otubes.valid_tubes(loc, HW, HW)
        assert np.abs(v - g["loc_valid%d" % i]).max() <= b_tol, (name, i)
        if "first%d" % i in g and h["pred_first_loc"] is not None:
            assert np.abs(h["pred_first_loc"].cpu().numpy() - g["first%d" % i]).max() <= b_tol
            assert np.abs(h["pred_last_loc"].cpu().numpy() - g["last%d" % i]).max() <= b_tol
        assert list(h["tubes_nums"]) == g["nums%d" % i].tolist()
        tr = np.concatenate([t[0] for t in traj[i]], 0)
        assert tr.shape == g["traj%d" % i].shape and np.abs(tr - g["traj%d" % i]).max() <= b_tol, (name, i)


@pytest.mark.parametrize("fp16", [False, True], ids=["fp32", "fp16"])
@pytest.mark.parametrize("name", list(PIPES))
def test_pipeline_matches_reference_golden(golden, name, fp16):
    g = golden(name)
    cfg, cf, ctx, hist, traj = run(name, g, fp16, **PIPES[name])
    assert tuple(cf.shape) == (int(g["B"]), int(g["T_in"]) // 4, 832, int(g["HW"]) // 16, int(g["HW"]) // 16)
    check(name, g, cfg, cf, hist, traj, fp16)


@pytest.mark.parametrize("fp16", [False, True], ids=["fp32", "fp16"])
def test_native_ava_shape_with_context(golden, fp16):
    """36x400x400, N=3, temporal predict, ContextNet on -- the reference's shipped configuration."""
    g = golden("pipe_ava_context")
    cfg, cf, ctx, hist, traj = run("pipe_ava_context", g, fp16, context=True, T=3, max_iter=3,
                                   NUM_CHUNKS={1: 1, 2: 1, 3: 3}, no_context=False, image_size=(400, 400))
    sub = cf.float().cpu().numpy()[:, ::4, ::13, ::6, ::6]
    ref = g["conv_feat_sub"]
    tol = (2e-2 if fp16 else 1e-4) * np.abs(ref).max()
    assert np.abs(sub - ref).max() <= tol
    cref = g["context_feat"]
    assert ctx.shape == cref.shape
    assert np.abs(ctx.float().cpu().numpy() - cref).max() <= (2e-2 if fp16 else 1e-4) * np.abs(cref).max()
    check("pipe_ava_context", g, cfg, cf, hist, traj, fp16)


def test_reference_style_driver_calls():
    """The call pattern of test.py:145-162: module(...) on tensors, .contiguous() slices, ROINet on
    logical tensors, TwoBranchNet.forward on the 5-D pooled tensor -- results equal the fused path."""
    import step_b200
    cfg = synth.make_cfg(fp16=True, T=4, max_iter=1, NUM_CHUNKS={1: 1}, image_size=(112, 112))
    nets = build(cfg)
    x = synth.make_clips(2, 16, 112, 112).cuda()
    tubes = synth.make_proposals(2, 3, 4, 112, 112)
    with torch.no_grad():
        cf = nets["base_net"](x)
        hist, _ = step_b200.inference(cfg, cf, None, nets, 1, tubes)
        flat, nums = step_b200.tube_utils.flatten_tubes(tubes, batch_idx=True)
        flat = torch.from_numpy(flat).cuda()
        pooled = nets["roi_net"](cf[:, 0:4].contiguous(), flat)           # utils.py:48 (NCHW copy path)
        pooled2 = nets["roi_net"](cf, flat)                                 # channels-last view path
        assert torch.equal(pooled.float(), pooled2.float())
        _, C, W, H = pooled.shape
        prob, loc, first, last, l0, l1, l2 = nets["det_net0"](pooled2.view(-1, 4, C, W, H))
    # the fused pipeline pools with the packed-half2 ROIAlign fast path, the op-level call with the exact one
    assert torch.allclose(prob, hist[0]["pred_prob"][:, 0], atol=5e-3)
    dec = step_b200.tube_utils.decode_coef(flat.view(-1, 5)[:, 1:].contiguous(), loc.view(-1, 4))
    assert torch.allclose(dec.view(loc.shape), hist[0]["pred_loc"], atol=0.5)
    assert l0.numel() == 1 and float(l0) == 0.0


def test_full_size_c4_properties():
    """BASELINE.json config 4 at full size (B=8, T=32, 224x224, 11 proposals, 3 steps), size-independent
    properties: (1) determinism; (2) the CUDA-graph replay equals the eager launch sequence bit for bit;
    (3) clips are independent units -- the first 4 clips run alone reproduce their rows of the 8-clip batch
    bit for bit (what makes the clip-parallel multi-GPU sharding exact); (4) per-class NMS on the result is
    idempotent and keeps ascending indices."""
    import step_b200
    from step_b200.roi_layers import nms
    cfg = synth.make_cfg(fp16=True, T=8, max_iter=3, NUM_CHUNKS={1: 1, 2: 1, 3: 1}, image_size=(224, 224))
    nets = build(cfg)
    B, N = 8, 11
    x = synth.make_clips(B, 32, 224, 224).cuda()
    tubes = synth.make_proposals(B, N, cfg.T, 224, 224)

    def eager(xx, tb):
        with torch.no_grad():
            cf = nets["base_net"](xx)
            h, _ = step_b200.inference(cfg, cf, None, nets, cfg.max_iter, tb, want_trajectory=False)
        return [(d["pred_prob"][:, 0].clone(), d["pred_loc"].clone()) for d in h]

    a, b = eager(x, tubes), eager(x, tubes)
    for (p0, l0), (p1, l1) in zip(a, b):
        assert torch.equal(p0, p1) and torch.equal(l0, l1)                      # (1)
    runner = step_b200.StepRunner(cfg, nets, B, 32, 224, 224, tubes)
    g = [(d["pred_prob"][:, 0].clone(), d["pred_loc"].clone()) for d in runner(x)]
    g2 = [(d["pred_prob"][:, 0].clone(), d["pred_loc"].clone()) for d in runner(x)]
    for (p0, l0), (p1, l1), (p2, l2) in zip(a, g, g2):
        assert torch.equal(p0, p1) and torch.equal(l0, l1) and torch.equal(p1, p2) and torch.equal(l1, l2)   # (2)
    half = eager(x[:4].contiguous(), tubes[:4])
    for (p0, l0), (ph, lh) in zip(a, half):
        assert torch.equal(p0[:4 * N], ph) and torch.equal(l0[:4 * N], lh)      # (3)
    assert all(torch.isfinite(p).all() and torch.isfinite(l).all() for p, l in a)
    prob, loc = a[-1]
    boxes = loc[:N, cfg.T // 2].contiguous()
    keep = nms(boxes, prob[:N, 0].contiguous(), 0.4)
    again = nms(boxes[keep], prob[:N, 0][keep].contiguous(), 0.4)
    assert torch.equal(again.cpu(), torch.arange(keep.numel())) and bool((keep[1:] > keep[:-1]).all())   # (4)


@pytest.mark.parametrize("mode", ["spatial", "predict"])
def test_ragged_and_empty_clips_match_oracle(mode):
    """Clips with different tube counts, one of them with none (flatten_tubes skips it but still counts it,
    tube_utils.py:214-246): frame indices, per-clip bookkeeping and the between-steps update must agree with the
    reference arithmetic (oracle/model.py) on the fp32 path."""
    import step_b200
    from oracle import model as om
    if mode == "spatial":
        kw = dict(T=4, max_iter=2, NUM_CHUNKS={1: 1, 2: 1}, image_size=(112, 112))
        T_in = 16
    else:
        kw = dict(T=3, max_iter=2, NUM_CHUNKS={1: 1, 2: 3}, temporal_mode="predict", image_size=(112, 112))
        T_in = 36
    cfg = synth.make_cfg(fp16=False, **kw)
    nets = build(cfg)
    B = 3
    x = synth.make_clips(B, T_in, 112, 112)
    tubes = synth.make_proposals(B, 3, cfg.T * cfg.NUM_CHUNKS[1], 112, 112)
    tubes[1] = tubes[1][:0]
    tubes[2] = tubes[2][:2]
    with torch.no_grad():
        cf = nets["base_net"](x.cuda())
        hist, traj = step_b200.inference(cfg, cf, None, nets, cfg.max_iter, [t.copy() for t in tubes])
        torch.cuda.synchronize()
        sd = synth.base_net_state_dict()
        heads = [synth.head_state_dict(100 + i, cfg) for i in range(cfg.max_iter)]
        rhist, rtraj = om.inference(cfg, om.base_net(x, sd), None, heads, cfg.max_iter, [t.copy() for t in tubes])
    for i, (h, r) in enumerate(zip(hist, rhist)):
        assert list(h["tubes_nums"]) == list(r["tubes_nums"]) == [3, 0, 2]
        assert np.abs(h["pred_prob"].float().cpu().numpy() - r["pred_prob"].numpy()).max() <= 2e-5, i
        extends = i + 1 < cfg.max_iter and cfg.NUM_CHUNKS[i + 2] == cfg.NUM_CHUNKS[i + 1] + 2
        loc, rloc = h["pred_loc"].cpu().numpy(), r["pred_loc"].numpy()
        if not extends:   # the reference's CPU path validates pred_loc in place on these steps (aliasing)
            loc, rloc = otubes.valid_tubes(loc, 112, 112), otubes.valid_tubes(rloc.copy(), 112, 112)
        assert np.abs(loc - rloc).max() <= 2e-3, i
        for b in range(B):
            got, ref = traj[i][b][0], rtraj[i][b][0]
            assert got.shape == ref.shape
            if got.size:
                assert np.abs(got - ref).max() <= 2e-3, (i, b)


# ---- parity at the MEASURED configurations (BASELINE.json configs[3] = C4, configs[1] = C2) -------------------------
C4 = dict(T=8, max_iter=3, NUM_CHUNKS={1: 1, 2: 1, 3: 1}, image_size=(224, 224))


def _feat_check(got_sub, ref_sub, fp16):
    mx = np.abs(ref_sub).max()
    err = np.abs(got_sub - ref_sub)
    if fp16:
        assert err.max() <= 2e-2 * mx, err.max() / mx
        assert err.mean() <= 1e-2 * np.abs(ref_sub).mean()
    else:
        assert np.allclose(got_sub, ref_sub, rtol=1e-4, atol=1e-4 * mx), err.max() / mx
    return float(err.max() / mx)


@pytest.mark.parametrize("fp16", [False, True], ids=["fp32", "fp16"])
def test_c4_bench_batch_matches_reference_golden(golden, fp16):
    """The exact batch bench.py times (B=8 clips of T=32 x 224 x 224, 11 proposals, 3 steps, seeded) against the
    reference's outputs for clips 0 and 7 (tests/golden/pipe_c4.npz): trunk features, scores, boxes, neighbour boxes
    and proposals of every refinement step.  At B=8 every conv layer takes the dispatch branch the benchmark takes
    (persistent / pair kernels with one CTA per SM, the shared-memory patch kernel at grid 3136, deep single-CTA
    pipelines, multiple N tiles), so a wrong branch fails here.  Through the CUDA-graph runner on the fp16 path."""
    import step_b200
    g = golden("pipe_c4")
    cfg = synth.make_cfg(fp16=fp16, **C4)
    nets = build(cfg)
    B, N = int(g["B"]), int(g["N"])
    x = synth.make_clips(B, int(g["T_in"]), 224, 224).cuda()
    tubes = synth.make_proposals(B, N, cfg.T, 224, 224)
    with torch.no_grad():
        if fp16:
            runner = step_b200.StepRunner(cfg, nets, B, int(g["T_in"]), 224, 224, tubes)
            hist = runner(x)
            cf = nets["base_net"](x)
        else:
            cf = nets["base_net"](x)
            hist, _ = step_b200.inference(cfg, cf, None, nets, cfg.max_iter, tubes, want_trajectory=False)
    torch.cuda.synchronize()
    p_tol, b_tol = (5e-3, 1.5) if fp16 else (2e-5, 2e-3)
    for c in g["clips"].tolist():
        sub = cf[c:c + 1].float().cpu().numpy()[:, :, ::4]
        _feat_check(sub, g["feat_sub_c%d" % c], fp16)
        rows = slice(c * N, (c + 1) * N)
        for i, h in enumerate(hist):
            assert np.abs(h["pred_prob"][rows, 0].float().cpu().numpy() - g["prob%d_c%d" % (i, c)]).max() <= p_tol, (c, i)
            loc = otubes.valid_tubes(h["pred_loc"][rows].cpu().numpy(), 224, 224)
            assert np.abs(loc - g["loc_valid%d_c%d" % (i, c)]).max() <= b_tol, (c, i)
            assert np.abs(h["pred_first_loc"][rows].cpu().numpy() - g["first%d_c%d" % (i, c)]).max() <= b_tol, (c, i)
            assert np.abs(h["pred_last_loc"][rows].cpu().numpy() - g["last%d_c%d" % (i, c)]).max() <= b_tol, (c, i)


def test_c2_trunk_batch4_matches_reference_golden(golden):
    """BASELINE.json configs[1]: I3D trunk, batch 4, T=32, 224x224, fp16 tensor-core path, against the reference's
    trunk output for clips 0 and 3 of the seeded batch (tests/golden/trunk_c2.npz)."""
    import step_b200
    g = golden("trunk_c2")
    cfg = synth.make_cfg(fp16=True, T=8, max_iter=1, NUM_CHUNKS={1: 1}, image_size=(224, 224))
    net = step_b200.BaseNet(cfg)
    net.load_state_dict(synth.base_net_state_dict(), strict=True)
    net = net.cuda().eval()
    x = synth.make_clips(4, 32, 224, 224).cuda()
    with torch.no_grad():
        cf = net(x)
    torch.cuda.synchronize()
    assert tuple(cf.shape) == (4, 8, 832, 14, 14)
    for c in (0, 3):
        _feat_check(cf[c:c + 1].float().cpu().numpy()[:, :, ::4], g["feat_sub_c%d" % c], True)


def test_c4_detection_set_fp16_equals_fp32_reference(golden):
    """Detection-level agreement: per-class NMS detections (test.py:156-218, run on the device by
    step_b200.postprocess inside the captured step) computed from OUR fp16 pipeline vs the rows the reference's own
    evaluation loop wrote from ITS fp32 outputs for the same two clips (postprocess_cases.npz 'c4').  The confidence
    threshold sits in the widest score gap, so fp16 score noise cannot move a candidate across it: the kept
    (clip, class, tube) sets must be identical, scores within 5e-3 and normalised boxes within 1.5 px."""
    import step_b200
    from step_b200 import postprocess as pp
    g, pc = golden("pipe_c4"), golden("postprocess_cases")
    conf, thr, topk, width, height = pc["c4_cfg"].tolist()
    cfg = synth.make_cfg(fp16=True, **C4)
    nets = build(cfg)
    N = int(g["N"])
    xs = synth.make_clips(8, 32, 224, 224)
    x = torch.stack([xs[0], xs[7]]).cuda()
    tubes = synth.make_proposals(2, N, cfg.T, 224, 224)
    runner = step_b200.StepRunner(cfg, nets, 2, 32, 224, 224, tubes,
                                  detect=dict(conf_thresh=conf, nms_thresh=thr, topk=int(topk)))
    with torch.no_grad():
        hist = runner(x)
    torch.cuda.synchronize()
    last = hist[cfg.max_iter - 1]
    # the in-graph detector == the stand-alone call on the same history (bit for bit)
    again = pp.detect(last["pred_prob"], last["pred_loc"], runner.tubes_nums, conf, thr, width, height, topk=int(topk))
    ing = runner.detections[cfg.max_iter - 1]
    assert torch.equal(again["count"], ing["count"]) and torch.equal(again["keep"], ing["keep"])
    # The reference rows come from its CPU run, where valid_tubes(image_size) has already clamped history['pred_loc']
    # in place through the shared numpy view (utils.py:107-121, DESIGN.md section 5); on the GPU it does not.  Apply
    # the same clamp first so that the two detection sets describe the same boxes.
    loc_v = step_b200.tube_utils.valid_tubes(last["pred_loc"].clone(), 224, 224)
    got = pp.to_lists(pp.detect(last["pred_prob"], loc_v, runner.tubes_nums, conf, thr, width, height, topk=int(topk)))
    ref = pc["c4_rows"]
    # reference rows (clip, class, score, box) -> tube index by matching against the reference's own candidates
    rprob = np.concatenate([g["prob2_c0"], g["prob2_c7"]], 0)
    worst_s, worst_b = 0.0, 0.0
    for b in range(2):
        rr = ref[ref[:, 0] == b]
        assert len(got[b]) == rr.shape[0], (b, len(got[b]), rr.shape[0])
        # same classes in the same file order, same number of detections per class
        assert [c for _, c, _ in got[b]] == rr[:, 1].astype(int).tolist()
        for (bx, c, s), r in zip(got[b], rr):
            worst_s = max(worst_s, abs(s - r[2]))
            worst_b = max(worst_b, float(np.abs(bx * 224.0 - r[3:7] * 224.0).max()))
    assert worst_s <= 5e-3 and worst_b <= 1.5, (worst_s, worst_b)
    assert rprob.shape == (2 * N, cfg.num_classes)


def test_reference_driver_loop_through_compat_patch():
    """The structure of the reference's test.py:62-218 (a restatement -- the GPU box has no /root/reference) run against the
    names the reference imports, after `step_b200.compat.patch()`: `from models import ...`,
    `from external.maskrcnn_benchmark.roi_layers import nms`, `nn.DataParallel(base_net)`, `.cuda()`,
    `load_state_dict(checkpoint[...])`, `set_device`, `.eval()`, `inference(...)`, then the per-clip x per-class evaluation
    loop with `valid_tubes` and `nms` on CPU tensors.  Its detections must equal the on-device post-processing."""
    import sys
    from collections import OrderedDict
    import step_b200.compat as compat
    saved = {k: sys.modules.get(k) for k in ("models", "external", "external.maskrcnn_benchmark", "external.maskrcnn_benchmark.roi_layers")}
    try:
        compat.patch()
        from models import BaseNet, ROINet, TwoBranchNet                         # test.py:21
        from external.maskrcnn_benchmark.roi_layers import nms                    # test.py:23
        from step_b200 import inference, postprocess as pp
        from step_b200.tube_utils import valid_tubes
        args = synth.make_cfg(fp16=True, T=4, max_iter=2, NUM_CHUNKS={1: 1, 2: 1}, image_size=(112, 112))
        args.conf_thresh, args.nms_thresh, args.topk, args.evaluate_topk = 0.3, 0.4, 20, 20
        checkpoint = {"base_net": OrderedDict(("module." + k, v) for k, v in synth.base_net_state_dict().items())}
        for i in range(args.max_iter):
            checkpoint["det_net%d" % i] = synth.head_state_dict(100 + i, args)
        nets = OrderedDict()                                                      # test.py:62-95
        nets['base_net'] = BaseNet(args)
        nets['roi_net'] = ROINet(args.pool_mode, args.pool_size)
        for i in range(args.max_iter):
            nets['det_net%d' % i] = TwoBranchNet(args)
        for key in nets:
            nets[key] = nets[key].cuda()
        nets['base_net'] = torch.nn.DataParallel(nets['base_net'], device_ids=[0])
        for i in range(args.max_iter):
            nets['det_net%d' % i].to('cuda:0')
            nets['det_net%d' % i].set_device('cuda:0')
        nets['base_net'].load_state_dict(checkpoint['base_net'])
        for i in range(args.max_iter):
            nets['det_net%d' % i].load_state_dict(checkpoint['det_net%d' % i])
        for _, net in nets.items():
            net.eval()
        images = synth.make_clips(2, 16, 112, 112)
        tubes = synth.make_proposals(2, 5, 4, 112, 112)
        width = height = 112
        with torch.no_grad():                                                     # test.py:121-162
            conv_feat = nets['base_net'](images.cuda())
            history, _ = inference(args, conv_feat, None, nets, args.max_iter, tubes)
            per_step = []
            for i in range(len(history)):
                pred_prob = history[i]['pred_prob'].cpu()
                pred_prob = pred_prob[:, int(pred_prob.shape[1] / 2)]
                pred_tubes = history[i]['pred_loc'].cpu()
                pred_tubes = pred_tubes[:, int(pred_tubes.shape[1] / 2)]
                tubes_nums = history[i]['tubes_nums']
                tubes_count, clips_out = 0, []
                for b in range(len(tubes_nums)):                                  # test.py:166-210
                    seq_start = tubes_count
                    tubes_count = tubes_count + tubes_nums[b]
                    cur_prob, cur_tubes = pred_prob[seq_start:seq_start + tubes_nums[b]], pred_tubes[seq_start:seq_start + tubes_nums[b]]
                    scores_list = []
                    for cl_ind in range(args.num_classes):
                        scores = cur_prob[:, cl_ind].reshape(-1)
                        c_mask = scores.gt(args.conf_thresh)
                        scores = scores[c_mask]
                        if len(scores) == 0:
                            continue
                        boxes = cur_tubes.clone()[c_mask.unsqueeze(1).expand_as(cur_tubes)].view(-1, 4)
                        boxes = torch.from_numpy(valid_tubes(boxes.view(-1, 1, 4).numpy())).view(-1, 4)
                        keep = nms(boxes, scores, args.nms_thresh)
                        assert keep.device.type == "cpu" and keep.dtype == torch.int64
                        for j in keep.tolist():
                            scores_list.append((float(scores[j]), cl_ind, (boxes[j] / torch.tensor([width, height, width, height])).tolist()))
                    scores_list.sort(key=lambda t: t[0])
                    scores_list = scores_list[::-1][:args.topk]
                    clips_out.append(scores_list)
                per_step.append(clips_out)
            last = history[-1]
            det = pp.to_lists(pp.detect(last['pred_prob'], last['pred_loc'], last['tubes_nums'], args.conf_thresh, args.nms_thresh,
                                        width, height, topk=args.topk))
        for b in range(2):
            ref = per_step[-1][b]
            assert len(ref) == len(det[b]) and len(ref) > 0
            assert [c for _, c, _ in ref] == [c for _, c, _ in det[b]]
            for (s, c, bx), (dbx, dc, ds) in zip(ref, det[b]):
                assert abs(s - ds) <= 1e-6 and np.abs(np.asarray(bx) - dbx).max() <= 1e-5
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def test_fused_bottleneck_exit_does_not_change_the_pipeline(golden):
    """fp16 inference with the fused block exits (step_bottleneck_exit_f16, three launches per refinement step) produces
    the same bits as the layer-by-layer launches."""
    from step_b200 import engine as E
    name = "pipe_spatial"
    g = golden(name)
    outs = []
    old = E.FUSE_EXIT
    try:
        for fuse in (True, False):
            E.FUSE_EXIT = fuse
            cfg, cf, ctx, hist, traj = run(name, g, True, **PIPES[name])
            outs.append(hist)
    finally:
        E.FUSE_EXIT = old
    for a, b in zip(*outs):
        assert torch.equal(a["pred_prob"], b["pred_prob"])
        assert torch.equal(a["pred_loc"], b["pred_loc"])


def test_bench_with_three_batches_in_flight_completes():
    """bench.py's measured configuration (CUDA graphs, three batches in flight on separate streams) runs to completion and
    prints its JSON line.  A kernel that only works when it has the GPU to itself shows up here as a timeout: an
    experimental variant of the fused bottleneck exit passed every single-stream test and stalled exactly this run
    (tools/experiments/README.md).  What --dump-outputs writes equals one eager step on the same seeded inputs."""
    import json
    import os
    import subprocess
    import sys
    import tempfile
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with tempfile.TemporaryDirectory() as td:
        r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "40", "--warmup", "3", "--skip-cpu",
                            "--dump-outputs", td], capture_output=True, text=True, timeout=240, cwd=root)
        assert r.returncode == 0, r.stderr[-2000:]
        j = json.loads(r.stdout.strip().splitlines()[-1])
        assert j["config"]["batches_in_flight"] == 3 and j["value"] > 0 and j["gpu_launches"] > 0
        # the last timed step's outputs: 8 clips x 11 proposals, 60 classes, 3 refinement steps, the kept detections
        det, count = np.load(os.path.join(td, "det.npy")), np.load(os.path.join(td, "count.npy"))
        prob = np.load(os.path.join(td, "step2_pred_prob.npy"))
        assert det.dtype == count.dtype == prob.dtype == np.float32
        assert prob.shape == (88, 60) and np.isfinite(prob).all() and det.shape[0] == count.shape[0] == 8
        assert count.sum() > 0 and (count <= det.shape[1]).all()
        # ... and they are what one eager step of the same workload computes, bit for bit
        import importlib.util
        import step_b200
        spec = importlib.util.spec_from_file_location("bench", os.path.join(root, "bench.py"))
        bench = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(bench)
        cfg, clips, tubes = bench.workload(0)
        W = bench.WORKLOAD
        runner = step_b200.StepRunner(cfg, bench.build_nets(cfg, torch.device("cuda", 0)), W["B"], W["T_in"], W["HW"], W["HW"],
                                      tubes, use_graph=False, detect=bench.DETECT)
        with torch.no_grad():
            hist = runner(clips.cuda())
        torch.cuda.synchronize()
        eager = os.path.join(td, "eager")
        bench.dump_outputs(eager, hist, runner.detections[cfg.max_iter - 1], None)
        names = sorted(n for n in os.listdir(td) if n.endswith(".npy"))
        assert names == sorted(os.listdir(eager)) and "step2_pred_loc.npy" in names
        for n in names:
            assert np.array_equal(np.load(os.path.join(td, n)), np.load(os.path.join(eager, n))), n

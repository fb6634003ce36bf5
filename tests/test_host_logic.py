"""CPU: host-side logic of the package -- weight packing, BN folding, the space-to-depth stem
rewrite, pooling extents, tube list bookkeeping, state-dict key parity."""
import pytest
import numpy as np
import torch
import torch.nn.functional as F

from oracle import model as om
from oracle import tubes as otubes
from step_b200 import engine as E
from step_b200 import synth, tube_utils


def test_pool_extent_matches_torch():
    for size in (7, 8, 13, 14, 16, 25, 28, 56, 112):
        for k, s in ((3, 2), (3, 1), (1, 1), (2, 2)):
            lo, hi = E.same_pad(k, s)
            x = torch.zeros(1, 1, size + lo + hi, 1, 1)
            ref = F.max_pool3d(x, (k, 1, 1), (s, 1, 1), ceil_mode=True).shape[2]
            assert E.pool_out(size, k, s)[0] == ref, (size, k, s)


def test_pack_conv_weight_layout():
    w = torch.randn(5, 3, 2, 3, 4)
    p = E.pack_conv_weight(w, 0)
    assert p.shape == (5, 24, 4)
    assert torch.equal(p[2, (1 * 3 + 2) * 4 + 3, :3], w[2, :, 1, 2, 3]) and float(p[..., 3].abs().max()) == 0


def test_s2d_stem_is_the_same_convolution():
    """7x7x7/2 'SAME' conv == 4x4x4/1 conv (pad 1 low, 2 high) over the space-to-depth input."""
    g = torch.Generator().manual_seed(0)
    w = torch.randn(4, 3, 7, 7, 7, generator=g)
    x = torch.randn(1, 3, 8, 12, 10, generator=g)
    ref = F.conv3d(F.pad(x, (2, 3, 2, 3, 2, 3)), w, stride=2)
    wp = E.pack_stem_s2d(w).float()                       # [4, 64, 32]
    xs = x.view(1, 3, 4, 2, 6, 2, 5, 2).permute(0, 2, 4, 6, 3, 5, 7, 1).reshape(1, 4, 6, 5, 24)  # N,T2,H2,W2,(rt,rh,rw,c)
    xs = F.pad(xs, (0, 8)).permute(0, 4, 1, 2, 3)          # -> N,32,T2,H2,W2
    w2 = wp.view(4, 4, 4, 4, 32).permute(0, 4, 1, 2, 3)    # co, c, qt, qh, qw
    out = F.conv3d(F.pad(xs, (1, 2, 1, 2, 1, 2)), w2)
    assert out.shape == ref.shape
    assert torch.allclose(out, ref, atol=2e-2, rtol=1e-2)  # fp16-rounded weights


def test_fold_bn_matches_batchnorm():
    bn = torch.nn.BatchNorm3d(6).eval()
    with torch.no_grad():
        bn.weight.uniform_(0.5, 1.5); bn.bias.normal_(); bn.running_mean.normal_(); bn.running_var.uniform_(0.5, 2)
    s, b = E.fold_bn(bn, None, 6, "cpu")
    x = torch.randn(2, 6, 3, 4, 5)
    assert torch.allclose(bn(x), x * s.view(1, -1, 1, 1, 1) + b.view(1, -1, 1, 1, 1), atol=1e-5)


def test_flatten_tubes_matches_oracle():
    rs = np.random.RandomState(0)
    lst = [rs.rand(2, 3, 4).astype(np.float32), np.zeros((0, 3, 4), np.float32), rs.rand(4, 3, 4).astype(np.float32)]
    a, na = tube_utils.flatten_tubes(lst, True)
    b, nb = otubes.flatten_tubes(lst, True)
    assert np.array_equal(a, b) and na == nb


def test_state_dict_keys_match_reference_counts():
    import step_b200
    cfg = synth.make_cfg(no_context=False)
    assert len(step_b200.BaseNet(cfg).state_dict()) == 270       # SURVEY.md section 5 [probe]
    assert len(step_b200.TwoBranchNet(cfg).state_dict()) == 94
    assert len(step_b200.ContextNet(cfg).state_dict()) == 72
    step_b200.BaseNet(cfg).load_state_dict(synth.base_net_state_dict(), strict=True)
    step_b200.TwoBranchNet(cfg).load_state_dict(synth.head_state_dict(1, cfg), strict=True)


def test_oracle_same_pad_table():
    assert om.same_pad(7, 2) == (2, 3) and om.same_pad(3, 1) == (1, 1) and om.same_pad(3, 2) == (0, 1)
    assert E.same_pad(7, 2) == (2, 3) and E.same_pad(1, 1) == (0, 0)


# The part of the reference tree its drivers' import lines (test.py:19-25) reach: a `models` package, `utils/utils.py`
# (the progressive `inference`, which imports its helpers from `utils/tube_utils.py`) and `utils/tube_utils.py`.  The
# stand-in below has that layout; importing its `models` package or calling any of its functions fails.
STAND_IN_REFERENCE = {
    "models/__init__.py": "raise ImportError('the stand-in reference models package was imported')\n",
    "utils/__init__.py": "",
    "utils/tube_utils.py": "".join("def %s(*args, **kwargs):\n    raise AssertionError('stand-in')\n\n\n" % n for n in (
        "compute_box_iou", "compute_tube_iou", "decode_coef", "extrapolate_tubes", "flatten_tubes", "valid_tubes")),
    # the helpers the reference's utils/utils.py takes from utils.tube_utils at import time (utils.py:13)
    "utils/utils.py": ("from utils.tube_utils import (compute_tube_iou, decode_coef, extrapolate_tubes, flatten_tubes,\n"
                       "                              valid_tubes)\n"
                       "\n\ndef inference(args, conv_feat, context_feat, nets, exec_iter, tubes):\n"
                       "    raise AssertionError('the stand-in reference inference ran')\n"),
}


def test_compat_patch_substitutes_the_names_the_reference_drivers_import(tmp_path):
    """After compat.patch(<reference root>) the reference's own import lines (test.py:19-25) resolve to step_b200, and
    its utils.utils.inference IS ours -- without editing a reference file.  Runs on a stand-in tree with the reference's
    module layout, so that a `models` package in the tree must lose to ours."""
    import sys
    import step_b200
    import step_b200.compat as compat
    for rel, text in STAND_IN_REFERENCE.items():
        (tmp_path / rel).parent.mkdir(parents=True, exist_ok=True)
        (tmp_path / rel).write_text(text)
    saved = dict(sys.modules)
    saved_path = list(sys.path)
    try:
        for k in [k for k in sys.modules if k == "models" or k.startswith("models.") or k.startswith("external") or k == "utils" or k.startswith("utils.")]:
            del sys.modules[k]
        compat.patch(str(tmp_path))
        ns = {}
        exec("from models import BaseNet, ROINet, TwoBranchNet, ContextNet\n"
             "from external.maskrcnn_benchmark.roi_layers import nms\n"
             "from utils.utils import inference\n"
             "from utils.tube_utils import flatten_tubes, valid_tubes", ns)          # the import lines of test.py:19-25
        assert ns["BaseNet"] is step_b200.BaseNet and ns["TwoBranchNet"] is step_b200.TwoBranchNet
        assert ns["nms"] is step_b200.roi_layers.nms and ns["inference"] is step_b200.inference
        assert ns["valid_tubes"].__module__ == "utils.tube_utils"                    # host helpers stay the reference's own
        assert sys.modules["utils.tube_utils"].__file__.startswith(str(tmp_path))
        cfg = __import__("step_b200.synth", fromlist=["x"]).make_cfg()
        net = ns["TwoBranchNet"](cfg)
        net.load_state_dict(__import__("step_b200.synth", fromlist=["x"]).head_state_dict(100, cfg), strict=True)
        with pytest.raises(RuntimeError):                                            # no CPU fallback on the hot path
            net(__import__("torch").zeros(1, 8, 832, 7, 7))
    finally:
        sys.path[:] = saved_path
        for k in list(sys.modules):
            if k not in saved:
                del sys.modules[k]
        sys.modules.update(saved)


def test_fused_exit_barrier_protocol_survives_adversarial_interleavings():
    """tools/protocol_sim.py replays the mbarrier protocol of the fused bottleneck-exit kernel (csrc/bottleneck_exit.cu: TMA
    producers, two MMA-issuing threads, eight epilogue warps per CTA of the pair, asynchronous commit / complete_tx
    deliveries) under random and skewed schedules: no schedule may end blocked (a deadlock or a parity overrun)."""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location(
        "protocol_sim", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "protocol_sim.py"))
    sim = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(sim)
    slow_cta = lambda n: isinstance(n, tuple) and len(n) > 1 and n[1] == 1
    for skew in (None, slow_cta):
        for p_deliver in (0.25, 0.0):
            for store_y in (True, False):
                for seed in range(4):
                    res, info = sim.simulate("v3", seed, tiles=2, store_y=store_y, skew=skew, p_deliver=p_deliver)
                    assert res == "ok", (res, info)


def test_fused_exit_dispatch_rule():
    """engine.can_fuse_exit: the one-launch block exit is used for the reference's head widths on the fp16 inference path only;
    the training forward (tape recording) and every other width keep the per-layer launches."""
    from step_b200 import _lib as L
    from step_b200 import engine as E
    assert E.can_fuse_exit(L.F16, 256, 1024, 256)
    assert not E.can_fuse_exit(L.F32, 256, 1024, 256)
    assert not E.can_fuse_exit(L.F16, 128, 1024, 256)
    assert not E.can_fuse_exit(L.F16, 256, 1024, 512)
    old = E.TAPE
    try:
        E.TAPE = []
        assert not E.can_fuse_exit(L.F16, 256, 1024, 256)
    finally:
        E.TAPE = old
    old = E.FUSE_EXIT
    try:
        E.FUSE_EXIT = False
        assert not E.can_fuse_exit(L.F16, 256, 1024, 256)
    finally:
        E.FUSE_EXIT = old

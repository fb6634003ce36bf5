"""`BaseNet` and `ROINet` with the reference's constructor / forward signatures and state_dict keys
(models/networks.py:17-142), running on libstep_b200.so.

BaseNet.forward(x[N,T,C,H,W]) -> [N,T/4,832,H/16,W/16] (same logical shape as the reference,
networks.py:69-83).  The result is a permuted *view* of a channels-last buffer: downstream code of
ours (ROINet, inference) consumes the physical layout directly; a caller that does
`.contiguous()` (utils/utils.py:48) simply gets the reference's NCHW layout.
"""
import os

import torch
import torch.nn as nn
import torch.nn.init as init

from . import _lib as L
from . import engine as E
from .engine import Act
from .i3d import build_trunk_stages
from .roi_layers import ROIAlign, ROIPool


def weights_init(m):
    """networks.py:101-105"""
    if isinstance(m, (nn.Conv2d, nn.Linear, nn.Conv3d)):
        init.xavier_normal_(m.weight.data)
        if m.bias is not None:
            init.constant_(m.bias.data, 0.0)


def act_of(t):
    """Recover the channels-last handle behind a logical [N,T,C,H,W] tensor we produced, or None."""
    if t.dim() != 5:
        return None
    phys = t.permute(0, 1, 3, 4, 2)
    if phys.is_contiguous():
        return Act(phys)
    # channel slice of a wider contiguous buffer
    n, tt, h, w, c = phys.shape
    st = phys.stride()
    if st[4] == 1 and st[2] == w * st[3] and st[1] == h * st[2] and st[0] == tt * st[1] and st[3] >= c:
        ld = st[3]
        base = torch.as_strided(phys, (n, tt, h, w, ld), (tt * h * w * ld, h * w * ld, w * ld, ld, 1))
        return Act(base, c, 0)
    return None


def to_act(t, code):
    """Any logical [N,T,C,H,W] CUDA tensor -> Act in `code` precision (zero-copy when it is ours)."""
    L.need_cuda(t)
    a = act_of(t)
    if a is not None and a.code == code:
        return a
    n, tt, c, h, w = t.shape
    src = t.detach().to(torch.float32).contiguous()
    out = Act.empty(n, tt, h, w, c, code, t.device)
    # [N*T, C, H*W] planar -> channels-last
    L.check(L.lib().step_nchw_to_nhwc(L.ptr(src), n * tt, h * w, c, L.ptr(out.buf), code, c, L.stream()))
    return out


class ROINet(nn.Module):
    """networks.py:17-47.  ROIAlign((7,7), 1/16, 0) | ROIPool((7,7), 1/16) over flattened tubes."""

    def __init__(self, pool_mode, pool_size=7):
        super(ROINet, self).__init__()
        self.pool_mode = pool_mode
        self.pool_size = pool_size
        if self.pool_mode == 'pool':
            self.pool_layer = ROIPool((self.pool_size, self.pool_size), 1. / 16.)
        elif self.pool_mode == 'align':
            self.pool_layer = ROIAlign((self.pool_size, self.pool_size), 1. / 16., 0)
        else:
            raise NotImplementedError

    def forward(self, conv_feat, tubes):
        """conv_feat [N,T,C,W,H], tubes [num_tubes,T,5] -> [num_tubes*T, C, 7, 7] (networks.py:34-47)."""
        L.same_device(conv_feat, tubes)
        _, _, C, W, H = conv_feat.size()
        a = act_of(conv_feat)
        if a is not None and self.pool_mode == 'align':
            # channels-last storage: a view [N*T, C, H, W] with channels-last strides, no copy
            feat = a.buf.view(-1, a.H, a.W, a.ld)[..., a.coff:a.coff + a.C].permute(0, 3, 1, 2)
        else:
            feat = conv_feat.reshape(-1, C, W, H)
        return self.pool_layer(feat, tubes.view(-1, 5).detach())

    def pool_into(self, feat, flat_tubes, out, roi_T, feat_T, t_start):
        """Pipeline entry: feat Act [B, feat_T, H, W, C]; flat_tubes [R, roi_T, 5] fp32 CUDA;
        out Act [R*roi_T, 1, 7, 7, ld] channel slice.  Frame indices are relative to the slice
        conv_feat[:, t_start:t_start+roi_T] exactly as utils/utils.py:48 builds it."""
        R = flat_tubes.shape[0] * flat_tubes.shape[1]
        ps = self.pool_size
        fn = L.lib().step_roi_align_fwd_nhwc if self.pool_mode == 'align' else L.lib().step_roi_pool_fwd_nhwc
        args = [L.c_void_p(feat.data_ptr()), feat.code, feat.N * feat.T, feat.H, feat.W, feat.C, feat.ld,
                L.ptr(flat_tubes), R, 1.0 / 16.0, ps, ps]
        if self.pool_mode == 'align':
            args.append(0)
        args += [L.c_void_p(out.data_ptr()), out.ld, roi_T, feat_T, t_start]
        if self.pool_mode == 'align':
            args.append(0 if feat.code == L.F16 else 1)   # fp16 pipeline: FMA fast path (within 1 fp16 ulp)
        args.append(L.stream())
        L.check(fn(*args))
        return out


class BaseNet(nn.Module):
    """networks.py:50-99: the I3D trunk conv3d_1a ... mixed_4f."""

    def __init__(self, cfg):
        super(BaseNet, self).__init__()
        self.base_name = cfg.base_net
        self.kinetics_pretrain = cfg.kinetics_pretrain
        self.freeze_stats = cfg.freeze_stats
        self.freeze_affine = cfg.freeze_affine
        self.fp16 = cfg.fp16
        if self.base_name == "i3d":
            self.base_model = build_base_i3d(self.kinetics_pretrain, self.freeze_affine)
        else:
            raise NotImplementedError

    def forward(self, x):
        """x [N,T,C,H,W] fp32 CUDA -> conv_feat [N,T/4,832,H/16,W/16] (logical view)."""
        L.need_cuda(x)
        with torch.cuda.device(x.device):   # nn.DataParallel replicas (test.py:83) run on their own device + stream
            return self.forward_act(x).logical()

    def forward_act(self, x):
        L.need_cuda(x)
        if x.dim() != 5:
            raise RuntimeError("BaseNet: expected [N,T,C,H,W]")
        code = E.dtype_code(self.fp16)
        N, T, C, H, W = x.shape
        src = x.detach().to(torch.float32).contiguous()
        m = self.base_model
        if code == L.F16 and T % 2 == 0 and H % 2 == 0 and W % 2 == 0 and C == 3:
            # stride-2 stem as a stride-1 4x4x4 filter over the space-to-depth clip (engine.pack_stem_s2d)
            s2d = Act.empty(N, T // 2, H // 2, W // 2, 32, L.F16, x.device)
            L.check(L.lib().step_clip_to_s2d_f16(L.ptr(src), N, T, C, H, W, L.ptr(s2d.buf), 32, L.stream()))
            return self.forward_s2d(s2d)
        if code == L.F16:
            raise RuntimeError("BaseNet(fp16): T, H, W must be even and C == 3")
        cp = (C + 3) // 4 * 4
        a = Act.empty(N, T, H, W, cp, code, x.device)
        L.check(L.lib().step_clip_to_ndhwc(L.ptr(src), N, T, C, H, W, L.ptr(a.buf), code, cp, L.stream()))
        return self._after_stem(m[0](a))

    def forward_s2d(self, s2d):
        """fp16 trunk from the stem's space-to-depth input, an Act [N, T/2, H/2, W/2, 32] (step_clip_to_s2d_f16's layout,
        or step_frames_to_s2d_f16 straight from decoded frames)."""
        if not self.fp16:
            raise RuntimeError("BaseNet.forward_s2d: the space-to-depth stem is the fp16 path")
        return self._after_stem(self.base_model[0].forward_s2d(s2d))

    def _after_stem(self, a):
        m = self.base_model
        for i in range(1, len(m)):
            a = m[i](a)
        return a

    def train(self, mode=True):
        """networks.py:85-99: BatchNorm statistics stay frozen when cfg.freeze_stats (the kernels
        always use running statistics; training through them is not implemented, DESIGN.md)."""
        nn.Module.train(self, mode)
        return self


def build_base_i3d(kinetics_pretrain=None, freeze_affine=True):
    """networks.py:107-142."""
    stages = build_trunk_stages()
    base_model = nn.Sequential(*stages)
    if kinetics_pretrain is not None:
        if os.path.isfile(kinetics_pretrain):
            full = torch.load(kinetics_pretrain, map_location="cpu")
            names = ["conv3d_1a_7x7", None, "conv3d_2b_1x1", "conv3d_2c_3x3", None, "mixed_3b", "mixed_3c", None,
                     "mixed_4b", "mixed_4c", "mixed_4d", "mixed_4e", "mixed_4f"]
            sd = {}
            for i, nme in enumerate(names):
                if nme is None:
                    continue
                for k, v in full.items():
                    if k.startswith(nme + "."):
                        sd["%d.%s" % (i, k[len(nme) + 1:])] = v
            base_model.load_state_dict(sd)
        else:
            raise ValueError("Kinetics_pretrain doesn't exist: {}".format(kinetics_pretrain))
    if freeze_affine:
        for mod in base_model.modules():
            if mod.__class__.__name__.find('BatchNorm') != -1:
                for p in mod.parameters():
                    p.requires_grad = False
    return base_model

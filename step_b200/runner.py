"""`StepRunner` -- one CUDA graph for the whole batch step.

The reference runs ~600 PyTorch kernels per batch from Python with B*max_iter host round trips
(SURVEY.md section 3.1).  Our step is ~155 launches with no host dependency, so the entire
trunk -> (ROIAlign -> head -> tube update) x max_iter chain is captured ONCE per (B, T, H, W, N) shape into
a CUDA graph (TMA descriptors and buffer addresses are baked at capture) and replayed with a single
`cudaGraphLaunch`: launch latency and Python overhead disappear from the timed path.

    runner = StepRunner(cfg, nets, B, T_in, H, W, tubes)     # captures
    hist = runner(clips)          # clips: [B,T_in,3,H,W] fp32, CUDA or pinned host (copied in asynchronously)
or, from decoded frames (frames.py), with the input transform captured into the same graph:
    runner = StepRunner(cfg, nets, B, T_in, H, W, tubes, frames=dict(max_hw=(Hmax, Wmax), mean=..., stds=..., scale=...))
    hist = runner(frames=frames, sizes=sizes)     # frames_packed [B,T_in,Hmax,Wmax,3] uint8, sizes [B,2] (pack_frames)
`hist` is the same structure `inference()` returns (tensors are static graph outputs: copy them out
before the next call if they must survive it).
"""
import torch

from . import _lib as L
from . import engine as E
from . import frames as F
from .inference import inference_device, stage_tubes
from .postprocess import Detector


class StepRunner:
    def __init__(self, cfg, nets, B, T_in, H, W, tubes, device=None, context=False, use_graph=True, warmup=2,
                 detect=None, frames=None):
        """detect: None, or dict(conf_thresh, nms_thresh, topk[, steps]) -- the reference drivers' detection
        post-processing (test.py:156-218: confidence threshold, valid_tubes, per-class NMS, top-k) appended to the
        captured step for the listed refinement steps (default: the last one); results in `self.detections`.
        frames: None, or dict(max_hw=(Hmax, Wmax)[, mean=(0, 0, 0), stds=(1, 1, 1), scale=1]) -- the step starts from
        decoded uint8 BGR frames (frames.py): BaseTransform((W, H), mean, stds, scale) and the BGR -> RGB swap run inside the
        graph, straight into the stem's space-to-depth input on the fp16 path.  The per-clip source sizes live in a device
        table, so one capture serves any mix of sizes up to max_hw."""
        self.cfg, self.nets = cfg, nets
        self.device = device or torch.device("cuda", torch.cuda.current_device())
        self.context = context and not cfg.no_context
        self.x = torch.zeros((B, T_in, 3, H, W), dtype=torch.float32, device=self.device)
        self.frames = None
        if frames is not None:
            Hmax, Wmax = (int(v) for v in frames["max_hw"])
            self.frames = dict(size=(W, H), mean=tuple(frames.get("mean", (0, 0, 0))), stds=tuple(frames.get("stds", (1, 1, 1))),
                               scale=int(frames.get("scale", 1)))
            self.frames_buf = torch.zeros((B, T_in, Hmax, Wmax, 3), dtype=torch.uint8, device=self.device)
            self.sizes = torch.tensor([[Hmax, Wmax]] * B, dtype=torch.int32, device=self.device)
        self.flat, self.clip_of_tube, self.tubes_nums = stage_tubes(tubes, self.device)
        self.graph = None
        self.history = None
        self.detections = None
        self.detectors = {}
        if detect is not None:
            for i in detect.get("steps", [cfg.max_iter - 1]):
                self.detectors[i] = Detector(self.tubes_nums, cfg.num_classes, self.device, detect["conf_thresh"],
                                             detect["nms_thresh"], W, H, topk=detect.get("topk", 0))
        if not use_graph:
            return
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            for _ in range(warmup):  # packs weights, sets kernel attributes, warms the allocator
                self._body()
        torch.cuda.current_stream(self.device).wait_stream(side)
        torch.cuda.synchronize(self.device)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self.history = self._body()
        self.graph = g

    def _body(self):
        with torch.no_grad():
            base, fr = self.nets["base_net"], self.frames
            if fr is None:
                feat = base.forward_act(self.x)
            elif base.fp16:
                feat = base.forward_s2d(F.frames_to_s2d(self.frames_buf, self.sizes, fr["size"], fr["mean"], fr["stds"], fr["scale"]))
            else:
                F.launch(L.lib().step_frames_to_clip_f32, self.frames_buf, self.sizes, fr["size"], fr["mean"], fr["stds"],
                         fr["scale"], self.x)
                feat = base.forward_act(self.x)
            ctx_all = self.nets["context_net"].forward_act(feat) if self.context else None
            hist, _ = inference_device(self.cfg, feat, ctx_all, self.nets, self.cfg.max_iter, self.flat,
                                       self.clip_of_tube, self.tubes_nums)
            if self.detectors:
                self.detections = {i: d.run(hist[i]["pred_prob"], hist[i]["pred_loc"]) for i, d in self.detectors.items()}
        return hist

    def __call__(self, clips=None, frames=None, sizes=None):
        """clips: [B,T_in,3,H,W] fp32; or, for a runner built with frames=, frames [B,T_in,Hmax,Wmax,3] uint8 and sizes [B,2]
        (H0, W0), both from pack_frames(..., max_hw=(Hmax, Wmax)).  Host inputs are copied in asynchronously on the current
        stream: like `clips`, they must stay unchanged until that copy has run (pinned buffers of the caller's own)."""
        if frames is not None:
            if self.frames is None:
                raise RuntimeError("StepRunner: built without frames=, call it with clips")
            if clips is not None:
                raise RuntimeError("StepRunner: pass clips or frames, not both")
            if frames.shape != self.frames_buf.shape or frames.dtype != torch.uint8:
                raise ValueError("StepRunner: frames must be uint8 %s, got %s %s"
                                 % (tuple(self.frames_buf.shape), frames.dtype, tuple(frames.shape)))
            if sizes is None:
                raise ValueError("StepRunner: frames need their sizes")
            B, _, Hmax, Wmax, _ = frames.shape
            if torch.is_tensor(sizes) and not sizes.is_cuda:
                F.check_sizes(sizes, B, Hmax, Wmax)      # validates the caller's tensor; the copy reads that same tensor
                src = sizes
            else:   # a list, array or device tensor: a fresh host table the caller cannot change, copied synchronously
                src = F.check_sizes(sizes, B, Hmax, Wmax)
            if frames.data_ptr() != self.frames_buf.data_ptr():
                self.frames_buf.copy_(frames, non_blocking=True)
            self.sizes.copy_(src, non_blocking=torch.is_tensor(sizes) and not sizes.is_cuda)
        elif self.frames is not None and clips is not None:
            raise RuntimeError("StepRunner: built with frames=, call it with frames and sizes")
        elif clips is not None and clips.data_ptr() != self.x.data_ptr():
            self.x.copy_(clips, non_blocking=True)
        if self.graph is None:
            return self._body()
        self.graph.replay()
        return self.history

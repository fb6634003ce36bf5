#!/usr/bin/env python
"""bench.py -- STEP inference throughput (clips/s) on B200, BASELINE.json config 4.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic clips: I3D trunk -> (ROIAlign ->
two-branch head -> tube update) x max_iter=3, B=8 clips per GPU, T=32, 224x224, 11 proposals/clip,
fp16 storage / fp32 accumulate.  Clips are independent, so N GPUs each take their own 8 clips
(weak scaling, no data-path collective) and the fixed-shape detections are gathered once per batch
over NCCL.  Prints ONE JSON line (contract in the task brief).

value : clips/s with the batch already resident in HBM (device-timed, max over ranks).
e2e   : same call through the public API with pinned-host clips: H2D of the batch and D2H of the
        last step's scores/boxes inside the timed region.
roofline : the dominant kernel class (conv_umma_kernel, tcgen05 implicit GEMM): algorithmic conv
        FLOPs of one step (SURVEY.md section 8d: 362.06 GFLOP/clip) / the device time of exactly those
        launches replayed back-to-back, against MEASURED_PEAKS.json's sustained bf16 figure.
cpu_baseline : the oracle port (oracle/model.py, torch-CPU fp32 == the reference's arithmetic) on
        this box's host cores on a bounded sample (1 clip per timed pass).
--impl reference : the same oracle timed as the reference arm (its own CPU implementation of the path).
--dump-outputs DIR : after the K timed steps, the outputs of the last one as .npy files (see dump_outputs); the inputs
        are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALG_GFLOP_PER_CLIP = 362.06          # SURVEY.md section 8d / BASELINE.md section 3 (trunk 109.29 + 3 x 84.26)
WORKLOAD = dict(B=8, T_in=32, HW=224, N=11, max_iter=3)
# detection post-processing of the reference drivers (test.py:156-218) with the values its scripts ship:
# config.py:62-63 (conf_thresh 0.01, nms_thresh 0.4), scripts/train_step.sh:50-51 (topk 300)
DETECT = dict(conf_thresh=0.01, nms_thresh=0.4, topk=300)


CONV_CLASS_SOURCES = ("bottleneck_exit.cu", "common.cuh", "conv_halo.cu", "conv_umma.cu", "umma_ptx.cuh")


def csrc_sha():
    """Hash of the sources of the tcgen05 conv class (the kernels whose DRAM traffic profiles/r2_conv_traffic.json holds), to tie
    that capture to the build it was taken from; edits to the other kernels do not invalidate it."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "step_b200", "csrc")
    for f in CONV_CLASS_SOURCES:
        h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tflops=d.get("bf16_tflops_sustained", 1451.1), hbm=d.get("hbm_gbs", 6586.1), src="measured")
    return dict(tflops=1400.0, hbm=6650.0, src="fallback")


class ClockSampler:
    """nvidia-smi clock / throttle-reason samples during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except Exception:
                continue
            for n, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def build_nets(cfg, device):
    import step_b200
    from step_b200 import synth
    nets = {"base_net": step_b200.BaseNet(cfg), "roi_net": step_b200.ROINet(cfg.pool_mode, cfg.pool_size)}
    nets["base_net"].load_state_dict(synth.base_net_state_dict())
    for i in range(cfg.max_iter):
        h = step_b200.TwoBranchNet(cfg)
        h.load_state_dict(synth.head_state_dict(100 + i, cfg))
        nets["det_net%d" % i] = h
    for k in nets:
        nets[k] = nets[k].to(device).eval()
        if hasattr(nets[k], "set_device"):
            nets[k].set_device(device)
    return nets


def workload(rank):
    """cfg, clips [B, T_in, 3, HW, HW] (host) and proposals of the measured workload: rank r owns clips [r*B, (r+1)*B) of
    the synthetic stream (different seed per rank)."""
    from step_b200 import synth
    W = WORKLOAD
    cfg = synth.make_cfg(fp16=True, T=W["T_in"] // 4, max_iter=W["max_iter"], NUM_CHUNKS={1: 1, 2: 1, 3: 1},
                         image_size=(W["HW"], W["HW"]))
    clips = synth.make_clips(W["B"], W["T_in"], W["HW"], W["HW"], seed=1234 + rank)
    return cfg, clips, synth.make_proposals(W["B"], W["N"], cfg.T, W["HW"], W["HW"])


def run_ours(args):
    import torch
    import torch.distributed as dist
    import step_b200
    from step_b200 import _lib, engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus != world and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W = WORKLOAD
    cfg, clips_host, tubes = workload(rank)
    nets = build_nets(cfg, dev)
    B = W["B"]
    clips_host = clips_host.pin_memory()
    clips_dev = clips_host.to(dev)
    cap = min(DETECT["topk"], W["N"] * cfg.num_classes)
    # what leaves the GPU per step: the kept detections of every clip {x1,y1,x2,y2,score,class,tube,0} and their count
    out_host = {"det": torch.empty((B, cap, 8), dtype=torch.float32).pin_memory(),
                "cnt": torch.empty((B,), dtype=torch.int32).pin_memory()}
    gather = None
    if world > 1:
        gather = torch.empty((world, B, cap * 8 + 1), dtype=torch.float32, device=dev)

    def mark(msg):
        if getattr(args, "verbose", False):
            print("[bench %.1fs] %s" % (time.time() - t_start, msg), file=sys.stderr, flush=True)
    t_start = time.time()
    if getattr(args, "verbose", False):   # a stalled run prints where every Python thread is after 40 s
        import faulthandler
        faulthandler.dump_traceback_later(40, exit=False, file=sys.stderr)
    mark("setup done")
    # eager step first: packs weights, counts the launches of one step (trunk, 3 refinement steps, detection)
    eager = step_b200.StepRunner(cfg, nets, B, W["T_in"], W["HW"], W["HW"], tubes, device=dev, use_graph=False, detect=DETECT)
    eager(clips_dev)
    torch.cuda.synchronize()
    l_before = _lib.launch_count()
    hist0 = eager(clips_dev)
    torch.cuda.synchronize()
    launches_per_step = _lib.launch_count() - l_before
    # rank 0 keeps clip 0's outputs for the same-run parity check against the CPU pass of cpu_baseline
    gpu_clip0 = None
    if rank == 0 and not args.skip_cpu:
        N0 = W["N"]
        with torch.no_grad():
            cf0 = nets["base_net"](clips_dev[0:1])
        d0 = eager.detections[cfg.max_iter - 1]
        gpu_clip0 = {"feat": cf0.float().cpu(), "prob": [h["pred_prob"][:N0, 0].float().cpu() for h in hist0],
                     "loc": [h["pred_loc"][:N0].float().cpu() for h in hist0],
                     "det": d0["det"][0].cpu().numpy().copy(), "cnt": int(d0["count"][0].item())}
        del cf0
    del hist0, eager
    mark("eager step done, %d launches" % launches_per_step)
    # the public fast path: the whole step captured once into a CUDA graph (step_b200/runner.py)
    # args.inflight independent batches are kept in flight on separate streams (double buffering):
    # the H2D copy / small-grid layers of one batch overlap the other batch's kernels.
    n_run = max(1, args.inflight)
    streams = [torch.cuda.Stream(device=dev) for _ in range(n_run)]
    runners = []
    for st in streams:
        st.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(st):
            runners.append(step_b200.StepRunner(cfg, nets, B, W["T_in"], W["HW"], W["HW"], tubes, device=dev,
                                                use_graph=not args.no_graph, detect=DETECT))
    torch.cuda.synchronize()
    mark("graphs captured")
    turn = [0]

    def step(x):
        i = turn[0] % n_run
        turn[0] += 1
        cur = torch.cuda.current_stream(dev)
        streams[i].wait_stream(cur)
        with torch.cuda.stream(streams[i]):
            step.hist = runners[i](x)
            last = runners[i].detections[cfg.max_iter - 1]     # per-class NMS + top-k ran inside the captured step
        step.det = last
        step.last_stream = streams[i]
        if n_run == 1:
            cur.wait_stream(streams[i])
        if gather is not None:  # one NCCL all_gather of the fixed-shape detections per batch
            with torch.cuda.stream(streams[i]):
                det = torch.cat([last["det"].view(B, -1), last["count"].view(B, 1).float()], dim=1).contiguous()
                dist.all_gather_into_tensor(gather.view(-1, det.shape[1]), det)
        return last

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        cur = torch.cuda.current_stream(dev)
        for st in streams:      # the timed region ends when every in-flight batch has finished
            cur.wait_stream(st)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    host_out = [{"det": torch.empty_like(out_host["det"]).pin_memory(), "cnt": torch.empty_like(out_host["cnt"]).pin_memory()}
                for _ in range(n_run)]
    pending = [None] * n_run

    def e2e_step():
        # public API with host buffers: H2D of the batch (pinned, async on the batch's stream), the step, D2H of
        # the detections; the caller consumes batch i's detections before re-using its slot (one event wait).
        i = turn[0] % n_run
        if pending[i] is not None:
            pending[i].synchronize()
        last = step(clips_host)       # StepRunner copies the pinned host batch into its static input
        with torch.cuda.stream(streams[i]):
            host_out[i]["det"].copy_(last["det"], non_blocking=True)
            host_out[i]["cnt"].copy_(last["count"], non_blocking=True)
            pending[i] = streams[i].record_event()

    # clocks / throttle reasons are sampled (100 ms period) from the warm-up through both timed regions: the
    # timed regions themselves are only tens of milliseconds long
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step(clips_dev)
    mark("warm-up enqueued")
    ms = timed(lambda: step(clips_dev), args.steps)
    mark("device-resident region timed")
    if args.dump_outputs and rank == 0:     # before later steps reuse the runners' static output buffers
        dump_outputs(args.dump_outputs, step.hist, step.det, gather)
    launches = launches_per_step * args.steps

    # Insurance for the measured number: should the end-to-end region ever fail to drain (seen with programmatic dependent
    # launch on, DESIGN.md section 3.1), say so on the JSON line with the device-resident value already measured instead of
    # hanging the caller.  A stalled CUDA context cannot be torn down, hence os._exit.
    def stalled():
        if rank == 0:
            print(json.dumps({
                "metric": "clips/sec (T=32,224x224) STEP max_iter=3", "value": round(world * B * args.steps / (ms * 1e-3), 3),
                "unit": "clips/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": round(ms / args.steps, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f16", "data": "synthetic",
                "config": {"workload": "C4: full STEP inference, two_branch, 11 proposals, max_iter=3, batch 8/GPU, T=32, 224x224 "
                                       "(BASELINE.json configs[3])", "batch_per_gpu": B, "global_batch": B * world,
                           "batches_in_flight": n_run, "parallelism": "clip-parallel x%d" % world},
                "e2e": None, "gpu_launches": int(launches), "clocks": None, "roofline": None, "cpu_baseline": None,
                "stalled": "the end-to-end region did not drain within 180 s; value is the device-resident measurement"}),
                flush=True)
        os._exit(0)
    watchdog = threading.Timer(180.0, stalled)
    watchdog.daemon = True
    watchdog.start()
    for _ in range(2):
        e2e_step()
    ms_e2e = timed(e2e_step, args.steps)
    watchdog.cancel()
    mark("end-to-end region timed")
    if rank == 0 and len(sampler.rows) < 3:   # keep the GPU busy until nvidia-smi has delivered a few samples
        t_end = time.time() + 1.0
        while time.time() < t_end:
            step(clips_dev)
        torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None

    mark("timed regions done")
    # roofline of the dominant kernel class: replay exactly the conv launches of one step
    roof = None
    if rank == 0:
        rec = []
        engine.RECORDER = rec
        try:
            with torch.no_grad():
                cf0 = nets["base_net"](clips_dev)
                step_b200.inference(cfg, cf0, None, nets, cfg.max_iter, tubes, want_trajectory=False)
        finally:
            engine.RECORDER = None
        torch.cuda.synchronize()
        real_lib = _lib.lib()

        def replay():
            s = _lib.stream()
            for q, _ in rec:
                if isinstance(q, tuple):      # fused bottleneck exit (engine.bottleneck_exit)
                    _lib.check(real_lib.step_bottleneck_exit_f16(*q[1], s))
                else:
                    _lib.check(real_lib.step_conv3d_fwd(q, s))
        replay()
        # the recorded launches back to back on one stream; as a CUDA graph, so that the Python / ctypes launch path
        # (5-10 us per call, longer than the shortest kernels) does not show up as gaps between them
        replay_fn = replay
        if not args.no_graph:
            try:
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    replay()
                torch.cuda.current_stream().wait_stream(side)
                torch.cuda.synchronize()
                rg = torch.cuda.CUDAGraph()
                with torch.cuda.graph(rg):
                    replay()
                replay_fn = rg.replay
                replay_fn()
            except Exception as ex:   # keep the eager replay if capture is refused
                print("conv replay: graph capture failed (%s); timing eager launches" % ex, file=sys.stderr)
                replay_fn = replay
        mark("conv replay captured")
        ms_conv = timed_local(torch, replay_fn, max(3, args.steps))
        mark("conv replay timed")
        pk = peaks()
        # algorithmic bytes of the same launches: input + weights + output (+ residual), fp16
        alg_bytes = 0
        for q, _ in rec:
            if isinstance(q, tuple):
                alg_bytes += q[2]
                continue
            taps = q.KT * q.KH * q.KW
            alg_bytes += 2 * (q.N * q.T * q.H * q.W * q.Cin + q.Cout * taps * q.Cin +
                              q.N * q.OT * q.OH * q.OW * q.Cout * (2 if q.residual else 1))
        # DRAM bytes the same launches moved in one ncu capture (tools/gpu_profiles.sh -> profiles/r2_conv_traffic.json).
        # Only reported when that capture was taken from THIS build (the file is stamped with a hash of the kernel
        # sources); otherwise null -- a stale number is worse than none.
        traffic, traffic_src = None, None
        tp = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r2_conv_traffic.json")
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                if tj.get("csrc_sha") == csrc_sha():
                    traffic, traffic_src = tj.get("dram_bytes_per_step"), "profiles/r2_conv_traffic.json (ncu, same kernel sources %s)" % tj.get("csrc_sha")
            except Exception:
                traffic = None
        flops = ALG_GFLOP_PER_CLIP * 1e9 * B
        achieved = flops / (ms_conv / max(3, args.steps) * 1e-3) / 1e12
        roof = {"bound": "tensor", "kernel": "tcgen05 conv class: conv_umma_kernel + conv_umma_persist_kernel + conv_halo_kernel + bottleneck_exit_kernel",
                "achieved": round(achieved, 2),
                "peak": pk["tflops"], "peak_source": pk["src"] + " bf16 sustained", "unit": "TFLOP/s",
                "frac": round(achieved / pk["tflops"], 4), "traffic": traffic, "traffic_unit": "DRAM bytes per step, all conv launches (ncu)", "traffic_source": traffic_src,
                "algorithmic_bytes_per_step": int(alg_bytes),
                "launches_per_step": len(rec), "replay": "cuda graph" if replay_fn is not replay else "eager", "ms_per_step_in_kernel": round(ms_conv / max(3, args.steps), 4),
                "algorithmic_gflop_per_step": round(flops / 1e9, 1)}
        del rec

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    ms_step = ms / args.steps
    total_clips = world * B * args.steps
    cpu, parity = None, None
    if not args.skip_cpu:
        cpu, ref_out = cpu_baseline(sample_clips=1, passes=2)
        parity = parity_vs_oracle(gpu_clip0, ref_out, cfg, W)
    line = {
        "metric": "clips/sec (T=32,224x224) STEP max_iter=3", "value": round(total_clips / (ms * 1e-3), 3),
        "unit": "clips/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms_step, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16", "data": "synthetic",
        "config": {"workload": "C4: full STEP inference, two_branch, 11 proposals, max_iter=3, batch 8/GPU, "
                               "T=32, 224x224 (BASELINE.json configs[3])", "batch_per_gpu": B,
                   "global_batch": B * world, "proposals": W["N"], "l2": "inputs+activations > L2 (batch = 154 MB fp32)",
                   "a_mode": os.environ.get("STEP_B200_AMODE", "best"), "cuda_graph": not args.no_graph,
                   "batches_in_flight": n_run,
                   "parallelism": "clip-parallel x%d" % world},
        "e2e": {"value": round(total_clips / (ms_e2e * 1e-3), 3), "unit": "clips/s",
                "h2d_bytes_per_step": int(clips_host.numel() * 4),
                "d2h_bytes_per_step": int(out_host["det"].numel() * 4 + out_host["cnt"].numel() * 4)},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "parity": parity,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, hist, det, gather):
    """Writes what one step hands its caller to out_dir/<name>.npy (float32), so that two builds can be compared output
    for output on the same seeded inputs: per refinement step k the `inference` history entry (step<k>_pred_prob
    [R, classes] -- the same scores on every frame --, step<k>_pred_loc [R, T, 4] and, in temporal-predict mode, the
    neighbour boxes), then the kept detections det [B, cap, 8] and their counts [B]; with several GPUs also the
    detections gathered from every rank [ranks, B, cap * 8 + 1].  Detection rows at or past a clip's count are written
    as zeros: the step does not write them, they hold whatever an earlier step left in the buffer."""
    import numpy as np

    def blank_unwritten(d, count):   # d [clips, cap, 8], count [clips]
        d[np.arange(d.shape[1])[None, :] >= count[:, None]] = 0.0
    out = {}
    for k, h in enumerate(hist):
        out["step%d_pred_prob" % k] = h["pred_prob"][:, 0]
        for name in ("pred_loc", "pred_first_loc", "pred_last_loc"):
            if h[name] is not None:
                out["step%d_%s" % (k, name)] = h[name]
    out["det"], out["count"] = det["det"], det["count"]
    if gather is not None:
        out["gathered"] = gather
    arrays = {k: v.detach().float().cpu().numpy().copy() for k, v in out.items()}
    blank_unwritten(arrays["det"], arrays["count"])
    if gather is not None:
        g = arrays["gathered"]
        d = g[..., :-1].reshape(-1, arrays["det"].shape[1], 8)
        blank_unwritten(d, g[..., -1].reshape(-1))
        g[..., :-1] = d.reshape(g.shape[:-1] + (-1,))
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def timed_local(torch, fn, steps):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def oracle_pass(n_clips, want_outputs=False):
    """The reference's own arithmetic (torch-CPU fp32 modules restated in oracle/model.py) on n clips
    of the C4 shape: trunk + 3 refinement steps.  Returns seconds."""
    import torch
    from oracle import model as om
    from step_b200 import synth
    W = WORKLOAD
    cfg = synth.make_cfg(fp16=False, T=W["T_in"] // 4, max_iter=W["max_iter"], NUM_CHUNKS={1: 1, 2: 1, 3: 1},
                         image_size=(W["HW"], W["HW"]))
    sd = synth.base_net_state_dict()
    heads = [synth.head_state_dict(100 + i, cfg) for i in range(cfg.max_iter)]
    x = synth.make_clips(n_clips, W["T_in"], W["HW"], W["HW"])
    tubes = synth.make_proposals(n_clips, W["N"], cfg.T, W["HW"], W["HW"])
    t0 = time.perf_counter()
    with torch.no_grad():
        cf = om.base_net(x, sd)
        hist, _ = om.inference(cfg, cf, None, heads, cfg.max_iter, tubes)
    dt = time.perf_counter() - t0
    return (dt, (cf, hist)) if want_outputs else dt


def parity_vs_oracle(gpu, ref_out, cfg, W):
    """Same-run parity: the GPU outputs of clip 0 of the timed batch (fp16 tensor-core path) against the fp32 CPU pass
    that cpu_baseline just timed on the same clip (oracle/model.py == the reference's arithmetic, pinned by
    tests/golden/pipe_c4.npz).  Detection level: the reference's evaluation loop (oracle/postprocess.py, pinned to
    test.py:156-218) on the CPU outputs vs the device post-processing that ran inside the timed step."""
    import numpy as np
    from oracle import postprocess as opp
    from oracle import tubes as otubes
    cf, hist = ref_out
    N = W["N"]
    ref_feat = cf.numpy()
    d = np.abs(gpu["feat"].numpy() - ref_feat)
    out = {"clip": 0, "trunk_rel": round(float(d.max() / np.abs(ref_feat).max()), 6),
           "trunk_mean_rel": round(float(d.mean() / np.abs(ref_feat).mean()), 6)}
    s_abs, b_px = 0.0, 0.0
    for i, h in enumerate(hist):
        s_abs = max(s_abs, float(np.abs(gpu["prob"][i].numpy() - h["pred_prob"][:N, 0].numpy()).max()))
        # the CPU run has already clamped pred_loc in place (valid_tubes through the shared numpy view, utils.py:107-121)
        g_loc = otubes.valid_tubes(gpu["loc"][i].numpy().copy(), W["HW"], W["HW"])
        r_loc = otubes.valid_tubes(h["pred_loc"][:N].numpy().copy(), W["HW"], W["HW"])
        b_px = max(b_px, float(np.abs(g_loc - r_loc).max()))
    out["score_abs"], out["box_px"] = round(s_abs, 6), round(b_px, 4)
    def det_set(prob, centre_boxes, nms_thr=DETECT["nms_thresh"]):
        d = opp.detections(prob, centre_boxes, [N], DETECT["conf_thresh"], nms_thr, float(W["HW"]), float(W["HW"]),
                           topk=DETECT["topk"])[0]
        out_ = set()
        for bx, c, sc in d:   # the rows carry no tube index: recover it from the score
            out_.add((int(c), int(np.argmin(np.abs(prob[:, c] - sc)))))
        return out_

    def pair_ious(boxes):
        b = otubes.valid_tubes(boxes.reshape(-1, 1, 4).copy()).reshape(-1, 4).astype(np.float64)   # test.py:191
        area = (b[:, 2] - b[:, 0] + 1) * (b[:, 3] - b[:, 1] + 1)
        w = np.maximum(0, np.minimum(b[:, None, 2], b[None, :, 2]) - np.maximum(b[:, None, 0], b[None, :, 0]) + 1)
        h = np.maximum(0, np.minimum(b[:, None, 3], b[None, :, 3]) - np.maximum(b[:, None, 1], b[None, :, 1]) + 1)
        iou = w * h / (area[:, None] + area[None, :] - w * h)
        return iou[np.triu_indices(b.shape[0], 1)]
    last = hist[-1]
    mid = last["pred_loc"].shape[1] // 2
    # the reference's CPU run clamps history['pred_loc'] in place (valid_tubes through the shared numpy view,
    # utils.py:107-121); apply that clamp to both sides so that the two detection sets describe the same boxes
    r_prob = last["pred_prob"][:N, 0].numpy()
    r_loc = otubes.valid_tubes(last["pred_loc"][:N].numpy().copy(), W["HW"], W["HW"])
    g_prob = gpu["prob"][-1].numpy()
    g_loc_raw = gpu["loc"][-1].numpy()
    g_loc = otubes.valid_tubes(g_loc_raw.copy(), W["HW"], W["HW"])                               # same clamp as the CPU run
    ref_set, gpu_set = det_set(r_prob, r_loc[:, mid].copy()), det_set(g_prob, g_loc[:, mid].copy())
    diff = ref_set ^ gpu_set
    borderline = sum(1 for (c, t) in diff if abs(float(r_prob[t, c]) - DETECT["conf_thresh"]) < 1e-3)
    out["nms_keep_equal"] = len(diff) == 0
    out["detections_ref"], out["detections_gpu"], out["detections_differing"] = len(ref_set), len(gpu_set), len(diff)
    out["differing_within_1e-3_of_conf_thresh"] = borderline
    # Greedy NMS visits boxes in score order: where two overlapping tubes of a class score within fp16 noise of each other
    # the survivor can swap (the 11 synthetic proposals overlap heavily and 24 of 60 classes have a top-2 score gap below
    # 2e-3).  Count the differing detections that are such swaps: same class, a counterpart on the other side whose score
    # is within 5e-3 and whose box overlaps it with IoU >= nms_thresh.
    def box_iou(a, b):
        w = max(0.0, min(a[2], b[2]) - max(a[0], b[0]) + 1); h = max(0.0, min(a[3], b[3]) - max(a[1], b[1]) + 1)
        return w * h / ((a[2] - a[0] + 1) * (a[3] - a[1] + 1) + (b[2] - b[0] + 1) * (b[3] - b[1] + 1) - w * h)
    rb, gb = otubes.valid_tubes(r_loc[:, mid].reshape(-1, 1, 4).copy()).reshape(-1, 4), otubes.valid_tubes(g_loc[:, mid].reshape(-1, 1, 4).copy()).reshape(-1, 4)
    swaps = 0
    for (c, t) in diff:
        mine, other = (ref_set, gpu_set) if (c, t) in ref_set else (gpu_set, ref_set)
        sc = float(r_prob[t, c])
        if any(cc == c and abs(float(r_prob[tt, c]) - sc) <= 5e-3 and box_iou(rb[t], rb[tt]) >= DETECT["nms_thresh"] for (cc, tt) in other):
            swaps += 1
    out["differing_explained_by_near_tied_score_order"] = swaps
    # Boxes are shared by all classes, so ONE box pair whose IoU sits at the NMS threshold flips the kept set of every
    # class at once under <= 0.4 px of fp16 box noise.  Say how many such pairs this synthetic scene has, and compare the
    # sets again with the threshold moved to the middle of the widest IoU gap near it (a scene-independent statement).
    ious = np.sort(pair_ious(r_loc[:, mid].copy()))
    out["ref_box_pairs_with_iou_within_0.01_of_nms_thresh"] = int((np.abs(ious - DETECT["nms_thresh"]) < 0.01).sum())
    near = ious[(ious > DETECT["nms_thresh"] - 0.1) & (ious < DETECT["nms_thresh"] + 0.1)]
    if near.size >= 2:
        k = int(np.argmax(np.diff(near)))
        gap_thr = float(0.5 * (near[k] + near[k + 1]))
        out["gap_nms_thresh"] = round(gap_thr, 4)
        out["nms_keep_equal_at_gap_thresh"] = det_set(r_prob, r_loc[:, mid].copy(), gap_thr) == det_set(g_prob, g_loc[:, mid].copy(), gap_thr)
    # the device post-processing that ran inside the timed step == the reference loop on the same (GPU) history
    in_graph = set((int(r[5]), int(r[6])) for r in gpu["det"][:gpu["cnt"]])
    out["device_detect_equals_reference_loop"] = in_graph == det_set(g_prob, g_loc_raw[:, mid].copy())
    out["tolerance"] = "fp16 path vs fp32 reference arithmetic: trunk <= 2e-2 of max, scores <= 5e-3, boxes <= 1.5 px (tests/test_gpu_pipeline.py)"
    out["ok"] = bool(out["trunk_rel"] <= 2e-2 and s_abs <= 5e-3 and b_px <= 1.5)
    return out


_THREADS = None


def host_threads():
    """The thread count the CPU arm runs best with on this box: every core the process may use (BASELINE.md section 4),
    unless 32 threads are faster -- oneDNN convolutions stop scaling, and on shared hosts collapse, well below 128
    threads.  Both are timed once (this doubles as the warm-up) and the faster one is kept: the CPU arm gets its best
    configuration, and `cores` reports the count actually used."""
    global _THREADS
    if _THREADS is None:
        import torch
        allc = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        cands = sorted(set([allc, min(allc, 32)]), reverse=True)
        best = None
        for c in cands:
            torch.set_num_threads(c)
            oracle_pass(1)                       # oneDNN primitive creation for this thread count
            t = oracle_pass(1)
            if best is None or t < best[1]:
                best = (c, t)
        _THREADS = best[0]
        torch.set_num_threads(_THREADS)
    return _THREADS


def cpu_baseline(sample_clips=1, passes=2):
    import torch
    cores = host_threads()
    torch.set_num_threads(cores)
    ts, outs = [], None
    for _ in range(passes):
        t, outs = oracle_pass(sample_clips, want_outputs=True)
        ts.append(t)
    best = sorted(ts)[len(ts) // 2]
    return ({"value": round(sample_clips / best, 4), "unit": "clips/s", "cores": cores, "kind": "port",
             "sample": "%d clip(s) of the C4 shape (T=32, 224x224, 11 proposals, 3 steps), fp32 torch-CPU oracle, "
                       "median of %d passes after warm-up; its outputs are the parity reference of this run"
                       % (sample_clips, passes)}, outs)


def run_reference(args):
    """Reference arm: the reference's CPU implementation of the path (oracle port -- the reference's
    Python cannot travel to the GPU box; oracle/model.py is bit-identical to it in the build container)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    cores = host_threads()        # times a warm-up pass per candidate thread count and keeps the faster
    torch.set_num_threads(cores)
    t = sum(oracle_pass(1) for _ in range(args.steps))
    v = round(args.steps / t, 4)
    print(json.dumps({
        "impl": "reference", "metric": "clips/sec (T=32,224x224) STEP max_iter=3", "value": v, "unit": "clips/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": round(t / args.steps * 1e3, 2),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "C4 shape, bounded sample: 1 clip per step (T=32, 224x224, 11 proposals, max_iter=3)"},
        "cpu_baseline": {"value": v, "unit": "clips/s", "cores": cores, "kind": "port",
                         "sample": "1 clip per step, %d steps" % args.steps},
        "e2e": {"value": v, "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default: 250 for ours, ~1 s of device time; 5 for reference, one clip per step)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--skip-cpu", action="store_true", help="omit the cpu_baseline leg (profiling runs)")
    ap.add_argument("--no-graph", action="store_true", help="launch the step eagerly instead of replaying the CUDA graph")
    ap.add_argument("--inflight", type=int, default=3, help="independent batches kept in flight on separate streams")
    ap.add_argument("--verbose", action="store_true", help="phase markers on stderr (to locate a stall)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (float32; rank 0)")
    a = ap.parse_args()
    if a.steps is None:
        a.steps = 250 if a.impl == "ours" else 5
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    a.warmup = max(a.warmup, 3) if a.impl == "ours" else a.warmup
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)

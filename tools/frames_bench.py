"""Input transform from decoded frames on one B200: kernel times and the end-to-end step from uint8 frames vs fp32 clips.

    python tools/frames_bench.py --out profiles/frames_bench.json [--iters 50] [--steps 60]

Writes one JSON line.  Kernel times are CUDA-event times over `--iters` back-to-back launches after a warm-up, alternating
between two C4 source batches (2 x 177 MB, more than the 126 MB L2), so each pass reads its input from HBM.  Algorithmic
bytes are what the transform must move: source bytes read + output bytes written.  The end-to-end region is bench.py's:
three batches in flight on three streams, each step copying its pinned host batch in and its detections out; the uint8
and the fp32 arm are timed in the same process, alternating.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import step_b200  # noqa: E402
from step_b200 import _lib as L  # noqa: E402
from step_b200 import frames as F  # noqa: E402
from step_b200 import synth  # noqa: E402

B, T_IN, HW, N_PROP = 8, 32, 224, 11
H0, W0 = 360, 640
HBM_GBS = 6586.1   # bench.py's HBM figure when no measured peak is present
DETECT = dict(conf_thresh=0.01, nms_thresh=0.4, topk=300)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [v.strip() for v in q.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:   # the numbers stay valid; only the annotation is missing
        return {"name": torch.cuda.get_device_name(), "power_limit": None, "error": str(e)}


def time_kernel(fn, inputs, iters):
    for i in range(3):
        fn(inputs[i % len(inputs)])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        fn(inputs[i % len(inputs)])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters   # us


def kernel_entry(us, nbytes):
    return {"us": round(us, 2), "bytes": nbytes, "gbs": round(nbytes / (us * 1e-6) / 1e9, 1),
            "hbm_fraction": round(nbytes / (us * 1e-6) / 1e9 / HBM_GBS, 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "frames_bench.json"))
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--steps", type=int, default=60)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("frames_bench: needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    info = card()
    gen = torch.Generator().manual_seed(7)
    inputs = [torch.randint(0, 256, (B, T_IN, H0, W0, 3), dtype=torch.uint8, generator=gen).to(dev) for _ in range(2)]
    sizes = torch.tensor([[H0, W0]] * B, dtype=torch.int32, device=dev)
    size, norm = (HW, HW), dict(mean=(0, 0, 0), stds=(1, 1, 1), scale=2)   # the I3D setting (config.py:126-129)
    s2d = torch.empty((B, T_IN // 2, HW // 2, HW // 2, 32), dtype=torch.float16, device=dev)
    clips = [torch.empty((B, T_IN, 3, HW, HW), dtype=torch.float32, device=dev) for _ in range(2)]
    lib = L.lib()
    src_bytes, s2d_bytes, clip_bytes = inputs[0].numel(), s2d.numel() * 2, clips[0].numel() * 4
    k = {}
    us = time_kernel(lambda x: F.launch(lib.step_frames_to_s2d_f16, x, sizes, size, norm["mean"], norm["stds"], norm["scale"], s2d),
                     inputs, args.iters)
    k["frames_to_s2d_f16"] = kernel_entry(us, src_bytes + s2d_bytes)
    for x, c in zip(inputs, clips):
        F.launch(lib.step_frames_to_clip_f32, x, sizes, size, norm["mean"], norm["stds"], norm["scale"], c)
    idx = {id(x): i for i, x in enumerate(inputs)}
    us = time_kernel(lambda x: F.launch(lib.step_frames_to_clip_f32, x, sizes, size, norm["mean"], norm["stds"], norm["scale"],
                                        clips[idx[id(x)]]), inputs, args.iters)
    k["frames_to_clip_f32"] = kernel_entry(us, src_bytes + clip_bytes)
    us = time_kernel(lambda c: L.check(lib.step_clip_to_s2d_f16(L.ptr(c), B, T_IN, 3, HW, HW, L.ptr(s2d), 32, L.stream())),
                     clips, args.iters)
    k["clip_to_s2d_f16 (of the clip)"] = kernel_entry(us, clip_bytes + s2d_bytes)
    del inputs, clips
    torch.cuda.empty_cache()

    # end to end, three batches in flight per arm
    cfg = synth.make_cfg(fp16=True, T=T_IN // 4, max_iter=3, NUM_CHUNKS={1: 1, 2: 1, 3: 1}, image_size=(HW, HW))
    nets = {"base_net": step_b200.BaseNet(cfg), "roi_net": step_b200.ROINet(cfg.pool_mode, cfg.pool_size)}
    nets["base_net"].load_state_dict(synth.base_net_state_dict())
    for i in range(cfg.max_iter):
        h = step_b200.TwoBranchNet(cfg)
        h.load_state_dict(synth.head_state_dict(100 + i, cfg))
        nets["det_net%d" % i] = h
    nets = {n: m.to(dev).eval() for n, m in nets.items()}
    tubes = synth.make_proposals(B, N_PROP, cfg.T, HW, HW)
    frames_host, sizes_host = F.pack_frames([torch.randint(0, 256, (T_IN, H0, W0, 3), dtype=torch.uint8, generator=gen)
                                             for _ in range(B)])
    clips_host = synth.make_clips(B, T_IN, HW, HW).pin_memory()
    n_run = 3
    arms = {}
    for arm in ("frames", "clips"):
        streams = [torch.cuda.Stream(device=dev) for _ in range(n_run)]
        runners = []
        for st in streams:
            st.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(st):
                runners.append(step_b200.StepRunner(cfg, nets, B, T_IN, HW, HW, tubes, device=dev, detect=DETECT,
                                                    frames=dict(max_hw=(H0, W0), **norm) if arm == "frames" else None))
        torch.cuda.synchronize()
        cap = runners[0].detections[cfg.max_iter - 1]["det"].shape[1]
        outs = [{"det": torch.empty((B, cap, 8)).pin_memory(), "cnt": torch.empty((B,), dtype=torch.int32).pin_memory()}
                for _ in range(n_run)]
        arms[arm] = dict(streams=streams, runners=runners, outs=outs, pending=[None] * n_run, turn=0, ms=[])

    def e2e_step(a, arm):
        i = a["turn"] % n_run
        a["turn"] += 1
        if a["pending"][i] is not None:
            a["pending"][i].synchronize()
        st = a["streams"][i]
        st.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(st):
            if arm == "frames":
                a["runners"][i](frames=frames_host, sizes=sizes_host)
            else:
                a["runners"][i](clips_host)
            last = a["runners"][i].detections[cfg.max_iter - 1]
            a["outs"][i]["det"].copy_(last["det"], non_blocking=True)
            a["outs"][i]["cnt"].copy_(last["count"], non_blocking=True)
            a["pending"][i] = st.record_event()

    def timed(arm):
        a = arms[arm]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_step(a, arm)
        for st in a["streams"]:
            st.synchronize()
        return (time.perf_counter() - t0) * 1e3

    for arm in arms:
        for _ in range(4):
            e2e_step(arms[arm], arm)
    torch.cuda.synchronize()
    for _ in range(3):       # alternate the arms: other work on the host moves both alike
        for arm in ("frames", "clips"):
            arms[arm]["ms"].append(timed(arm))
    e2e = {}
    for arm, h2d in (("frames", frames_host.numel() + sizes_host.numel() * 4), ("clips", clips_host.numel() * 4)):
        ms = arms[arm]["ms"]
        e2e["from_" + arm] = {"clips_per_s": [round(B * args.steps / (m * 1e-3), 1) for m in ms],
                              "ms_per_step": [round(m / args.steps, 3) for m in ms], "h2d_bytes_per_step": h2d}
    res = {"tool": "frames_bench", "card": info, "hbm_gbs_assumed": HBM_GBS,
           "workload": "C4 batch: %d clips x %d frames of %dx%d uint8 BGR -> %dx%d, scale 2 (I3D)" % (B, T_IN, H0, W0, HW, HW),
           "kernels": k, "kernel_iters": args.iters, "kernel_inputs": "two source batches alternated (2 x %d MB)" % (src_bytes >> 20),
           "e2e": e2e, "e2e_steps": args.steps, "batches_in_flight": n_run}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(res) + "\n")
    print(json.dumps(res))


if __name__ == "__main__":
    main()

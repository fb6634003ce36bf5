"""CPU, world_size 2, gloo: the N>1 host logic of bench.py's clip-parallel mode -- each rank owns a
disjoint batch, fixed-shape detections are all-gathered once per batch, rank order is preserved and the
max-over-ranks timing reduction works.  (No GPU kernels are called here.)"""
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from step_b200 import synth
    B, cap = 2, 5
    # rank r owns clips [r*B, (r+1)*B): per-rank seed as in bench.py; what is gathered has the layout of bench.py's
    # step(): per clip the compact detections [cap, 8] of step_detect_f32 flattened, then the count (stand-in values here:
    # the kernels need a GPU; tests/test_gpu_multi.py checks the real thing on 2 GPUs)
    clips = synth.make_clips(B, 4, 8, 8, seed=1234 + rank)
    det = torch.full((B, cap * 8 + 1), float(rank)) + clips.mean()
    gather = torch.empty((world, B, cap * 8 + 1))
    dist.all_gather_into_tensor(gather.view(-1, cap * 8 + 1), det)
    ms = torch.tensor([10.0 + rank])
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    dist.barrier()
    if rank == 0:
        torch.save({"gather": gather, "ms": ms}, out)
    dist.destroy_process_group()


def test_clip_parallel_gather_two_ranks(tmp_path):
    out = str(tmp_path / "r0.pt")
    mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    r = torch.load(out)
    from step_b200 import synth
    for rank in range(2):
        exp = float(rank) + synth.make_clips(2, 4, 8, 8, seed=1234 + rank).mean()
        assert torch.allclose(r["gather"][rank], torch.full((2, 41), float(exp)))
    assert float(r["ms"]) == 11.0


def test_bench_dump_outputs_writes_what_the_step_returns(tmp_path):
    """bench.py --dump-outputs: every array of the step's history and detections as float32 .npy, fp16 scores widened,
    the per-frame copies of the scores (an expand view) stored once, absent neighbour boxes skipped, detection rows past a
    clip's count (never written by the step) zeroed, also in the detections gathered from every rank."""
    import importlib.util
    import numpy as np
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    g = torch.Generator().manual_seed(0)
    prob = torch.rand(6, 1, 60, generator=g).half().expand(-1, 4, -1)
    loc = torch.rand(6, 4, 4, generator=g)
    hist = [{"pred_prob": prob, "pred_loc": loc, "pred_first_loc": loc + 1, "pred_last_loc": loc + 2, "tubes_nums": [3, 3]},
            {"pred_prob": prob, "pred_loc": loc, "pred_first_loc": None, "pred_last_loc": None, "tubes_nums": [3, 3]}]
    det = {"det": torch.rand(2, 5, 8, generator=g), "count": torch.tensor([5, 2], dtype=torch.int32)}
    # two ranks' [clip, cap * 8 + 1] rows as bench.py gathers them: rank 1 kept 1 and 0 detections
    gather = torch.stack([torch.cat([det["det"].view(2, -1), det["count"].view(2, 1).float()], 1),
                          torch.cat([torch.rand(2, 40, generator=g), torch.tensor([[1.0], [0.0]])], 1)])
    before = {k: v.clone() for k, v in det.items()}
    bench.dump_outputs(str(tmp_path / "out"), hist, det, gather)
    names = sorted(p.name for p in (tmp_path / "out").iterdir())
    assert names == ["count.npy", "det.npy", "gathered.npy", "step0_pred_first_loc.npy", "step0_pred_last_loc.npy",
                     "step0_pred_loc.npy", "step0_pred_prob.npy", "step1_pred_loc.npy", "step1_pred_prob.npy"]
    got = {n[:-4]: np.load(str(tmp_path / "out" / n)) for n in names}
    assert all(a.dtype == np.float32 for a in got.values())
    assert np.array_equal(got["step1_pred_prob"], prob[:, 0].float().numpy())
    assert np.array_equal(got["step0_pred_last_loc"], (loc + 2).numpy())
    kept = before["det"].numpy().copy()
    kept[1, 2:] = 0.0
    assert np.array_equal(got["det"], kept) and got["count"].tolist() == [5.0, 2.0]
    assert all(torch.equal(det[k], before[k]) for k in det)                     # the caller's tensors are left alone
    exp = gather.numpy().copy()
    exp[0, 1, 16:40] = 0.0
    exp[1, 0, 8:40] = 0.0
    exp[1, 1, :40] = 0.0
    assert np.array_equal(got["gathered"], exp)


def test_reference_arm_under_torchrun_prints_one_line():
    """`bench.py --impl reference` launched the way the driver launches N > 1 (torchrun, one process per GPU):
    rank 0 alone runs the reference arithmetic on the host cores and prints ONE JSON line, the other ranks exit 0."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2",
           "--steps", "1", "--warmup", "0"]
    r = subprocess.run(cmd, cwd=root, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["value"] > 0 and d["unit"] == "clips/s"
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["e2e"]["h2d_bytes_per_step"] == 0


def test_reference_arm_times_exactly_the_steps_asked_for():
    """`--steps` sets the number of timed passes of the reference arm too; 6 is above its default of 5."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "6", "--warmup", "0"],
                       cwd=root, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 6 and d["cpu_baseline"]["sample"] == "1 clip per step, 6 steps"

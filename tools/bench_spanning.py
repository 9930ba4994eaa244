"""Untiled S3 (doTile 0: regions cross the slab cuts and are solved with the shared-region reduction) on 1, 2, 4 and 8 GPUs.

One process per GPU, as bench.py runs N > 1.  Per GPU count: steps/s (CUDA events on the solver's stream around K steps that end in a
device synchronise, then a barrier; the slowest rank counts), microseconds per CG iteration (ps_time_kernel "cg_iteration"), the
shared-region count, and iterations plus a strided velocity sample compared with the 1-GPU run.  Then one run with PS_TRACE at the
largest GPU count: the CUDA-event timeline of one CG iteration, whose "shared regions" entry is the per-iteration cost of
the reduction.  Writes profiles/<out>.json (trace lines included) with the card name and power limit read in the same call.

usage: python tools/bench_spanning.py [--n 256] [--gpus 1,2,4,8] [--steps 3] [--warmup 1] [--out spanning_s3_256_notile]
(the worker mode, --worker, is what the parent starts once per rank)
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
SAMPLE_STRIDE = 97


def worker(a):
    import torch
    import torch.distributed as dist
    from polystokes_b200 import PolyStokesSolver, scenes, PS_SUCCESS
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
    sc = scenes.scene_s3(a.n, doTile=0)
    s = PolyStokesSolver.from_scene(sc, device=rank)
    zlo, zhi = 0, sc.nz
    if world > 1:
        _, _, zlo, zhi, _ = s.init_distributed()
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    d_in = [dev(sc.surface), dev(sc.collision), dev(sc.viscosity)]
    d_vel, d_cvel = [dev(v) for v in sc.vel], [dev(v) for v in sc.colvel]
    d_out, d_valid = [v.clone() for v in d_vel], [torch.zeros_like(v) for v in d_vel]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def step():
        rc = s.step(d_in[0], d_in[1], d_in[2], d_vel, d_cvel, d_out, d_valid)
        if rc != PS_SUCCESS:
            raise SystemExit(f"bench_spanning: solver returned {rc}")
    for _ in range(max(1, a.warmup)):
        step()
    res = {}
    if not a.trace:
        barrier()
        s.timer_start()
        for _ in range(a.steps):
            step()
        ms = s.timer_stop()
        barrier()
        iters = s.count("iterations")
        cg_ms = s.time_kernel("cg_iteration", 20)
        # strided velocity sample of the own slab (z is the slowest axis); summed over the ranks it is the full sample
        sample = []
        for v in d_out:
            h = v.cpu().numpy()
            top = h.shape[0] if zhi >= sc.nz else zhi
            idx = np.arange(0, h.size, SAMPLE_STRIDE)
            z = idx // (h.shape[1] * h.shape[2])
            sample.append(np.where((z >= zlo) & (z < top), h.reshape(-1)[idx], 0.0).astype(np.float64))
        t = torch.tensor(np.concatenate(sample + [np.array([ms, cg_ms])]), device="cuda", dtype=torch.float64)
        if world > 1:
            mx = t[-2:].clone()
            dist.all_reduce(t)
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            t[-2:] = mx
        t = t.cpu().numpy()
        res = dict(gpus=world, steps=a.steps, ms_per_step=float(t[-2]) / a.steps, steps_per_s=a.steps / (float(t[-2]) * 1e-3), us_per_cg_iteration=float(t[-1]) * 1e3,
                   iterations=int(iters), sharedRegions=int(s.count("sharedRegions")), regionCount=int(s.count("regionCount")), nSystemSize=int(s.count("nSystemSize")),
                   stage_ms={k: round(v, 3) for k, v in s.stage_ms().items()}, result=int(s.stats.result))
        if rank == 0:
            np.save(os.path.join(a.tmp, f"sample_{world}.npy"), t[:-2])
            with open(os.path.join(a.tmp, f"res_{world}.json"), "w") as f:
                json.dump(res, f)
    s.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def launch(a, world, trace=False):
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(29400 + world + (50 if trace else 0)), WORLD_SIZE=str(world))
    if trace:
        env["PS_TRACE"] = "5"
    args = [sys.executable, os.path.abspath(__file__), "--worker", "--n", str(a.n), "--steps", str(a.steps), "--warmup", str(a.warmup), "--tmp", a.tmp] + (["--trace"] if trace else [])
    procs = [subprocess.Popen(args, env=dict(env, RANK=str(r), LOCAL_RANK=str(r)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(world)]
    outs = [p.communicate(timeout=1800)[0] for p in procs]
    bad = [f"rank {r}: exit {p.returncode}\n{o[-3000:]}" for r, (p, o) in enumerate(zip(procs, outs)) if p.returncode != 0]
    if bad:
        raise SystemExit("\n".join(bad))
    return outs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--trace", action="store_true")
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--gpus", default="1,2,4,8")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--tmp", default=None)
    ap.add_argument("--out", default="spanning_s3_256_notile")
    a = ap.parse_args()
    if a.worker:
        return worker(a)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_spanning: no CUDA device")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    counts = [g for g in (int(x) for x in a.gpus.split(",")) if g <= torch.cuda.device_count() and 16 * g <= a.n]
    a.tmp = tempfile.mkdtemp(prefix="bench_spanning_")
    runs = []
    for g in counts:
        launch(a, g)
        with open(os.path.join(a.tmp, f"res_{g}.json")) as f:
            runs.append(json.load(f))
    base = np.load(os.path.join(a.tmp, f"sample_{counts[0]}.npy"))
    scale = max(float(np.abs(base).max()), 1e-30)
    for r in runs:
        smp = np.load(os.path.join(a.tmp, f"sample_{r['gpus']}.npy"))
        r["velocity_sample_max_rel_diff_vs_first"] = float(np.abs(smp - base).max()) / scale
        r["iterations_vs_first"] = r["iterations"] - runs[0]["iterations"]
    trace = launch(a, counts[-1], trace=True) if counts[-1] > 1 else []
    lines = [l for o in trace for l in o.splitlines() if l.startswith("[ps trace")]
    os.makedirs(os.path.join(ROOT, "profiles"), exist_ok=True)
    out = dict(scene=f"S3 {a.n}^3 doTile=0", card=card, timing="CUDA events on the solver stream around K synchronised ps_step calls (device arrays), slowest rank; "
                                                                     "us per CG iteration from ps_time_kernel('cg_iteration', 20)",
               runs=runs, trace_gpus=counts[-1], trace=lines)
    path = os.path.join(ROOT, "profiles", a.out + ".json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()

"""Even against work-balanced z cuts (ps_rebalance) on several GPUs, both arms in the same call, alternating.

Configurations: S5 512x256x256 tile 16 (BASELINE.json configs[4]) and S4 384^3 (configs[3]) at 2 / 4 / 8 GPUs with one process per GPU,
S5 at 8 GPUs behind one ps_create_multi handle, and S3 256^3 at 8 GPUs as the control (its parity against the committed 256^3 digest,
tests/golden/fullsize_S3.json, as bench.py checks it).  Per configuration: a warm-up step on the even cuts, ps_rebalance (timed), the
first step on the new cuts (timed: the re-layout), then `--reps` rounds of [even, balanced]: ps_set_partition, one untimed step, `--steps`
timed steps (CUDA events on the solver stream, slowest rank) and ps_time_kernel("cg_iteration", 20) (slowest rank).  Reported per arm:
steps/s (median of the rounds), us per CG iteration, the cuts, the per-slab sums of unitLoad.  Writes profiles/<out>.json with the card
name and power limit read in the same call.

usage: python tools/bench_partition.py [--only S5:2,S4:4,...] [--steps 3] [--reps 3] [--out partition_balance]
(--worker is what the parent starts once per rank)
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
CONFIGS = [("S5", 2), ("S5", 4), ("S5", 8), ("S4", 2), ("S4", 4), ("S4", 8), ("S5multi", 8), ("S3", 8)]


def scene(name):
    from polystokes_b200 import scenes
    if name.startswith("S5"):
        return scenes.scene_s5(1.0, tileSize=16)
    return scenes.scene_s4(384) if name == "S4" else scenes.scene_s3(256)


def slab_loads(load, cuts, unit):
    return [float(sum(load[c0 // unit:-(-c1 // unit)])) for c0, c1 in zip(cuts[:-1], cuts[1:])]


def measure(s, sc, world, step, barrier, reduce_max, a):
    """The two arms on one handle; returns the result dict (identical on every rank)."""
    from polystokes_b200 import PS_SUCCESS
    step()
    even = s.partition()[4]
    load = [float(v) for v in s.vector("unitLoad")]
    unit = 32 if sc.params.get("tileSize") == 32 else 16
    barrier()
    t0 = time.perf_counter()
    rc, balanced = s.rebalance()
    t_rebalance = reduce_max(time.perf_counter() - t0)
    barrier()
    s.timer_start()
    step()
    t_first = reduce_max(s.timer_stop())
    arms = {"even": {"cuts": even, "steps_per_s": [], "us_per_cg_iteration": []}, "balanced": {"cuts": balanced, "steps_per_s": [], "us_per_cg_iteration": []}}
    for _ in range(a.reps):
        for name in ("even", "balanced"):
            arm = arms[name]
            assert s.set_partition(arm["cuts"]) == PS_SUCCESS
            step()
            barrier()
            s.timer_start()
            for _ in range(a.steps):
                step()
            ms = reduce_max(s.timer_stop())
            barrier()
            arm["steps_per_s"].append(a.steps / (ms * 1e-3))
            arm["us_per_cg_iteration"].append(reduce_max(s.time_kernel("cg_iteration", 20)) * 1e3)
            arm["iterations"] = s.count("iterations")
    for arm in arms.values():
        arm["slab_unitLoad"] = slab_loads(load, arm["cuts"], unit)
        arm["max_slab_unitLoad"] = max(arm["slab_unitLoad"])
        arm["steps_per_s_median"] = float(np.median(arm["steps_per_s"]))
        arm["us_per_cg_iteration_median"] = float(np.median(arm["us_per_cg_iteration"]))
    return dict(gpus=world, rebalance_rc=int(rc), rebalance_s=t_rebalance, first_step_after_move_ms=t_first, unit=unit,
                unitLoad=load, arms=arms, gain_steps_per_s=arms["balanced"]["steps_per_s_median"] / arms["even"]["steps_per_s_median"],
                gain_cg_iteration=arms["even"]["us_per_cg_iteration_median"] / arms["balanced"]["us_per_cg_iteration_median"])


def s3_parity(s, sc, d_out, d_valid, zlo, zhi, dist):
    """bench.py's check of the 256^3 step against tests/golden/fullsize_S3.json (the slabs summed into full fields first)."""
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import make_fullsize
    outs, vals = [t.clone() for t in d_out], [t.clone() for t in d_valid]
    for t in outs + vals:
        top = zhi if zhi < sc.nz else t.shape[0]
        t[:zlo] = 0
        t[top:] = 0
        if dist is not None:
            dist.all_reduce(t)
    with open(os.path.join(ROOT, "tests", "golden", "fullsize_S3.json")) as f:
        gold = json.load(f)
    got = make_fullsize.velocity_sample([t.cpu().numpy() for t in outs], [t.cpu().numpy() for t in vals])
    bad = [k for k, v in gold["counts"].items() if s.count(k) != v]
    worst = max(float(np.abs(np.array(gold[f"vel{ax}_sample"]) - np.array(got[f"vel{ax}_sample"])).max()) / gold[f"vel{ax}_absmax"] for ax in range(3))
    its = s.count("iterations")
    ok = (not bad and abs(its - gold["iterations"]) <= max(2, gold["iterations"] // 100) and worst <= 10 * sc.params["tolerance"]
          and all(got[f"valid{ax}"] == gold[f"valid{ax}"] for ax in range(3)))
    return dict(ok=bool(ok), counts_differ=bad, iterations=its, gold_iterations=gold["iterations"], velocity_sample_max_rel=worst)


def worker(a):
    import torch
    from polystokes_b200 import PolyStokesSolver, PS_SUCCESS
    sc = scene(a.scene)
    multi = a.scene == "S5multi"
    if multi:
        world, dist = a.gpus, None
        s = PolyStokesSolver.from_scene(sc, devices=list(range(world)))
        arrays = [sc.surface, sc.collision, sc.viscosity, sc.vel, sc.colvel, [v.copy() for v in sc.vel], [np.zeros_like(v) for v in sc.vel]]
        step_args = arrays
        rank = 0
    else:
        import torch.distributed as dist
        rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
        s = PolyStokesSolver.from_scene(sc, device=rank)
        s.init_distributed()
        dev = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
        d_vel = [dev(v) for v in sc.vel]
        step_args = [dev(sc.surface), dev(sc.collision), dev(sc.viscosity), d_vel, [dev(v) for v in sc.colvel], [v.clone() for v in d_vel],
                     [torch.zeros_like(v) for v in d_vel]]

    def step():
        rc = s.step(*step_args)
        if rc != PS_SUCCESS:
            raise SystemExit(f"bench_partition: solver returned {rc}")

    def barrier():
        if dist is not None:
            torch.cuda.synchronize()
            dist.barrier()

    def reduce_max(v):
        if dist is None:
            return float(v)
        t = torch.tensor([float(v)], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    res = measure(s, sc, world, step, barrier, reduce_max, a)
    res["config"] = a.scene + (" (ps_create_multi)" if multi else " (one process per GPU)")
    if a.scene == "S3":
        _, _, zlo, zhi, _ = s.partition()
        res["parity_balanced_cuts"] = s3_parity(s, sc, step_args[5], step_args[6], zlo, zhi, dist)
    if rank == 0:
        with open(os.path.join(a.tmp, f"{a.scene}_{world}.json"), "w") as f:
            json.dump(res, f)
    s.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def launch(a, name, world):
    args = [sys.executable, os.path.abspath(__file__), "--worker", "--scene", name, "--gpus", str(world), "--steps", str(a.steps), "--reps", str(a.reps), "--tmp", a.tmp]
    n = 1 if name == "S5multi" else world
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(29500 + 10 * world + len(name)), WORLD_SIZE=str(world))
    procs = [subprocess.Popen(args, env=dict(env, RANK=str(r), LOCAL_RANK=str(r)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(n)]
    outs = [p.communicate(timeout=1800)[0] for p in procs]
    bad = [f"rank {r}: exit {p.returncode}\n{o[-3000:]}" for r, (p, o) in enumerate(zip(procs, outs)) if p.returncode != 0]
    if bad:
        return {"config": name, "gpus": world, "error": "\n".join(bad)[-4000:]}
    with open(os.path.join(a.tmp, f"{name}_{world}.json")) as f:
        return json.load(f)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--scene", default="S5")
    ap.add_argument("--gpus", type=int, default=2)
    ap.add_argument("--only", default="", help="comma list of scene:gpus (scene S5, S4, S5multi, S3)")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--tmp", default=None)
    ap.add_argument("--out", default="partition_balance")
    a = ap.parse_args()
    if a.worker:
        return worker(a)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_partition: no CUDA device")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    todo = [(c.split(":")[0], int(c.split(":")[1])) for c in a.only.split(",")] if a.only else CONFIGS
    todo = [(n, g) for n, g in todo if g <= torch.cuda.device_count()]
    if not todo:
        raise SystemExit(f"bench_partition: every configuration needs more GPUs than the {torch.cuda.device_count()} present")
    a.tmp = tempfile.mkdtemp(prefix="bench_partition_")
    runs = []
    for name, g in todo:
        r = launch(a, name, g)
        runs.append(r)
        print(json.dumps({k: v for k, v in r.items() if k not in ("unitLoad", "arms")} | ({"cuts": {n: r["arms"][n]["cuts"] for n in r["arms"]},
              "steps_per_s": {n: r["arms"][n]["steps_per_s_median"] for n in r["arms"]}} if "arms" in r else {})), flush=True)
    out = dict(card=card, timing="CUDA events on the solver stream around --steps synchronised ps_step calls (device arrays; host arrays on the "
                                  "ps_create_multi handle), slowest rank, median of --reps alternating rounds; us per CG iteration from "
                                  "ps_time_kernel('cg_iteration', 20), slowest rank", steps=a.steps, reps=a.reps, runs=runs)
    os.makedirs(os.path.join(ROOT, "profiles"), exist_ok=True)
    with open(os.path.join(ROOT, "profiles", a.out + ".json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()

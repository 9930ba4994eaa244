"""Per-iteration timing of the slab-decomposed CG under torchrun (one process per GPU): cg_iteration / pass1 / pass2 /
apply on this rank's slab of S3.  Run once per setting of PS_COMM (the library reads it once)."""
import argparse, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist
from polystokes_b200 import PolyStokesSolver, scenes

ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, default=256)
ap.add_argument("--reps", type=int, default=200)
ap.add_argument("--tag", default="")
a = ap.parse_args()
rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
if world > 1:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
sc = scenes.scene_s3(a.n)
s = PolyStokesSolver.from_scene(sc, device=local)
if world > 1:
    s.init_distributed()
d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
s.setup(d(sc.surface), d(sc.collision), d(sc.viscosity), [d(v) for v in sc.vel], [d(v) for v in sc.colvel])
res = {}
for k in ("cg_iteration", "pass1", "pass2", "apply"):
    s.time_kernel(k, 20)
    res[k] = s.time_kernel(k, a.reps)
t = torch.tensor([res[k] for k in res], device="cuda", dtype=torch.float64)
if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
if rank == 0:
    env = {k: os.environ.get(k) for k in ("PS_COMM",) if os.environ.get(k)}
    print(f"[dist_probe {a.tag}] world={world} peer={s.count('peerTransport')} env={env} max over ranks, us: " +
          "  ".join(f"{k} {float(v)*1e3:.1f}" for k, v in zip(res, t.tolist())), flush=True)
if world > 1:
    dist.destroy_process_group()

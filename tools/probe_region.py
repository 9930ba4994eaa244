"""Probe of the reduced term on the GPU box: one setup of S3, then the region kernel alone, pass 1 + regions and a CG iteration."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from polystokes_b200 import PolyStokesSolver, scenes
n = int(sys.argv[1]) if len(sys.argv) > 1 else 256
sc = scenes.scene_s3(n)
d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
s = PolyStokesSolver.from_scene(sc)
s.setup(d(sc.surface), d(sc.collision), d(sc.viscosity), [d(v) for v in sc.vel], [d(v) for v in sc.colvel])
tag = f"regionPath={s.count('regionPath')}"
print(tag, " ".join(f"{k} {s.time_kernel(k, 40) * 1e3:.1f} us" for k in ("reduced", "pass1", "cg_iteration")), flush=True)

"""Child process of tests/test_cg_iterates.py: the CG loop stopped after exactly k iterations (ps_time_kernel("cg_iteration", k)) on
several ranks.

  python cg_iterates_worker.py <scene> <outdir> <k>...               one rank of a gloo job on the host-emulation twin (RANK /
                                                                     WORLD_SIZE / MASTER_* in the env); writes <outdir>/rank<r>.npz
  python cg_iterates_worker.py --devices N <scene> <outdir> <k>...   one ps_create_multi handle on N GPUs and a single-GPU handle;
                                                                     writes <outdir>/multi.npz

b and Ax (A of test_cg_iterates.probe_x), and per k: x<k> -- this rank's share of each vector, the global vector on a multi handle --
xmag<k>, err<k> (solveError) and its<k> (iterations); on a multi handle the same of the single-GPU handle, prefixed one_.
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from polystokes_b200 import PolyStokesSolver, scenes  # noqa: E402

# nz >= 16 x ranks; tile 8 cuts at multiples of 16
SCENES = {
    "blob48_tile8": lambda: scenes.blob_scene(48, seed=21, tile=8, pad=1),
    "box48_uniform": lambda: scenes.box_scene(48, doReduced=0),
}


def iterates(s, ks, out, prefix=""):
    out[prefix + "b"] = s.vector("b")
    out[prefix + "Ax"] = s.apply(np.random.default_rng(7).standard_normal(s.count("nSystemSize")))     # test_cg_iterates.probe_x
    for k in ks:
        s.time_kernel("cg_iteration", k)
        out[f"{prefix}x{k}"] = s.vector("solution")
        out[f"{prefix}xmag{k}"] = s.real("xmag")
        out[f"{prefix}err{k}"] = s.real("solveError")
        out[f"{prefix}its{k}"] = s.count("iterations")


def main(argv):
    ap = argparse.ArgumentParser()
    ap.add_argument("--devices", type=int, default=0)
    ap.add_argument("scene", choices=list(SCENES))
    ap.add_argument("outdir")
    ap.add_argument("ks", type=int, nargs="+")
    a = ap.parse_args(argv)
    sc = SCENES[a.scene]()
    out = {}
    if a.devices:
        many = PolyStokesSolver.from_scene(sc, devices=list(range(a.devices)))
        many.setup_scene(sc)
        out["nranks"] = many.partition()[1]
        iterates(many, a.ks, out)
        many.close()
        one = PolyStokesSolver.from_scene(sc)
        one.setup_scene(sc)
        iterates(one, a.ks, out, "one_")
        one.close()
        np.savez(os.path.join(a.outdir, "multi.npz"), **out)
        return
    import torch.distributed as dist
    import parity
    from dist_worker import attach_gloo
    dist.init_process_group("gloo")
    s = PolyStokesSolver.from_scene(sc, lib_path=parity.EMUL_LIB)
    attach_gloo(s)
    rank, out["nranks"] = s.partition()[:2]
    s.setup_scene(sc)
    iterates(s, a.ks, out)
    np.savez(os.path.join(a.outdir, f"rank{rank}.npz"), **out)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main(sys.argv[1:])

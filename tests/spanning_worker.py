"""Worker of tests/test_distributed_spanning_emul.py and tests/test_gpu_spanning_regions.py: one rank of a slab-decomposed
step on a scene whose reduced regions cross the cuts (tests/spanning_cases.py).  Writes <outdir>/rank<k>.npz with what
tests/dist_worker.py writes (parity.check_distributed merges it) plus the shared-region count, how the shared moments were summed
and which kernels carried the reduced term (regionPath).  For a SWITCH case the handle
first steps the scene with other tiling parameters, then ps_set_params switches it to the case's own.
Usage: python spanning_worker.py <case> <outdir> [gpu]   (RANK / WORLD_SIZE / MASTER_* in the env)
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import parity  # noqa: E402
import spanning_cases  # noqa: E402
from dist_worker import REGION_VECTORS, applies_after_step, applies_before_step, attach_gloo  # noqa: E402


def set_params(s, **kw):
    for k, v in kw.items():
        setattr(s._P, k, v)
    assert s.lib.ps_set_params(s.h, s._P) == 1, s.last_error()


def main():
    case, outdir = sys.argv[1], sys.argv[2]
    gpu = len(sys.argv) > 3 and sys.argv[3] == "gpu"
    spanning_cases.register()
    from polystokes_b200 import PolyStokesSolver
    sc, ov = parity.DIST_CASES[case]()
    first = spanning_cases.SWITCH.get(case)
    if gpu:
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        s = PolyStokesSolver.from_scene(sc, device=local, **dict(ov, **(first or {})))
        s.init_distributed()
    else:
        dist.init_process_group("gloo")
        s = PolyStokesSolver.from_scene(sc, lib_path=parity.EMUL_LIB, **dict(ov, **(first or {})))
        attach_gloo(s)
    out = {}
    if first:
        # the other tiling first: other cuts (lcm(16, tileSize)), no shared region; then back to the case's parameters
        out["first_cuts"] = np.array(s.partition()[4])
        rc0, vel0, _ = s.step_scene(sc)
        out["first_rc"] = rc0
        out["first_shared"] = s.count("sharedRegions")
        set_params(s, **{k: sc.params[k] for k in first})
    rank, n, zlo, zhi, cuts = s.partition()
    s.setup_scene(sc)
    out.update(rank=rank, nranks=n, zlo=zlo, zhi=zhi, cuts=np.array(cuts), peer=s.count("peerTransport") if gpu else 0, local=s.count("slabLocal"),
               shared=s.count("sharedRegions"))
    for k in parity.COUNTS + ["maxRegionRows", "regionPath", "peerSharedCap"]:
        out["count_" + k] = s.count(k)
    for slot in range(7):
        out[f"labels{slot}"] = s.index_field(0, slot)
        out[f"active{slot}"] = s.index_field(1, slot)
        out[f"reduced{slot}"] = s.index_field(2, slot)
    for v in REGION_VECTORS:
        out["vec_" + v] = s.vector(v)
    state = applies_before_step(s, out, outdir)
    rc, vel, valid = s.step_scene(sc)
    out["rc"] = rc
    out["peerExchanges"] = s.count("sharedPeerExchanges")      # how the shared-region moments of this step were summed
    out["commExchanges"] = s.count("sharedCommExchanges")
    out["iterations"] = s.count("iterations")
    out["usedBiCGStab"] = s.count("usedBiCGStab")
    out["solution"] = s.vector("solution")
    out["velSolution"] = s.vector("velSolution")
    for a in range(3):
        out[f"vel{a}"] = vel[a]
        out[f"valid{a}"] = valid[a]
    applies_after_step(s, out, state)
    rc2, vel2, _ = s.step_scene(sc)
    out["repeat_ok"] = bool(rc2 == rc and all(np.array_equal(vel[a], vel2[a]) for a in range(3)))
    if first:
        # and back: the tiled step of the first call again, bit for bit
        set_params(s, **first)
        rc3, vel3, _ = s.step_scene(sc)
        out["back_ok"] = bool(rc3 == rc0 and s.count("sharedRegions") == 0 and all(np.array_equal(vel0[a], vel3[a]) for a in range(3)))
    np.savez(os.path.join(outdir, f"rank{rank}.npz"), **out)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()

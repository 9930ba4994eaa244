"""Worker of tests/test_partition_emul.py (and tests/test_gpu_partition.py): one rank of a job that moves the z cuts of a decomposed handle.

  python partition_worker.py <mode> <case> <outdir> [cuts] [gpu]     (RANK / WORLD_SIZE / MASTER_* in the env)

The ranks drive the host-emulation twin through torch.distributed / gloo, or with "gpu" the CUDA library (NCCL, one GPU per rank).
Modes:
  rebalance   setup, the unit table (unitLoad, unitCounts, cg_iteration bytes), ps_rebalance twice, then the record of
              tests/dist_worker.py on the new cuts (parity.check_distributed)
  set         ps_set_partition(cuts), the record on those cuts, the broken-rule calls (each must give PS_INVALID and leave the cuts),
              a step on the kept cuts, NULL (the even cuts), ps_set_params with a new dt (cuts kept) and with tileSize 32 (even cuts)
  restart     ps_set_partition(cuts) on a scene whose boundary fix-up has work: the slab-local attempt restarts replicated, the cuts stay
  move        a scene at the bottom of z, then at the top, on one handle that rebalances after each first step; every step against a
              fresh handle given the same cuts
  steps       (GPU) a step, ps_rebalance, a step on the new cuts: counts, index fields, iterations, velocity, unitLoad
Each rank writes <outdir>/rank<k>.npz.  Without RANK in the env, "steps" runs ONE process: a single-GPU handle (<ndev> = 1) or a
ps_create_multi handle over <ndev> GPUs, and writes <outdir>/single.npz or <outdir>/multi.npz.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import parity  # noqa: E402
import spanning_cases  # noqa: E402
from polystokes_b200 import scenes  # noqa: E402


def shifted_blob(nxy, nzb, nz, z0, seed=13, tile=16, pad=2, **ov):
    """A tiled blob scene of nzb layers placed at layers [z0, z0 + nzb) of a taller grid; the other layers hold air only, so the even
    cuts leave slabs (nearly) empty."""
    b = scenes.blob_scene((nxy, nxy, nzb), seed=seed, tile=tile, pad=pad, **ov)
    big = lambda a, fill, extra=0: np.full((nz + extra,) + a.shape[1:], fill, dtype=np.float32)
    sc = scenes.Scene(f"blob{nxy}x{nxy}x{nzb}_at{z0}_of{nz}", nxy, nxy, nz, b.dx, b.dt, b.density, big(b.surface, 1.0), big(b.collision, 1.0),
                      big(b.viscosity, 50.0), [], [], dict(b.params))
    for a, f in ((sc.surface, b.surface), (sc.collision, b.collision), (sc.viscosity, b.viscosity)):
        a[z0:z0 + nzb] = f
    for src, dst in ((b.vel, sc.vel), (b.colvel, sc.colvel)):
        for a in range(3):
            extra = 1 if a == 2 else 0
            v = big(src[a], 0.0, extra)
            v[z0:z0 + nzb + extra] = src[a]
            dst.append(np.ascontiguousarray(v))
    return sc


GPU_CASES = {
    "s5_half_tile16": lambda: (scenes.scene_s5(0.5, tileSize=16, tilePadding=3), {}),       # 256 x 128 x 128, S5's blob off-centre in x
    "s4_128_tile32": lambda: (scenes.scene_s4(128), {}),                                    # tile 32: 4 units of 32 layers
}

CASES = {
    # 40 blob layers at the top of 96: the even cuts of 2 / 3 / 4 ranks leave the lower slabs empty (slab-local setup)
    "offz_blob_tile16": lambda: (shifted_blob(32, 40, 96, 56), {}),
    "offz_blob_tile16_low": lambda: (shifted_blob(32, 40, 96, 0), {}),
    # the boundary fix-up of this blob has work: a slab-local attempt restarts with the setup replicated
    "fixup_blob_32x32x48_tile16": lambda: (scenes.blob_scene((32, 32, 48), seed=1, tile=16, pad=2), {}),
}


def register():
    spanning_cases.register()
    parity.DIST_CASES.update(CASES)
    parity.DIST_CASES.update(GPU_CASES)


def steps(s, sc, out, fields):
    """A step, ps_rebalance, a step on the cuts it chose."""
    out["rc1"], _, _ = s.step_scene(sc)
    out["unitLoad"] = s.vector("unitLoad")
    out["rb_rc"], out["rb_cuts"] = s.rebalance()
    out["rc"], vel, valid = s.step_scene(sc)
    out["iterations"] = s.count("iterations")
    out["unitLoad_after"] = s.vector("unitLoad")
    for k in parity.COUNTS:
        out["count_" + k] = s.count(k)
    for a in range(3):
        out[f"vel{a}"], out[f"valid{a}"] = vel[a], valid[a]
    if fields:
        for slot in range(7):
            for kind, name in ((0, "labels"), (1, "active"), (2, "reduced")):
                out[f"{name}{slot}"] = s.index_field(kind, slot)
    else:
        for m in ("G", "Dt", "JG"):
            for i, x in enumerate(s.csr(m)[1:]):
                out[f"csr_{m}_{i}"] = x


def single_or_multi(case, outdir, ndev):
    from polystokes_b200 import PolyStokesSolver
    register()
    sc, ov = parity.DIST_CASES[case]()
    out = {}
    if ndev == 1:
        s = PolyStokesSolver.from_scene(sc, **ov)
        steps(s, sc, out, True)
        for m in ("G", "Dt", "JG"):
            for i, x in enumerate(s.csr(m)[1:]):
                out[f"csr_{m}_{i}"] = x
    else:
        s = PolyStokesSolver.from_scene(sc, devices=list(range(ndev)), **ov)
        steps(s, sc, out, False)
    out["cuts"] = np.array(s.partition()[4])
    s.close()
    np.savez(os.path.join(outdir, "single.npz" if ndev == 1 else "multi.npz"), **out)


def make(case, gpu, **extra):
    from polystokes_b200 import PolyStokesSolver
    sc, ov = parity.DIST_CASES[case]()
    ov = dict(ov, **extra)
    if gpu:
        local = int(os.environ.get("LOCAL_RANK", "0"))
        s = PolyStokesSolver.from_scene(sc, device=local, **ov)
        s.init_distributed()
    else:
        from dist_worker import attach_gloo
        s = PolyStokesSolver.from_scene(sc, lib_path=parity.EMUL_LIB, **ov)
        attach_gloo(s)
    return s, sc


def record(s, sc, out, outdir, gpu):
    """What tests/dist_worker.py records for parity.check_distributed, on the handle's current cuts."""
    from dist_worker import REGION_VECTORS, applies_before_step, applies_after_step
    s.setup_scene(sc)
    rank, n, zlo, zhi, cuts = s.partition()
    out.update(rank=rank, nranks=n, zlo=zlo, zhi=zhi, cuts=np.array(cuts), local=s.count("slabLocal"), shared=s.count("sharedRegions"))
    for k in parity.COUNTS:
        out["count_" + k] = s.count(k)
    for slot in range(7):
        out[f"labels{slot}"] = s.index_field(0, slot)
        out[f"active{slot}"] = s.index_field(1, slot)
        out[f"reduced{slot}"] = s.index_field(2, slot)
    for v in REGION_VECTORS:
        out["vec_" + v] = s.vector(v)
    out["unitLoad_after"] = s.vector("unitLoad")
    state = applies_before_step(s, out, outdir)
    rc, vel, valid = s.step_scene(sc)
    out["rc"] = rc
    out["iterations"] = s.count("iterations")
    out["solution"] = s.vector("solution")
    for a in range(3):
        out[f"vel{a}"] = vel[a]
        out[f"valid{a}"] = valid[a]
    applies_after_step(s, out, state)
    rc2, vel2, _ = s.step_scene(sc)
    out["repeat_ok"] = bool(rc2 == rc and all(np.array_equal(vel[a], vel2[a]) for a in range(3)))
    return vel


def set_params(s, **kw):
    for k, v in kw.items():
        setattr(s._P, k, v)
    rc = s.lib.ps_set_params(s.h, s._P)
    assert rc == 1, s.last_error()


def main():
    mode, case, outdir = sys.argv[1], sys.argv[2], sys.argv[3]
    if mode == "steps" and "RANK" not in os.environ:
        return single_or_multi(case, outdir, int(sys.argv[4]))
    args = sys.argv[4:]
    gpu = "gpu" in args
    args = [a for a in args if a != "gpu"]
    cuts = [int(c) for c in args[0].split(",")] if args else None
    import torch
    import torch.distributed as dist
    register()
    if gpu:
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        dist.init_process_group("gloo")
    rank = dist.get_rank()
    out = {}
    s, sc = make(case, gpu)
    out["even_cuts"] = np.array(s.partition()[4])
    if mode == "rebalance":
        out["rb0_rc"] = s.rebalance()[0]              # before any setup
        s.setup_scene(sc)
        out["unitLoad"] = s.vector("unitLoad")
        out["unitCounts"] = s.vector("unitCounts")
        out["cg_bytes"] = s.kernel_bytes("cg_iteration")
        out["rb1_rc"], out["rb1_cuts"] = s.rebalance()
        out["rb2_rc"], out["rb2_cuts"] = s.rebalance()
        record(s, sc, out, outdir, gpu)
    elif mode == "set":
        out["set_rc"] = s.set_partition(cuts)
        vel = record(s, sc, out, outdir, gpu)
        n = len(cuts) - 1
        # one broken rule each: the ends, the order, an empty slab, a cut off the unit, and cuts that differ between the ranks
        bad = {"first": [16] + cuts[1:], "last": cuts[:-1] + [sc.nz - 16],
               "order": [0] + cuts[1:-1][::-1] + [sc.nz] if n > 2 else [0, sc.nz + 16, sc.nz],
               "empty": [0, 0] + cuts[2:], "unit": [0] + [c + 8 for c in cuts[1:-1]] + [sc.nz],
               "disagree": cuts if rank else [0] + [c + 16 if c + 16 < sc.nz else c - 16 for c in cuts[1:-1]] + [sc.nz]}
        for name, c in bad.items():
            out[f"bad_{name}_rc"] = s.set_partition(c)
            out[f"bad_{name}_cuts"] = np.array(s.partition()[4])
        _, vel2, _ = s.step_scene(sc)
        out["kept_step_ok"] = bool(all(np.array_equal(vel[a], vel2[a]) for a in range(3)))
        out["null_rc"] = s.set_partition(None)
        out["null_cuts"] = np.array(s.partition()[4])
        s.set_partition(cuts)
        set_params(s, dt=sc.dt * 0.5)
        out["dt_cuts"] = np.array(s.partition()[4])
        set_params(s, tileSize=32)
        out["tile32_cuts"] = np.array(s.partition()[4])
    elif mode == "restart":
        out["set_rc"] = s.set_partition(cuts)
        record(s, sc, out, outdir, gpu)
    elif mode == "steps":
        steps(s, sc, out, True)
        rank_, n, zlo, zhi, cuts_ = s.partition()
        out.update(rank=rank_, nranks=n, zlo=zlo, zhi=zhi, cuts=np.array(cuts_), peer=s.count("peerTransport"))
    elif mode == "move":
        low, _ = parity.DIST_CASES[case + "_low"]()
        for name, scene in (("low", low), ("high", sc)):
            for phase in ("first", "rebalanced"):
                rc, vel, _ = s.step_scene(scene)
                part = s.partition()[4]
                fresh, _ = make(case, gpu)
                out[f"{name}_{phase}_set"] = fresh.set_partition(part)
                rc2, vel2, _ = fresh.step_scene(scene)
                fresh.close()
                out[f"{name}_{phase}_cuts"] = np.array(part)
                out[f"{name}_{phase}_same"] = bool(rc == rc2 == 1 and all(np.array_equal(vel[a], vel2[a]) for a in range(3)))
                if phase == "first":
                    out[f"{name}_rb"], _ = s.rebalance()
    s.close()
    np.savez(os.path.join(outdir, f"rank{rank}.npz"), **out)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()

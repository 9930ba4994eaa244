"""Worker of tests/test_distributed_emul.py: one rank of a world_size-N gloo job.

Runs the z-slab decomposed step of the host-emulation twin (the product sources compiled with -DPS_EMULATE, see
tests/test_emulated_kernels.py); the two collectives of the distributed CG are served by torch.distributed/gloo
through host callbacks.  Writes this rank's results to <outdir>/rank<k>.npz for the parent test to merge and
compare with the oracle.  With a third argument "gpu" the worker drives the CUDA product library instead (one rank per
GPU, NCCL inside the library, tests/test_gpu_distributed.py).
Usage: python dist_worker.py <case> <outdir> [gpu]   (RANK / WORLD_SIZE / MASTER_* in the env)
"""
import ctypes as C
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

AR_CB = C.CFUNCTYPE(None, C.c_void_p, C.POINTER(C.c_double), C.c_int)
SR_CB = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_void_p), C.POINTER(C.c_size_t),
                    C.POINTER(C.c_void_p), C.POINTER(C.c_size_t))


def _bytes_view(addr, n):
    return torch.from_numpy(np.ctypeslib.as_array(C.cast(addr, C.POINTER(C.c_uint8)), shape=(n,)))


def _allreduce(ctx, buf, n):
    t = torch.from_numpy(np.ctypeslib.as_array(buf, shape=(n,)))
    dist.all_reduce(t)


def _sendrecv(ctx, npeers, peers, sb, sbytes, rb, rbytes):
    reqs, keep = [], []
    for i in range(npeers):
        if peers[i] < 0:
            continue
        if sbytes[i]:
            s = _bytes_view(sb[i], sbytes[i]).clone()
            keep.append(s)
            reqs.append(dist.isend(s, peers[i]))
        if rbytes[i]:
            reqs.append(dist.irecv(_bytes_view(rb[i], rbytes[i]), peers[i]))
    for q in reqs:
        q.wait()


_CALLBACKS = (AR_CB(_allreduce), SR_CB(_sendrecv))


def attach_gloo(solver):
    lib = solver.lib
    lib.ps_comm_init_callbacks.argtypes = [C.c_void_p, C.c_int, C.c_int, AR_CB, SR_CB, C.c_void_p]
    lib.ps_comm_init_callbacks.restype = C.c_int
    rc = lib.ps_comm_init_callbacks(solver.h, dist.get_rank(), dist.get_world_size(), _CALLBACKS[0], _CALLBACKS[1], None)
    assert rc == 1, solver.last_error()


REGION_VECTORS = ("b", "reducedRHS", "BinvDense", "MrDense", "ViscDense", "bestFit")


def applies_before_step(s, out, outdir):
    """apply(x1), apply(x2), apply(x1) again after one apply, then after two (parity.apply_inputs), then the single-region inputs of
    <outdir>/probes.npz if the parent wrote one (parity.write_region_probes).  Returns what applies_after_step needs."""
    import parity
    n = s.count("nSystemSize")
    if n == 0:
        out.update(apply=np.zeros(0), apply_x2=np.zeros(0))
        return None
    x1, x2 = parity.apply_inputs(n)
    out["apply"] = s.apply(x1)
    out["apply_x2"] = s.apply(x2)
    again = [s.apply(x1)]
    again += [s.apply(x2), s.apply(x2)]
    again.append(s.apply(x1))
    path = os.path.join(outdir, "probes.npz")
    if os.path.exists(path):
        P = np.load(path)
        for i in range(len(P["regions"])):
            x = np.zeros(n)
            x[P[f"cols{i}"]] = P[f"vals{i}"]
            y = s.apply(x)
            rows = P[f"rows{i}"]
            out[f"probe{i}"] = y[rows]
            y[rows] = 0.0
            out[f"probe{i}_outside"] = np.count_nonzero(y)
    return x1, again


def applies_after_step(s, out, state):
    """apply(x1) once more after the step; every apply(x1) and apply(x2) of this rank must be bit-identical to its first."""
    if state is None:
        out["apply_stable"] = True
        return
    x1, again = state
    y1, y2 = out["apply"], out["apply_x2"]
    out["apply_stable"] = bool(np.array_equal(again[0], y1) and np.array_equal(again[1], y2) and np.array_equal(again[2], y2)
                               and np.array_equal(again[3], y1) and np.array_equal(s.apply(x1), y1))


def main():
    case, outdir = sys.argv[1], sys.argv[2]
    gpu = len(sys.argv) > 3 and sys.argv[3] == "gpu"
    import parity
    from polystokes_b200 import PolyStokesSolver
    sc, ov = parity.DIST_CASES[case]()
    if gpu:
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        s = PolyStokesSolver.from_scene(sc, device=local, **ov)
        s.init_distributed()
    else:
        dist.init_process_group("gloo")
        s = PolyStokesSolver.from_scene(sc, lib_path=parity.EMUL_LIB, **ov)
        attach_gloo(s)
    rank, n, zlo, zhi, cuts = s.partition()
    s.setup_scene(sc)
    out = dict(rank=rank, nranks=n, zlo=zlo, zhi=zhi, cuts=np.array(cuts), peer=s.count("peerTransport") if gpu else 0, local=s.count("slabLocal"),
               shared=s.count("sharedRegions"))
    for k in parity.COUNTS:
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
    out["iterations"] = s.count("iterations")
    out["solution"] = s.vector("solution")
    for a in range(3):
        out[f"vel{a}"] = vel[a]
        out[f"valid{a}"] = valid[a]
    applies_after_step(s, out, state)
    # a second step on the same handle must reproduce the first bit for bit
    rc2, vel2, _ = s.step_scene(sc)
    out["repeat_ok"] = bool(rc2 == rc and all(np.array_equal(vel[a], vel2[a]) for a in range(3)))
    if case in parity.DIST_NEXT:        # a different scene on the same handle
        sc2 = parity.DIST_NEXT[case]()
        rc3, vel3, valid3 = s.step_scene(sc2)
        out["next_rc"] = rc3
        out["next_iterations"] = s.count("iterations")
        out["next_nSystemSize"] = s.count("nSystemSize")
        out["next_regionCount"] = s.count("regionCount")
        for a in range(3):
            out[f"next_vel{a}"] = vel3[a]
            out[f"next_valid{a}"] = valid3[a]
    np.savez(os.path.join(outdir, f"rank{rank}.npz"), **out)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()

"""Worker of tests/test_distributed_export_emul.py and tests/test_gpu_distributed_export.py: the file set of ps_export (exportMatrices /
exportComponentMatrices / exportStats, what = 7) from a slab-decomposed step, and the comparison with the export of one rank.

  python export_worker.py ref  <case> <outdir> [gpu]     a plain handle (world 1): <outdir>/ref/x_*.mtx
  python export_worker.py rank <case> <outdir> [gpu]     one rank of a job with one process per rank (RANK / WORLD_SIZE / MASTER_* in the
                                                         env; gloo and the emulation twin, or NCCL and the CUDA library with "gpu")
  python export_worker.py multi <case> <outdir> <ndev>   a ps_create_multi handle over ndev GPUs
  python export_worker.py views <case> <outdir> <ndev>   the global views of a ps_create_multi handle: the oracle checks of parity
                                                         (matrices, region blocks, operator) with it, and every ps_get_csr block equal
                                                         to the single-GPU handle's
  python export_worker.py auto <case> <outdir> <ndev>    a ps_create_multi step with the export toggles on against one with them off

Every rank passes its own prefix, <outdir>/rank<k>/x_: rank 0 must write the whole set there and the other ranks nothing.  With
EXPORT_AUTO=1 the files come from ps_step with the export toggles of ps_params, otherwise from ps_export after the step.  A rank then
exports into a directory that does not exist (every rank must fail, naming the prefix), steps and exports once more (must succeed).
Each run writes <outdir>/<name>.json with the result, iterations and those checks."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import parity  # noqa: E402
import spanning_cases  # noqa: E402

PREFIX = "x_"
COMPONENT_MATS = ["Mat_Mc", "Mat_McInv", "Mat_Mr", "Mat_Mr_plus_2JDtuDJ", "Mat_Inv_Mr_plus_2JDtuDJ", "Mat_u", "Mat_uInv", "Mat_G", "Mat_Dt", "Mat_JG", "Mat_JDt"]
COMPONENT_VECS = ["Vec_activeRHS", "Vec_reducedRHS", "Vec_pressureRHS", "Vec_stressRHS"]
BYTE_EQUAL = COMPONENT_MATS + COMPONENT_VECS + ["Mat_A", "Vec_b", "Vec_guess"]
FILES = BYTE_EQUAL + ["solutionVector", "dimData", "solveData"]      # the 21 files of one export
THREAD_COUNT = 22                                                     # dimData entry: SMs, summed over the ranks


def scene(case):
    """The case's scene and overrides, with the warm-start guess on and the factored CG solver."""
    spanning_cases.register()
    sc, ov = parity.DIST_CASES[case]()
    return sc, dict(ov, useWarmStart=1, solverType=0)


def toggles(prefix):
    return dict(exportMatrices=1, exportComponentMatrices=1, exportStats=1, exportDataPrefix=prefix)


def run_handle(s, sc, outdir, name, rank, auto):
    """Step + export (ps_step's toggles, or ps_export), the failing export, and one more step + export; returns the record."""
    d = os.path.join(outdir, f"rank{rank}")
    os.makedirs(d, exist_ok=True)
    rc, _, _ = s.step_scene(sc)
    if not auto:
        s.export(os.path.join(d, PREFIX), 7)
    rec = dict(rc=int(rc), iterations=s.count("iterations"))
    bad = os.path.join(outdir, "no_such_dir", PREFIX)
    rec["bad_rc"] = int(s.lib.ps_export(s.h, bad.encode(), 7))
    rec["bad_error"] = s.last_error()
    rec["bad_prefix"] = bad
    again = os.path.join(outdir, "again", f"rank{rank}")
    os.makedirs(again, exist_ok=True)
    rc2, _, _ = s.step_scene(sc)
    rec["again_rc"] = int(rc2)
    rec["again_export"] = int(s.lib.ps_export(s.h, os.path.join(again, PREFIX).encode(), 7))
    with open(os.path.join(outdir, f"{name}.json"), "w") as f:
        json.dump(rec, f)
    return rec


def main():
    mode, case, outdir = sys.argv[1], sys.argv[2], sys.argv[3]
    gpu = len(sys.argv) > 4 and sys.argv[4] == "gpu"
    auto = os.environ.get("EXPORT_AUTO") == "1"
    from polystokes_b200 import PolyStokesSolver
    sc, ov = scene(case)
    lib = None if gpu or mode == "multi" else parity.EMUL_LIB
    if mode == "ref":
        s = PolyStokesSolver.from_scene(sc, lib_path=lib, **ov)
        run_handle(s, sc, os.path.join(outdir, "ref"), "ref", 0, False)
        s.close()
    elif mode == "multi":
        ndev = int(sys.argv[4])
        prefix = os.path.join(outdir, "rank0", PREFIX)
        s = PolyStokesSolver.from_scene(sc, devices=list(range(ndev)), **dict(ov, **(toggles(prefix) if auto else {})))
        run_handle(s, sc, outdir, "rank0", 0, auto)
        s.close()
    elif mode == "views":
        views(case, int(sys.argv[4]))
    elif mode == "auto":
        auto_export(case, outdir, int(sys.argv[4]))
    else:
        import torch
        import torch.distributed as dist
        rank = int(os.environ["RANK"])
        prefix = os.path.join(outdir, f"rank{rank}", PREFIX)
        ov = dict(ov, **(toggles(prefix) if auto else {}))
        if gpu:
            local = int(os.environ.get("LOCAL_RANK", "0"))
            torch.cuda.set_device(local)
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            s = PolyStokesSolver.from_scene(sc, device=local, **ov)
            s.init_distributed()
        else:
            from dist_worker import attach_gloo
            dist.init_process_group("gloo")
            s = PolyStokesSolver.from_scene(sc, lib_path=lib, **ov)
            attach_gloo(s)
        run_handle(s, sc, outdir, f"rank{rank}", rank, auto)
        dist.barrier()
        dist.destroy_process_group()


def views(case, ndev):
    from oracle.oracle import Oracle
    from polystokes_b200 import PolyStokesSolver
    sc, ov = scene(case)
    o = Oracle(sc, **{k: v for k, v in ov.items() if k != "solverType"}).setup()
    many = PolyStokesSolver.from_scene(sc, devices=list(range(ndev)), **ov)
    many.setup_scene(sc)
    parity.check_matrices(o, many)
    parity.check_region_blocks(o, many)
    parity.check_operator(o, many)
    one = PolyStokesSolver.from_scene(sc, **ov)
    one.setup_scene(sc)
    for m in parity.BITEXACT_MATS + parity.TOL_MATS:
        a, b = one.csr(m), many.csr(m)
        assert tuple(a[0]) == tuple(b[0]) and all(np.array_equal(x, y) for x, y in zip(a[1:], b[1:])), f"{m}: multi handle differs from one GPU"
    many.close()
    one.close()


def auto_export(case, outdir, ndev):
    """ps_step with the export toggles on: the same result and velocities as without them, the same files as ps_export after the step
    (solveData holds times)."""
    from polystokes_b200 import PolyStokesSolver
    sc, ov = scene(case)
    on_dir, off_dir = os.path.join(outdir, "on"), os.path.join(outdir, "off")
    os.makedirs(on_dir)
    os.makedirs(off_dir)
    on = PolyStokesSolver.from_scene(sc, devices=list(range(ndev)), **dict(ov, **toggles(os.path.join(on_dir, PREFIX))))
    rc1, vel1, valid1 = on.step_scene(sc)
    on.close()
    off = PolyStokesSolver.from_scene(sc, devices=list(range(ndev)), **ov)
    rc2, vel2, valid2 = off.step_scene(sc)
    off.export(os.path.join(off_dir, PREFIX), 7)
    off.close()
    assert rc1 == rc2 == 1 and all(np.array_equal(vel1[a], vel2[a]) and np.array_equal(valid1[a], valid2[a]) for a in range(3))
    assert sorted(os.listdir(on_dir)) == sorted(os.listdir(off_dir)) == sorted(PREFIX + f + ".mtx" for f in FILES)
    for f in FILES:
        if f != "solveData":
            with open(os.path.join(on_dir, PREFIX + f + ".mtx"), "rb") as a, open(os.path.join(off_dir, PREFIX + f + ".mtx"), "rb") as b:
                assert a.read() == b.read(), f"{f}.mtx: automatic and explicit export differ"


# ---- the comparison (runs in the parent test) ----

def read_vector(path):
    with open(path) as f:
        lines = f.read().split("\n")
    return np.array([float(v) for v in lines[2:] if v])


def compare(case, outdir, world):
    """The export of the decomposed run (`world` ranks) under <outdir>/rank0 against the world-1 export under <outdir>/ref/rank0."""
    from oracle.oracle import Oracle
    ref_dir, got_dir = os.path.join(outdir, "ref", "rank0"), os.path.join(outdir, "rank0")
    want = sorted(PREFIX + f + ".mtx" for f in FILES)
    assert sorted(os.listdir(ref_dir)) == want, f"world 1 wrote {sorted(os.listdir(ref_dir))}"
    assert sorted(os.listdir(got_dir)) == want, f"rank 0 wrote {sorted(os.listdir(got_dir))}"
    for k in range(1, world):
        d = os.path.join(outdir, f"rank{k}")
        assert not os.path.isdir(d) or not os.listdir(d), f"rank {k} wrote {os.listdir(d)}"
    path = lambda d, f: os.path.join(d, PREFIX + f + ".mtx")
    for f in BYTE_EQUAL:      # also on shared regions: their rows are merged into the single-rank order before any sum (ps_api.cu, k_rows)
        with open(path(ref_dir, f), "rb") as a, open(path(got_dir, f), "rb") as b:
            assert a.read() == b.read(), f"{f}.mtx differs from the single-rank export"
    ra, rb = read_vector(path(ref_dir, "dimData")), read_vector(path(got_dir, "dimData"))
    assert ra.size == rb.size == 27
    keep = np.arange(27) != THREAD_COUNT
    assert np.array_equal(ra[keep], rb[keep]), "dimData differs outside the thread count"
    assert rb[THREAD_COUNT] == world * ra[THREAD_COUNT], f"thread count {rb[THREAD_COUNT]} on {world} ranks, {ra[THREAD_COUNT]} on one"
    with open(path(ref_dir, "dimData")) as a, open(path(got_dir, "dimData")) as b:
        la, lb = a.read().split("\n"), b.read().split("\n")
    assert [l for i, l in enumerate(la) if i != 2 + THREAD_COUNT] == [l for i, l in enumerate(lb) if i != 2 + THREAD_COUNT], "dimData bytes"
    # the oracle: the warm-start guess at the gate of parity.check_eigen_cg, the stop rule on the merged solution
    sc, ov = scene(case)
    o = Oracle(sc, **{k: v for k, v in ov.items() if k != "solverType"}).setup()
    o.construct_guess()
    guess = read_vector(path(got_dir, "Vec_guess"))
    assert parity.rel(o.vector("guess"), guess) <= 1e-10, f"Vec_guess vs oracle rel {parity.rel(o.vector('guess'), guess):.2e}"
    n = o.count("nSystemSize")
    x = read_vector(path(got_dir, "solutionVector"))
    assert x.size == n
    if n:
        e = o.vector("b") - o.apply(x)
        rr, xx = float(e @ e), float(x @ x)
        t2 = sc.params["tolerance"] ** 2
        got = min(rr, rr / max(xx, 1e-300))
        assert got < 1.5 * t2, f"exported solution does not satisfy the stop rule: {got:.3e} >= {t2:.1e}"
    sa, sb = read_vector(path(ref_dir, "solveData")), read_vector(path(got_dir, "solveData"))
    assert np.isfinite(sb[0]), "solveData error entry"
    assert abs(sa[1] - sb[1]) <= max(2, int(0.01 * sa[1])), f"iterations {sb[1]} vs {sa[1]} on one rank"


if __name__ == "__main__":
    main()

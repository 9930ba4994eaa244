"""Scenes that reach the grid border and SDF / viscosity values at the edges of their range (tests/edge_cases.py), against the oracle:
on the host-emulation twin here, on the GPU with -m gpu; slab-decomposed border runs on the twin (gloo) and on several GPUs.

Gates per case:
  - the 14 weight fields, the 21 index fields and the counts bit-exact (parity.check_classification); the valid faces bit-exact;
  - G, D^T, M_c, M_c^-1, mu, mu^-1 and the three right-hand sides bit-equal, every sparsity pattern bit-exact (parity.check_matrices);
  - the region blocks region by region against parity.REGION_GATES;
  - the apply componentwise against the oracle's factors evaluated by scipy (parity.scipy_factored) at parity.OPERATOR_GATE;
  - the solve with parity.check_solve's gates.  The viscosity cases run ~1600-1900 CG iterations, where two correct runs stop a few
    per cent apart: there the reference's stop rule is recomputed on the returned x with the oracle's apply, and the velocity is
    compared with the oracle's step solved to tol / 1000.
A sub-sample whose interpolated SDF is NaN counts as neither liquid nor fluid (BASELINE.md section 3).
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import edge_cases
import parity
from oracle import ref_classify
from oracle.oracle import Oracle
from polystokes_b200 import PolyStokesSolver
from test_distributed_emul import launch

HERE = os.path.dirname(os.path.abspath(__file__))

CASES = edge_cases.CASES

# Velocity gate of the viscosity cases: the distance to the oracle's tol / 1000 solve (max |diff| / max |v| per axis) may be at most
# VISC_VEL_SLACK times that of the oracle's own solve at the case's tolerance.  These systems are ill conditioned: at tol 1e-4 both runs
# land percents from the converged field (measured on the twin: mu = 0 on half the blob 2.2e-2, the oracle 1.9e-2 to 2.4e-2 from run
# to run with its OpenMP sums; six decades 7.0e-2 against 7.7e-2 to 7.8e-2).  A wrong solve is O(1) off.
VISC_VEL_SLACK = 2.0


def check_case(name, lib_path=None):
    """Every gate of the module docstring on one case; returns (worst componentwise apply error, worst region-block error / gate)."""
    sc, ov = CASES[name]()
    o = Oracle(sc, **ov).setup()
    s = PolyStokesSolver.from_scene(sc, lib_path=lib_path, **ov)
    s.setup_scene(sc)
    parity.check_classification(o, s)
    parity.check_matrices(o, s)
    blk = parity.check_region_blocks(o, s)
    op = 0.0
    n = o.count("nSystemSize")
    if n:
        apply = parity.scipy_factored(o.csr, sc.dt)
        for seed in (0, 1):
            x = np.random.default_rng(seed).standard_normal(n)
            Ax, bound = apply(x)
            e = parity.operator_error(s.apply(x), Ax, bound)
            assert e <= parity.OPERATOR_GATE, f"{name}: componentwise apply error {e:.2e} > {parity.OPERATOR_GATE:.0e}"
            op = max(op, e)
    if name in edge_cases.VISC_CASES:
        check_visc_solve(name, sc, ov, o, s)
    else:
        parity.check_solve(sc, o, s, ov)
    if ref_classify.available():
        # the reference's own classifier and blocks on the weights the library computed: the oracle is the right arbiter at the border
        from test_ref_classify import _check
        rc, vel, valid = s.step_scene(sc)
        _check(sc, ov, s.index_field, s.weight_field, s.count, lambda a: valid[a], s.csr, s.vector, exact_values=parity.BITEXACT_MATS, asm_tol=1e-9)
    s.close()
    return op, max(blk[v] / g for v, g in parity.REGION_GATES.items())


def check_visc_solve(name, sc, ov, o, s):
    rs, vel, valid = s.step_scene(sc)
    prm = dict(sc.params, **ov)
    tol = prm["tolerance"]
    assert rs == 1, f"{name}: solver result {rs}"
    # the reference's stop rule min(rr, rr / xx) < tol^2 (pcg.h:316-325) on the returned x, with the oracle's apply (slack 1.5: the
    # loop tests its recursively updated residual, this is the true one)
    x = s.vector("solution")
    e = o.vector("b") - o.apply(x)
    rr, xx = float(e @ e), float(x @ x)
    got = min(rr, rr / max(xx, 1e-300))
    assert got < 1.5 * tol ** 2, f"{name}: returned x does not satisfy the stop rule: {got:.3e} >= {tol ** 2:.1e}"
    assert abs(s.real("xmag") - xx) <= 1e-11 * max(xx, 1e-300), f"{name}: x.x recurrence drift"
    tight = Oracle(sc, **dict(ov, tolerance=tol / 1000, maxIterations=20000)).setup()
    assert tight.solve() == 1 and o.solve() == 1
    tvel, tvalid = tight.writeback()
    ovel, _ = o.writeback()
    dist = lambda v: max(float(np.abs(tvel[a] - v[a]).max()) / max(float(np.abs(tvel[a]).max()), 1e-30) for a in range(3))
    for a in range(3):
        assert np.array_equal(tvalid[a], valid[a]), f"{name}: valid field axis {a}"
    mine, oracle = dist(vel), dist(ovel)
    print(f"{name}: {s.count('iterations')} iterations (oracle {o.count('iterations')}), velocity {mine:.2e} from the tol / 1000 solve (oracle {oracle:.2e})")
    assert mine <= VISC_VEL_SLACK * oracle, f"{name}: velocity {mine:.2e} from the tol / 1000 solve, the oracle's {oracle:.2e}"


@pytest.mark.parametrize("case", list(CASES))
def test_emulated_input_edge_matches_oracle(built, case):
    op, blk = check_case(case, lib_path=parity.EMUL_LIB)
    print(f"emulated {case}: worst componentwise apply error {op:.2e}, worst region-block error {blk:.2e} of its gate")


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_gpu_input_edge_matches_oracle(built, case):
    op, blk = check_case(case)
    print(f"gpu {case}: worst componentwise apply error {op:.2e}, worst region-block error {blk:.2e} of its gate")


def _box_any(mask):
    """out[c] = mask anywhere in the 3x3x3 cell block around c, clamped at the border (the block of the weight kernel's pre-pass)."""
    p = np.pad(mask, 1, mode="edge")
    nz, ny, nx = mask.shape
    out = np.zeros_like(mask)
    for dz in range(3):
        for dy in range(3):
            for dx in range(3):
                out |= p[dz:dz + nz, dy:dy + ny, dx:dx + nx]
    return out


@pytest.mark.parametrize("case", list(edge_cases.SDF_CASES))
def test_sdf_value_case_reaches_both_paths(case):
    """The written values lie where the weight kernel decides by the signs of the block alone (no value < 0 next to one >= 0, NaN
    being neither) and where it interpolates (both signs in the block), and the base scene has liquid."""
    field, value = case.split("_", 1)
    sc, written = edge_cases.sdf_case(field, value)
    a = sc.surface if field == "surface" else sc.collision
    neg, nonneg = _box_any(a < 0), _box_any(a >= 0)
    by_signs, interpolated = written & ~(neg & nonneg), _box_any(written) & neg & nonneg
    assert by_signs.any() and interpolated.any(), f"{case}: {by_signs.sum()} cells decided by signs, {interpolated.sum()} interpolated"
    assert (sc.surface < 0).any()


def test_border_scenes_reach_the_border():
    """Liquid on every domain face of the tanks and the full grid, on the planes x = 0, y = 0, z = 0 and z = nz - 1 of the border blobs."""
    for name in edge_cases.BORDER:
        sc, _ = edge_cases.BORDER[name]()
        liq = sc.surface < 0
        faces = {"x0": liq[:, :, 0], "y0": liq[:, 0, :], "z0": liq[0], "ztop": liq[-1]}
        if not name.startswith("border_blob"):
            faces.update(x1=liq[:, :, -1])
        assert all(f.any() for f in faces.values()), f"{name}: no liquid on {[k for k, f in faces.items() if not f.any()]}"


# ---- slab-decomposed border runs (edge_cases.DIST, part of parity.DIST_CASES) ----------------------------------------------------
def run_dist(case, world, outdir, port, **kw):
    """The decomposed step with the single-region inputs of parity.write_region_probes, the partition facts the case relies on, then
    parity.check_distributed."""
    parity.write_region_probes(case, outdir)
    ranks = launch(case, world, outdir, port, **kw)
    o, sc = parity.dist_reference(case)["o"], parity.dist_reference(case)["sc"]
    cuts = [int(c) for c in ranks[0]["cuts"]]
    shared, local = [int(r["shared"]) for r in ranks], [int(r["local"]) for r in ranks]
    print(f"{case} on {world} ranks: cuts {cuts}, slabLocal {local}, sharedRegions {shared}, regionCount {o.count('regionCount')}", flush=True)
    # liquid in the layer z = 0 (first slab) and in the top layer z = nz of the z-face slot, which only the last slab owns
    assert (o.weight_field(1, 0)[0] > 0).any() and (o.weight_field(1, 3)[sc.nz] > 0).any(), f"{case}: no liquid at z = 0 or z = nz"
    assert (o.index_field(1, 3)[sc.nz] >= 0).any() or (o.index_field(2, 3)[sc.nz] >= 0).any(), f"{case}: no unknown on the plane z = nz"
    if case in edge_cases.SLAB_LOCAL:
        assert all(v == 1 for v in local), f"{case}: expected the slab-local setup"
    if case in edge_cases.SHARED:
        assert all(v == shared[0] for v in shared) and shared[0] > 0, f"{case}: no region crosses a cut"
    parity.check_distributed(case, ranks)


EMUL_DIST = [(c, w) for c in ("border_tank48_uniform", "border_tank48_tile16_pad2", "border_blob48_tile8_pad1", "border_blob48_notile") for w in (2, 3)]
EMUL_DIST.append(("border_tank_32x32x96_tile12_pad1", 2))


@pytest.mark.parametrize("case,world", EMUL_DIST)
def test_emulated_border_decomposed_step_matches_oracle(built, tmp_path, case, world):
    port = 29100 + (os.getpid() + hash(case) + 13 * world) % 90
    run_dist(case, world, tmp_path, port)


def _ngpu():
    import torch
    return torch.cuda.device_count()


GPU_DIST = ([(c, 2) for c in ("border_tank48_uniform", "border_tank48_tile16_pad2", "border_blob48_tile8_pad1", "border_blob48_notile",
                              "border_tank_32x32x96_tile12_pad1")]
            + [("border_blob48_notile", 3), ("border_tank_40x40x128_tile16_pad2", 4), ("border_tank_40x40x128_tile16_pad2", 8)])


@pytest.mark.gpu
@pytest.mark.parametrize("transport", ["peer", "nccl"])
@pytest.mark.parametrize("case,world", GPU_DIST)
def test_gpu_border_decomposed_step_matches_oracle(built, tmp_path, case, world, transport):
    if _ngpu() < world:
        pytest.skip(f"needs {world} GPUs")
    port = 29800 + (os.getpid() + hash(case) + world + (7 if transport == "nccl" else 0)) % 150
    run_dist(case, world, tmp_path, port, gpu=True, extra_env={"PS_COMM": "nccl" if transport == "nccl" else ""})


@pytest.mark.gpu
@pytest.mark.parametrize("case,ndev", [("border_tank48_uniform", 2), ("border_blob48_notile", 3), ("border_tank_40x40x128_tile16_pad2", 8)])
def test_gpu_multi_handle_border_matches_single_gpu(built, case, ndev):
    """ps_create_multi (one process, one handle, several GPUs) against the single-GPU handle (tests/multi_worker.py)."""
    if _ngpu() < ndev:
        pytest.skip(f"needs {ndev} GPUs")
    env = dict(os.environ, PS_MULTI_WATCHDOG_S="45")
    try:
        r = subprocess.run([sys.executable, os.path.join(HERE, "multi_worker.py"), case, str(ndev)], capture_output=True, text=True, timeout=300, env=env)
    except subprocess.TimeoutExpired as e:
        pytest.fail(f"multi-GPU handle hung on {case} x {ndev}:\n{e.stderr}")
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]

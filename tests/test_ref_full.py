"""The reference's COMPLETE per-step solver as compiled code -- all six exec/HDK_PolyStokesSolver*.cpp + lib/src/Preconditioner.cpp +
lib/include, unmodified from /root/reference, in oracle/_ref/libps_ref_full.so (oracle/Makefile `ref`, harness oracle/ref_full.cpp, HDK
stand-in oracle/hdk_shim, Eigen facade oracle/eigen_facade) -- run through the node's stage sequence (exec/HDK_PolyStokes.C:329-608) on the
synthetic scenes, against (a) the oracle's restatement, stage by stage, and (b) the product's full step.
The library is built from a checkout of the reference's sources, which is not part of this repository; without it these tests skip.
The *_matches_oracle_stage_by_stage tests make the product-side checks of (b) against the oracle instead, the restatement that (a) pins
to the compiled reference wherever the library is built: they do not compare with the reference themselves."""
import numpy as np
import pytest

import parity
from oracle import ref_full
from oracle.oracle import Oracle
from polystokes_b200 import PolyStokesSolver, scenes

needs_reference = pytest.mark.skipif(not ref_full.available(), reason="oracle/_ref/libps_ref_full.so not built (needs the reference's sources)")

CASES = {
    "uniform_box24": lambda: scenes.box_scene(24, doReduced=0, tolerance=1e-6),
    "tiles8pad1_box40": lambda: scenes.box_scene(40, tileSize=8, tilePadding=1),
    "blob40": lambda: scenes.blob_scene(40),
    "blob40_layers31": lambda: scenes.blob_scene(40, seed=11, tile=8, pad=2, liquidLayers=3, solidLayers=1),
    "blob_ragged_36x44x52": lambda: scenes.blob_scene((36, 44, 52), seed=5, tile=16, pad=1),
    "blob32_notile": lambda: scenes.blob_scene(32, seed=3, doTile=0),
    "S2_beam_48": lambda: scenes.scene_s2(48),
    "S3_jet_64": lambda: scenes.scene_s3(64),
    "S5_blob_quarter_tile8": lambda: scenes.scene_s5(0.25, tileSize=8),
}
MATS = ("G", "Dt", "JG", "JDt", "Mc", "McInv", "u", "uInv", "Mr", "B", "BInv")
EXACT_VECS = ("com", "activeRHS", "pressureRHS", "stressRHS")
REGION_VECS = ("bestFit", "MrDense", "ViscDense", "reducedRHS")


def _setup_parity(R, x, mat_exact, region_tol, b_tol, who="the compiled reference"):
    """x: an object with the Oracle accessors (the oracle itself, or the product); R: `who`, with the same accessors."""
    for liq in (1, 0):
        for slot in range(7):
            assert np.array_equal(R.weight_field(liq, slot), x.weight_field(liq, slot)), f"weights liquid={liq} slot {slot}"
    for kind in range(3):
        for slot in range(7):
            assert np.array_equal(R.index_field(kind, slot), np.asarray(x.index_field(kind, slot)).astype(np.int64)), f"index field kind {kind} slot {slot} vs {who}"
    for k in ("nCenter", "nActiveVs", "nReducedVs", "nPressures", "nStresses", "nTotalDOFs", "nSystemSize"):
        assert R.count(k) == x.count(k), k
    for m in MATS:
        (sr, pr, ir, vr), (sx, px, ix, vx) = R.csr(m), x.csr(m)
        assert tuple(sr) == tuple(sx) and np.array_equal(pr, px) and np.array_equal(ir, ix), f"{m}: sparsity pattern vs {who}"
        if m in mat_exact:
            assert np.array_equal(vr, vx), f"{m}: values not bit-equal to {who} (rel {parity.rel(vr, vx):.2e})"
        else:
            assert parity.rel(vr, vx) <= 1e-8, f"{m}: rel {parity.rel(vr, vx):.2e}"
    for v in EXACT_VECS:
        assert np.array_equal(R.vector(v), x.vector(v)), f"{v} not bit-equal to {who}"
    for v in REGION_VECS:
        a, b = R.vector(v), x.vector(v)
        assert a.shape == b.shape and (a.size == 0 or parity.rel(a, b) <= region_tol), f"{v}: rel {parity.rel(a, b):.2e} vs {who}"
    assert parity.rel(R.vector("b"), x.vector("b")) <= b_tol, f"b rel {parity.rel(R.vector('b'), x.vector('b')):.2e}"


@needs_reference
@pytest.mark.parametrize("case", list(CASES))
def test_oracle_matches_compiled_reference_step(built, case):
    """Every intermediate of the step: weights, classification, centres of mass, least-squares fits, reduced mass / viscosity matrices, matrix
    blocks, B / B^-1, right-hand sides BIT-EQUAL; b to rounding; then the solve: same result code and iteration count, error to 1e-2 (1e-13 on short runs), and the
    written-back valid fields equal and velocity (fp32) within the solver tolerance (a tenth of the parity gate)."""
    sc = CASES[case]()
    o = Oracle(sc, threads=1).setup()        # one thread: the oracle's OpenMP reductions are not reproducible from run to run
    R = ref_full.RefFull(sc).setup()
    _setup_parity(R, o, mat_exact=MATS, region_tol=0.0 if False else 1e-15, b_tol=1e-13)
    for v in REGION_VECS:      # bit-equal in fact: the oracle follows the reference's operation order
        assert np.array_equal(R.vector(v), o.vector(v)), f"{v} not bit-equal"
    rr, ro = R.solve(), o.solve()
    assert rr == ro == 1
    # identical counts; on solves of many hundreds of iterations the oracle's OpenMP dot products can tip the stop test by one iteration
    assert abs(R.count("iterations") - o.count("iterations")) <= o.count("iterations") // 500, f"iterations {R.count('iterations')} vs {o.count('iterations')}"
    if R.count("iterations") == o.count("iterations"):
        assert abs(R.real("solveError") - o.real("solveError")) <= 1e-2 * o.real("solveError")   # rounding, amplified over hundreds of iterations
    (rv, rvalid), (ov, ovalid) = R.writeback(), o.writeback()
    for a in range(3):
        assert np.array_equal(rvalid[a], ovalid[a])
        # same iteration, but the oracle's OpenMP dot products round differently: the iterates differ by rounding amplified by the conditioning
        assert float(np.abs(rv[a] - ov[a]).max()) <= max(sc.params["tolerance"], 4e-7) * max(float(np.abs(ov[a]).max()), 1e-30), f"velocity axis {a}"


def _product_vs(sc, lib_path, R, who):
    """The product's full step against R's (`who`: the compiled reference or the oracle) on the same scene, stage by stage."""
    s = PolyStokesSolver.from_scene(sc, lib_path=lib_path)
    rc, vel, valid = s.step_scene(sc)
    _setup_parity(R, s, mat_exact=parity.BITEXACT_MATS, region_tol=1e-6, b_tol=1e-10, who=who)
    rr = R.solve()
    assert rr == rc
    it = R.count("iterations")
    assert abs(it - s.count("iterations")) <= max(2, int(0.01 * it)), f"iterations: {who} {it}, product {s.count('iterations')}"
    rv, rvalid = R.writeback()
    tol = max(10 * sc.params["tolerance"], 4e-7)
    for a in range(3):
        assert np.array_equal(rvalid[a], valid[a]), f"valid axis {a}"
        assert float(np.abs(rv[a] - vel[a]).max()) <= tol * max(float(np.abs(rv[a]).max()), 1e-30), f"velocity axis {a} vs {who}"
    s.close()


EMULATED = ["uniform_box24", "blob40", "blob_ragged_36x44x52", "blob32_notile"]


def _reference(sc):
    return ref_full.RefFull(sc).setup(), "the compiled reference"


def _oracle(sc):
    return Oracle(sc, threads=1).setup(), "the oracle"


@needs_reference
@pytest.mark.parametrize("case", EMULATED)
def test_emulated_step_matches_compiled_reference(built, case):
    sc = CASES[case]()
    _product_vs(sc, parity.EMUL_LIB, *_reference(sc))


@needs_reference
@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_gpu_step_matches_compiled_reference(built, case):
    sc = CASES[case]()
    _product_vs(sc, None, *_reference(sc))


@pytest.mark.parametrize("case", EMULATED)
def test_emulated_step_matches_oracle_stage_by_stage(built, case):
    sc = CASES[case]()
    _product_vs(sc, parity.EMUL_LIB, *_oracle(sc))


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_gpu_step_matches_oracle_stage_by_stage(built, case):
    sc = CASES[case]()
    _product_vs(sc, None, *_oracle(sc))


@needs_reference
def test_compiled_reference_bicgstab_fallback_and_eigen_cg(built):
    """The reference's own fallback (S.cpp:784-799) and its solveEigenCG path (S.cpp:814-862, explicit A) against the oracle."""
    sc = scenes.blob_scene(32, seed=4, maxIterations=8, tolerance=1e-12, keepNonConvergedResults=1)
    o = Oracle(sc).setup(); R = ref_full.RefFull(sc).setup()
    assert R.solve() == o.solve() == 0 and R.count("iterations") == o.count("iterations") == 8
    (rv, _), (ov, _) = R.writeback(), o.writeback()
    for a in range(3):
        assert float(np.abs(rv[a] - ov[a]).max()) <= 4e-7 * max(float(np.abs(ov[a]).max()), 1e-30)
    sc = scenes.blob_scene(28, seed=6, tile=8, pad=1, solverType=1, useWarmStart=1)
    o = Oracle(sc).setup(); o.assemble_explicit_A(); o.construct_guess()
    R = ref_full.RefFull(sc).setup()
    (sr, pr, ir, vr), (so, po, io, vo) = R.csr("A"), o.csr("A")
    assert tuple(sr) == tuple(so) and np.array_equal(pr, po) and np.array_equal(ir, io) and parity.rel(vr, vo) <= 1e-13
    assert parity.rel(R.vector("guess"), o.vector("guess")) <= 1e-13
    ro = o.solve_eigen_cg()
    rr = R.solve()
    assert rr == ro and R.count("iterations") == o.count("iterations")
    assert abs(R.real("solveError") - o.real("solveError")) <= 1e-3 * o.real("solveError")

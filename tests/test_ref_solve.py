"""The reference's OWN solve stage -- lib/include/pcg.h (pcg_external_matrix_A, bicgstab_external_matrix_A) and
lib/include/ApplyPressureStressMatrix.h (applyMatrixVectorProducts), compiled unmodified from /root/reference into
oracle/_ref/libps_ref_solve.so (oracle/Makefile `ref`, on the Eigen facade of oracle/eigen_facade) -- against
(a) the oracle's restatement of the same stage and (b) the product's kernels, on the same matrices.
This is what pins SURVEY.md section 8a rows O1 / O2 / P1 and the fallback to reference CODE rather than to a reading of it.
The library is built from a checkout of the reference's sources, which is not part of this repository; without it these tests skip.
The *_match_oracle tests check the product's operator against the formula of test_reference_code_apply_matches_scipy evaluated by
scipy.sparse from the product's own component matrices, and its solve against the oracle's solve of the same scene (each on its own
system): they do not compare with the reference themselves."""
import numpy as np
import pytest

import parity
from oracle import ref_solve
from oracle.oracle import Oracle
from polystokes_b200 import PolyStokesSolver, scenes

needs_reference = pytest.mark.skipif(not ref_solve.available(), reason="oracle/_ref/libps_ref_solve.so not built (needs the reference's sources)")

CASES = {
    "uniform_box20": lambda: scenes.box_scene(20, doReduced=0, tolerance=1e-6),
    "blob40_tile8": lambda: scenes.blob_scene(40, seed=3),
    "blob32_notile": lambda: scenes.blob_scene(32, seed=5, doTile=0),
    "ragged_36x28x44": lambda: scenes.blob_scene((36, 28, 44), seed=9),
}


def rel(a, b):
    return float(np.abs(np.asarray(a) - np.asarray(b)).max()) / max(float(np.abs(np.asarray(a)).max()), 1e-300)


@needs_reference
@pytest.mark.parametrize("case", list(CASES))
def test_oracle_solve_stage_matches_reference_code(built, case):
    """Oracle restatement vs the compiled reference headers: operator apply to rounding, CG with the SAME iteration
    count and error, solution to 1e-7 (the only freedom left is the summation order of the oracle's OpenMP dots)."""
    sc = CASES[case]()
    o = Oracle(sc, threads=1).setup()        # one thread: reproducible dot products
    n = o.count("nSystemSize")
    R = ref_solve.RefSolve(o.csr, sc.dt)
    assert R.n == n
    rng = np.random.default_rng(7)
    for _ in range(2):
        x = rng.standard_normal(n)
        assert rel(R.apply(x), o.apply(x)) <= 1e-13
    ro = o.solve()
    res, it, xr, err, used = R.solve_spd(o.vector("b"), sc.params["tolerance"], sc.params["maxIterations"])
    assert (res, used) == (ro, o.count("usedBiCGStab"))
    assert it == o.count("iterations"), f"iterations: reference code {it}, oracle {o.count('iterations')}"
    assert abs(err - o.real("solveError")) <= 1e-9 * err
    assert rel(xr, o.vector("solution")) <= 1e-7       # dot-product order, amplified by the conditioning


@needs_reference
def test_reference_code_apply_matches_scipy(built):
    """Second opinion that does not involve the oracle's arithmetic or the Eigen facade's: the compiled reference operator
    (ApplyPressureStressMatrix::applyMatrixVectorProducts on the facade) against y = -dt K^T Mc^-1 K x - J^T B^-1 J x - 1/2 [0; mu^-1 x_tau]
    evaluated by scipy.sparse from the same component matrices, and the reference's explicit A (assembleSystemPressureStress) against the same
    formula as sparse triple products."""
    import scipy.sparse as sp
    from oracle import ref_full
    sc = scenes.blob_scene(28, seed=6, tile=8, pad=1, solverType=1)
    R = ref_full.RefFull(sc).setup()
    M = {}
    for name in ("BInv", "A"):
        shape, ptr, idx, val = R.csr(name)
        M[name] = sp.csr_matrix((val, idx, ptr), shape=shape)
    A = _scipy_operator(R.csr, sc.dt)
    assert abs(A - M["A"]).max() <= 1e-12 * abs(A).max(), "explicit A of the compiled reference vs scipy triple products"
    shape, ptr, idx, val = R.csr("B")
    B = sp.csr_matrix((val, idx, ptr), shape=shape)
    assert abs(M["BInv"] @ B - sp.identity(shape[0])).max() <= 1e-9, "B^-1 of the compiled reference (26 x 26 partial-pivot inverses) times B"
    x = np.random.default_rng(3).standard_normal(A.shape[0])
    S = ref_solve.RefSolve(R.csr, sc.dt)
    assert rel(S.apply(x), A @ x) <= 1e-12, "factored apply of the compiled reference vs scipy"


@needs_reference
def test_oracle_bicgstab_fallback_matches_reference_code(built):
    """CG cut after 8 iterations -> the reference restarts with bicgstab_external_matrix_A (S.cpp:784-799): same switch,
    same 8 iterations, iterates equal to rounding."""
    sc = scenes.blob_scene(32, seed=4, maxIterations=8, tolerance=1e-12, keepNonConvergedResults=1)
    o = Oracle(sc, threads=1).setup()
    ro = o.solve()
    R = ref_solve.RefSolve(o.csr, sc.dt)
    res, it, xr, err, used = R.solve_spd(o.vector("b"), sc.params["tolerance"], sc.params["maxIterations"])
    assert used == 1 == o.count("usedBiCGStab") and res == ro == 0 and it == o.count("iterations") == 8
    assert rel(xr, o.vector("solution")) <= 1e-9
    assert abs(err - o.real("solveError")) <= 1e-6 * abs(err)


_scipy_operator = parity.scipy_operator


def _product_vs_oracle(lib_path, sc):
    """The product's operator against the scipy.sparse formula on the product's OWN component matrices (ps_get_csr), and the product's
    solve against the oracle's solve of the same scene: each solves its own system (b equal to 1e-10, the matrices as tests/test_ref_full.py
    checks them), so iterations and solution are compared with the parity gates."""
    s = PolyStokesSolver.from_scene(sc, lib_path=lib_path)
    rc, vel, valid = s.step_scene(sc)
    n = s.count("nSystemSize")
    A = _scipy_operator(s.csr, sc.dt)
    assert A.shape == (n, n)
    x = np.random.default_rng(11).standard_normal(n)
    assert rel(A @ x, s.apply(x)) <= 1e-12, f"operator apply vs scipy on the product's matrices: {rel(A @ x, s.apply(x)):.2e}"
    o = Oracle(sc, threads=1).setup()
    ro = o.solve()
    it = o.count("iterations")
    assert ro == rc and o.count("usedBiCGStab") == s.count("usedBiCGStab")
    assert abs(it - s.count("iterations")) <= max(2, int(0.01 * it)), f"iterations: oracle {it}, product {s.count('iterations')}"
    assert rel(o.vector("solution"), s.vector("solution")) <= 10 * sc.params["tolerance"]
    if it == s.count("iterations"):
        err = o.real("solveError")
        assert abs(err - s.real("solveError")) <= 0.05 * err, f"error at iteration {it}: oracle {err:.6e}, product {s.real('solveError'):.6e}"
    s.close()


def _product_vs_reference(lib_path, sc):
    """The product assembles its own matrices; the reference's code then solves on THOSE matrices (exported through
    ps_get_csr) and must land where the product's own CG did."""
    s = PolyStokesSolver.from_scene(sc, lib_path=lib_path)
    rc, vel, valid = s.step_scene(sc)
    n = s.count("nSystemSize")
    R = ref_solve.RefSolve(s.csr, sc.dt)
    assert R.n == n
    x = np.random.default_rng(11).standard_normal(n)
    assert rel(R.apply(x), s.apply(x)) <= 1e-12, f"operator apply vs reference code: {rel(R.apply(x), s.apply(x)):.2e}"
    res, it, xr, err, used = R.solve_spd(s.vector("b"), sc.params["tolerance"], sc.params["maxIterations"])
    assert res == rc and used == s.count("usedBiCGStab")
    assert abs(it - s.count("iterations")) <= max(2, int(0.01 * it)), f"iterations: reference code {it}, product {s.count('iterations')}"
    assert rel(xr, s.vector("solution")) <= 10 * sc.params["tolerance"]
    # the stop test's error: only comparable at the same iteration, and only loosely -- the kernels sum their dot products in a
    # different (fixed) order than the reference code, and CG amplifies that over hundreds of iterations
    if it == s.count("iterations"):
        assert abs(err - s.real("solveError")) <= 0.05 * err, f"error at iteration {it}: reference code {err:.6e}, product {s.real('solveError'):.6e}"
    s.close()
    return it


@needs_reference
@pytest.mark.parametrize("case", list(CASES))
def test_emulated_kernels_match_reference_code(built, case):
    _product_vs_reference(parity.EMUL_LIB, CASES[case]())


def _export_vs_eigen_writer(lib_path, sc, tmp_path):
    """exportMatrices / exportComponentMatrices / exportStats (S.cpp:533-606): every file ps_export writes must be byte-identical
    to what Eigen's own writer (the checkout's MarketIO.h, compiled into oracle/_ref) produces from the same matrix / vector."""
    s = PolyStokesSolver.from_scene(sc, lib_path=lib_path)
    s.step_scene(sc)
    pre = str(tmp_path / "out_")
    s.export(pre, 7)
    mats = {"Mat_Mc.mtx": "Mc", "Mat_McInv.mtx": "McInv", "Mat_Mr.mtx": "Mr", "Mat_Mr_plus_2JDtuDJ.mtx": "B", "Mat_Inv_Mr_plus_2JDtuDJ.mtx": "BInv",
            "Mat_u.mtx": "u", "Mat_uInv.mtx": "uInv", "Mat_G.mtx": "G", "Mat_Dt.mtx": "Dt", "Mat_JG.mtx": "JG", "Mat_JDt.mtx": "JDt"}
    vecs = {"Vec_b.mtx": "b", "solutionVector.mtx": "solution", "Vec_activeRHS.mtx": "activeRHS", "Vec_reducedRHS.mtx": "reducedRHS",
            "Vec_pressureRHS.mtx": "pressureRHS", "Vec_stressRHS.mtx": "stressRHS"}
    for f, name in mats.items():
        ref_solve.save_market(s.csr(name), pre + "eigen_" + f)
        assert open(pre + f, "rb").read() == open(pre + "eigen_" + f, "rb").read(), f"{f} differs from Eigen::saveMarket's output"
    for f, name in vecs.items():
        ref_solve.save_market_vector(s.vector(name), pre + "eigen_" + f)
        assert open(pre + f, "rb").read() == open(pre + "eigen_" + f, "rb").read(), f"{f} differs from Eigen::saveMarketVector's output"
    for f, data in (("dimData.mtx", list(s.stats.dimData)), ("solveData.mtx", list(s.stats.solveData))):
        ref_solve.save_market_vector(np.array(data), pre + "eigen_" + f)
        assert open(pre + f, "rb").read() == open(pre + "eigen_" + f, "rb").read(), f
    s.close()


@needs_reference
def test_oracle_market_writer_matches_eigen_writer(built, tmp_path):
    sc = scenes.blob_scene(24, seed=2)
    o = Oracle(sc).setup()
    for name in ("G", "JDt", "BInv"):
        a, b = str(tmp_path / f"o_{name}.mtx"), str(tmp_path / f"e_{name}.mtx")
        o.save_csr(name, a); ref_solve.save_market(o.csr(name), b)
        assert open(a, "rb").read() == open(b, "rb").read(), name
    a, b = str(tmp_path / "o_b.mtx"), str(tmp_path / "e_b.mtx")
    o.save_vector("b", a); ref_solve.save_market_vector(o.vector("b"), b)
    assert open(a, "rb").read() == open(b, "rb").read()


@needs_reference
def test_emulated_export_matches_eigen_writer(built, tmp_path):
    _export_vs_eigen_writer(parity.EMUL_LIB, scenes.blob_scene(24, seed=2), tmp_path)


@needs_reference
@pytest.mark.gpu
def test_gpu_export_matches_eigen_writer(built, tmp_path):
    _export_vs_eigen_writer(None, scenes.blob_scene(24, seed=2), tmp_path)


@needs_reference
@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES) + ["S2_beam_64"])
def test_gpu_solve_matches_reference_code(built, case):
    sc = scenes.scene_s2(64) if case == "S2_beam_64" else CASES[case]()
    _product_vs_reference(None, sc)


@pytest.mark.parametrize("case", list(CASES))
def test_emulated_kernels_match_oracle(built, case):
    _product_vs_oracle(parity.EMUL_LIB, CASES[case]())


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES) + ["S2_beam_64"])
def test_gpu_solve_matches_oracle(built, case):
    _product_vs_oracle(None, scenes.scene_s2(64) if case == "S2_beam_64" else CASES[case]())

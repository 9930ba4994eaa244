"""Shared parity checks: the C-ABI library (CUDA product, or its host-emulation twin) vs the CPU oracle.

Gates (SURVEY.md section 8d): labels / DOF indices / counts / CSR patterns bit-exact; matrix values
<= 1e-8 relative (the K factors and diagonals are in fact bit-equal); b <= 1e-10; solved velocity within
10*tol (inf-norm, relative); CG iterations within max(2, 1%).
"""
import os

import numpy as np

import edge_cases
from polystokes_b200 import PolyStokesSolver, scenes
from oracle.oracle import Oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMUL_LIB = os.path.join(ROOT, "polystokes_b200", "libpolystokes_emul.so")

COUNTS = ["nCenter", "nFaceX", "nFaceY", "nFaceZ", "nEdgeYZ", "nEdgeXZ", "nEdgeXY", "regionCount", "nSystemSize",
          "nActiveVs", "nReducedVs", "nPressures", "nStresses", "nTotalDOFs"]
BITEXACT_MATS = ["G", "Dt", "Mc", "McInv", "uInv", "u"]
TOL_MATS = ["JG", "JDt", "Mr", "B", "BInv"]

# the scene matrix used by both the emulation tests (CPU) and the GPU tests
SCENE_CASES = {
    "uniform_box24": lambda: (scenes.box_scene(24, doReduced=0, tolerance=1e-6), {}),
    "tiles8pad1_box40": lambda: (scenes.box_scene(40, tileSize=8, tilePadding=1), {}),
    "blob40": lambda: (scenes.blob_scene(40), {}),
    "blob40_layers31": lambda: (scenes.blob_scene(40, seed=11, tile=8, pad=2, liquidLayers=3, solidLayers=1), {}),
    "blob_ragged_36x44x52": lambda: (scenes.blob_scene((36, 44, 52), seed=5, tile=16, pad=1), {}),
    "blob40_notile": lambda: (scenes.blob_scene(40, seed=3, doTile=0), {}),
    "blob33_uniform": lambda: (scenes.blob_scene(33, seed=9, doReduced=0), {}),
    "empty_air": lambda: (empty_scene(), {}),
}


# scenes for the slab-decomposed runs (nz >= 16 * ranks; reduced regions tiled with padding >= 1)
DIST_CASES = {
    "blob48_tile8": lambda: (scenes.blob_scene(48, seed=21, tile=8, pad=1), {}),
    "box48_uniform": lambda: (scenes.box_scene(48, doReduced=0, tolerance=1e-6), {}),
    "blob_36x40x64_tile16": lambda: (scenes.blob_scene((36, 40, 64), seed=8, tile=16, pad=2), {}),
    "blob64_tile16": lambda: (scenes.blob_scene(64, seed=13, tile=16, pad=2), {}),
    "blob64_tile16_then_shrunk": lambda: (scenes.blob_scene(64, seed=13, tile=16, pad=2, tolerance=1e-7), {}),
    "s3_128": lambda: (scenes.scene_s3(128), {}),
    "blob48_tile16_pad3_layers33": lambda: (scenes.blob_scene(48, seed=5, tile=16, pad=3, liquidLayers=3, solidLayers=3), {}),
    # tile 32: cuts at multiples of lcm(16, 32) = 32 -- 3 units over 2 ranks give slabs of 64 / 32 layers (the unequal case of S4 384^3 on 8 GPUs)
    "blob_40x36x96_tile32_pad3": lambda: (scenes.blob_scene((40, 36, 96), seed=11, tile=32, pad=3, liquidLayers=3, solidLayers=3, tolerance=1e-6), {}),
    # CG runs out of iterations -> BiCGSTAB fallback, itself stopped after 6 iterations (results kept): checks the arithmetic
    "blob48_bicgstab6": lambda: (scenes.blob_scene(48, seed=21, tile=8, pad=1, maxIterations=6, tolerance=1e-12, keepNonConvergedResults=1), {}),
    # liquid on the domain faces, in the first and the last slab (tests/test_input_edges.py)
    **edge_cases.DIST,
}


def _shrunk(sc, cells):
    sc.surface = sc.surface + cells * sc.dx
    return sc


# a second, DIFFERENT scene stepped on the same distributed handle (other system size, same grid): every per-step table and the
# layout of the shared vector arena must follow (tests/dist_worker.py steps it after the case's own scene)
DIST_NEXT = {"blob64_tile16_then_shrunk": lambda: _shrunk(scenes.blob_scene(64, seed=13, tile=16, pad=2, tolerance=1e-7), 3.0)}

# Velocity gate of the distributed comparison where 10 x tol is not meaningful: a long, thin domain is ill conditioned (650 iterations), two
# correct CG runs that sum their dot products in different orders stop at iterates whose recovered velocities differ by ~200 x tol.  The stop
# rule itself is re-verified from scratch on the merged solution for every case (check_distributed).
# The shrunk scene has a sliver face whose mass weight sits at the 0.01 clamp (S_CMB: M_c^-1 up to 100 / rho): the recovered velocity
# there amplifies the CG stopping difference a hundredfold, so that case solves to 1e-7 and is compared at 1e-3 (measured 1.4e-4; a wrong
# halo or a stale table shows up as O(1)).
DIST_VEL_GATE = {"blob_40x36x96_tile32_pad3": 1e-3, "blob64_tile16_then_shrunk": 1e-3}


def empty_scene():
    """No liquid at all: every count is 0, the solve is trivially successful."""
    sc = scenes.box_scene(16, doReduced=1)
    sc.surface[...] = 1.0
    return sc


def rel(a, b):
    if a.size == 0:
        return 0.0
    return float(np.abs(a - b).max() / max(float(np.abs(a).max()), 1e-300))


def check_classification(o, s):
    for k in COUNTS:
        assert o.count(k) == s.count(k), f"count {k}: oracle {o.count(k)} vs {s.count(k)}"
    for slot in range(7):
        for liquid in (1, 0):
            assert np.array_equal(o.weight_field(liquid, slot), s.weight_field(liquid, slot)), f"weights slot {slot} liquid {liquid}"
        for kind, name in ((0, "labels"), (1, "active"), (2, "reduced")):
            a, b = o.index_field(kind, slot), s.index_field(kind, slot)
            assert np.array_equal(a, b.astype(np.int64)), f"{name} field of slot {slot}: {(a != b).sum()} of {a.size} differ"


def check_matrices(o, s):
    for m in BITEXACT_MATS + TOL_MATS:
        so, po, io, vo = o.csr(m)
        ss, ps_, is_, vs = s.csr(m)
        assert tuple(so) == tuple(ss), f"{m} shape"
        assert np.array_equal(po, ps_) and np.array_equal(io, is_), f"{m} sparsity pattern differs"
        if m in BITEXACT_MATS:
            assert np.array_equal(vo, vs), f"{m} values not bit-equal (rel {rel(vo, vs):.2e})"
        else:
            assert rel(vo, vs) <= 1e-8, f"{m} values rel {rel(vo, vs):.2e}"
    for v in ["activeRHS", "pressureRHS", "stressRHS", "com"]:
        assert np.array_equal(o.vector(v), s.vector(v)), f"{v} not bit-equal"
    for v, tol in (("reducedRHS", 1e-8), ("bestFit", 1e-6), ("MrDense", 1e-8), ("ViscDense", 1e-8), ("BinvDense", 1e-8), ("b", 1e-10)):
        assert rel(o.vector(v), s.vector(v)) <= tol, f"{v} rel {rel(o.vector(v), s.vector(v)):.2e}"


# Per-region, per-entry gates of the dense region blocks.  A global max|diff| / max|ref| is blind to the small entries: the high-order
# moments are ~ (region size / domain)^4 below the largest entry, so an O(1) error in them, or in a whole small region, passes it.
# Measured with the host-emulation twin against the oracle: Mr / Visc <= 3.4e-13, B^-1 <= 2.7e-13, bestFit <= 1.5e-12.
REGION_GATES = {"MrDense": 1e-11, "ViscDense": 1e-11, "BinvDense": 1e-10, "bestFit": 1e-9}


def _ratio(diff, den):
    """diff / den, where den == 0 demands diff == 0 exactly (inf otherwise)."""
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(den > 0, diff / np.where(den > 0, den, 1.0), np.where(diff == 0, 0.0, np.inf))


def region_block_errors(ref, got, R):
    """Worst error of each region quantity in the unit of its gate.  `ref(name)` / `got(name)` return the flat vectors.
    MrDense / ViscDense: |dM_ij| / sqrt(M_ii M_jj), with the block's largest diagonal where M_ii or M_jj is 0.
    BinvDense / bestFit: max|diff| / max|ref| of each region separately."""
    err = {}
    if R == 0:
        return {v: 0.0 for v in REGION_GATES}
    for v in ("MrDense", "ViscDense"):
        a, b = ref(v).reshape(R, 26, 26), got(v).reshape(R, 26, 26)
        d = np.abs(np.einsum("rii->ri", a))
        den = np.sqrt(d[:, :, None] * d[:, None, :])
        den = np.where(den > 0, den, d.max(axis=1)[:, None, None])
        err[v] = float(_ratio(np.abs(a - b), den).max())
    for v in ("BinvDense", "bestFit"):
        a, b = ref(v).reshape(R, -1), got(v).reshape(R, -1)
        err[v] = float(_ratio(np.abs(a - b).max(axis=1), np.abs(a).max(axis=1)).max())
    return err


def check_region_blocks(o, s):
    R = o.count("regionCount")
    err = region_block_errors(o.vector, s.vector, R)
    for v, gate in REGION_GATES.items():
        assert err[v] <= gate, f"{v}: worst per-region error {err[v]:.2e} > {gate:.0e}"
    return err


# Componentwise gate of an apply against the factored scipy evaluation, in units of the factored bound.  Measured on the emulation
# twin: <= 2.0e-15 (the one-region scene), 5e-16 on the tiled ones; an error of one lost row is O(1).
OPERATOR_GATE = 1e-13


def operator_error(y, Ax, bound):
    """Componentwise error of an apply: max |y_i - (Ax)_i| / (|A||x|)_i, where a row with bound 0 must be exactly 0."""
    return float(_ratio(np.abs(y - Ax), bound).max()) if y.size else 0.0


def scipy_operator(csr, dt):
    """A = -dt K^T Mc^-1 K - J^T B^-1 J - 1/2 [0, 0; 0, mu^-1] by scipy.sparse from the component matrices `csr(name)`."""
    import scipy.sparse as sp
    M = {}
    for name in ("McInv", "BInv", "uInv", "G", "JG", "Dt", "JDt"):
        shape, ptr, idx, val = csr(name)
        M[name] = sp.csr_matrix((val, idx, ptr), shape=shape)
    K = sp.hstack([M["G"], M["Dt"]]).tocsr(); J = sp.hstack([M["JG"], M["JDt"]]).tocsr()
    nP = M["G"].shape[1]
    C22 = sp.block_diag([sp.csr_matrix((nP, nP)), M["uInv"]]).tocsr()
    return (-dt * (K.T @ M["McInv"] @ K) - J.T @ M["BInv"] @ J - 0.5 * C22).tocsr()


def scipy_factored(csr, dt):
    """The same A kept factored: returns (A x, bound) for a given x, where bound = (dt |K|^T |Mc^-1| |K| + |J|^T |B^-1| |J|
    + 1/2 |C22|) |x| is the componentwise rounding scale of evaluating A x through its factors.  A region without tiles couples
    every one of its DOFs to every other: its explicit J^T B^-1 J holds ~ 10^9 entries, the factors 10^6."""
    import scipy.sparse as sp
    M = {}
    for name in ("McInv", "BInv", "uInv", "G", "JG", "Dt", "JDt"):
        shape, ptr, idx, val = csr(name)
        M[name] = sp.csr_matrix((val, idx, ptr), shape=shape)
    K = sp.hstack([M["G"], M["Dt"]]).tocsr(); J = sp.hstack([M["JG"], M["JDt"]]).tocsr()
    nP = M["G"].shape[1]
    C22 = sp.block_diag([sp.csr_matrix((nP, nP)), M["uInv"]]).tocsr()
    KT, JT = K.T.tocsr(), J.T.tocsr()
    aK, aKT, aJ, aJT, aMc, aB, aC = abs(K), abs(KT), abs(J), abs(JT), abs(M["McInv"]), abs(M["BInv"]), abs(C22)

    def apply(x):
        y = -dt * (KT @ (M["McInv"] @ (K @ x))) - JT @ (M["BInv"] @ (J @ x)) - 0.5 * (C22 @ x)
        ax = np.abs(x)
        bound = dt * (aKT @ (aMc @ (aK @ ax))) + aJT @ (aB @ (aJ @ ax)) + 0.5 * (aC @ ax)
        return y, bound
    return apply


def check_operator(o, s, seed=0):
    n = o.count("nSystemSize")
    if n == 0:
        return
    x = np.random.default_rng(seed).standard_normal(n)
    ya, yb = o.apply(x), s.apply(x)
    assert rel(ya, yb) <= 1e-12, f"operator apply rel {rel(ya, yb):.2e}"


def check_solve(sc, o, s, ov):
    ro = o.solve()
    ovel, ovalid = o.writeback()
    rs, vel, valid = s.step_scene(sc)
    assert ro == rs, f"solver result oracle {ro} vs {rs}"
    io, is_ = o.count("iterations"), s.count("iterations")
    assert abs(io - is_) <= max(2, int(0.01 * io)), f"iterations oracle {io} vs {is_}"
    tol = max(10 * dict(sc.params, **ov)["tolerance"], 4e-7)      # the velocity fields are fp32
    for a in range(3):
        assert np.array_equal(ovalid[a], valid[a]), f"valid field axis {a}"
        scale = max(float(np.abs(ovel[a]).max()), 1e-30)
        assert float(np.abs(ovel[a] - vel[a]).max()) <= tol * scale, f"velocity axis {a}"
    # the stop test's x.x is advanced by |x + a p|^2 = x.x + 2a x.p + a^2 p.p instead of being summed (ps_pcg.cu): no drift allowed
    if s.count("usedBiCGStab") == 0 and dict(sc.params, **ov).get("solverType", 0) == 0 and s.count("nSystemSize") > 0:
        x = s.vector("solution")
        xx = float(x @ x)
        assert abs(s.real("xmag") - xx) <= 1e-11 * max(xx, 1e-300), f"x.x recurrence drift {abs(s.real('xmag') - xx) / max(xx, 1e-300):.2e} after {is_} iterations"
    return io, is_


def check_bicgstab_fallback(lib_path=None):
    """solveSPDwithMatrixVectorPCG falls back to BiCGSTAB when CG uses up maxSolverIterations (S.cpp:784-799 ->
    pcg.h:134-200).  (1) Both solvers cut after 8 iterations: the iterates must agree to rounding (BiCGSTAB amplifies
    rounding differences, so the comparison is made early).  (2) A run where the fallback converges: same result code,
    iteration count within 10 % + 2, velocity within the looseness of the reference's stop rule
    min(|e|^2, |e|/|x|) < tol."""
    sc = scenes.blob_scene(32, seed=4, maxIterations=8, tolerance=1e-12, keepNonConvergedResults=1)
    o = Oracle(sc).setup()
    ro = o.solve()
    s = PolyStokesSolver.from_scene(sc, lib_path=lib_path)
    rs, vel, valid = s.step_scene(sc)
    assert ro == rs == 0 and o.count("usedBiCGStab") == s.count("usedBiCGStab") == 1
    assert o.count("iterations") == s.count("iterations") == 8
    assert rel(o.vector("solution"), s.vector("solution")) <= 1e-9, f"BiCGSTAB iterate rel {rel(o.vector('solution'), s.vector('solution')):.2e}"
    ovel, ovalid = o.writeback()
    for a in range(3):   # keepNonConvergedResults: the non-converged field is written back
        assert np.array_equal(ovalid[a], valid[a])
        assert float(np.abs(ovel[a] - vel[a]).max()) <= 4e-7 * max(float(np.abs(ovel[a]).max()), 1e-30)
    s.close()
    sc = scenes.blob_scene(32, seed=4, maxIterations=60)
    o = Oracle(sc, threads=1).setup()        # one thread: the oracle's count moves between 37 and 44 from run to run with OpenMP reductions
    ro = o.solve()
    s = PolyStokesSolver.from_scene(sc, lib_path=lib_path)
    rs, vel, valid = s.step_scene(sc)
    assert ro == rs == 1 and o.count("usedBiCGStab") == s.count("usedBiCGStab") == 1
    io, is_ = o.count("iterations"), s.count("iterations")
    # a chaotic iteration: two correct implementations that round differently land in the same ballpark, not on the same count
    assert abs(io - is_) <= 2 + io // 2, f"BiCGSTAB iterations oracle {io} vs {is_}"
    # BiCGSTAB's trajectory is chaotic at rounding level (the oracle's OpenMP dot products are not even reproducible from run to run)
    # and its stop rule min(|e|^2, |e| / |x|) < tol (pcg.h:186-193) is loose: two correct runs may stop a few iterations apart with
    # velocities that differ by per cents.  What must hold exactly is the rule itself on the returned iterate, checked independently:
    x, b = s.vector("solution"), o.vector("b")
    e = b - o.apply(x)
    rsnew, xmag = float(e @ e), float(np.sqrt(x @ x))
    rre = min(rsnew, np.sqrt(rsnew) / xmag)
    tol = dict(sc.params)["tolerance"]
    assert rre < tol, f"returned BiCGSTAB iterate does not satisfy the reference's stop rule: {rre:.3e} >= {tol:.1e}"
    assert abs(rre - s.real("solveError")) <= 1e-6 * rre + 1e-14, f"reported error {s.real('solveError'):.6e} vs recomputed {rre:.6e}"
    ovel, _ = o.writeback()
    for a in range(3):
        assert float(np.abs(ovel[a] - vel[a]).max()) <= 1e-1 * max(float(np.abs(ovel[a]).max()), 1e-30)
    s.close()


EXPLICIT_CASES = {
    "blob32_tile8": lambda: scenes.blob_scene(32, seed=6, tile=8, pad=1),
    "box20_uniform": lambda: scenes.box_scene(20, doReduced=0),
    "blob20_notile": lambda: scenes.blob_scene(20, seed=3, doTile=0),
    "ragged_30x26x22": lambda: scenes.blob_scene((30, 26, 22), seed=5, tile=8, pad=2),
}


def check_explicit_A(case, lib_path=None, tmpdir=None):
    """Explicit A of assembleSystemPressureStress (S_AS:351-430), built on the device from the factors, against the
    oracle's sparse triple products: sparsity pattern bit-exact (Eigen's structural union incl. the explicit zeros of the
    dense region blocks), values <= 1e-8 (measured ~1e-16), symmetric to rounding, and A x equal to the factored operator."""
    sc = EXPLICIT_CASES[case]()
    o = Oracle(sc).setup()
    o.assemble_explicit_A()
    s = PolyStokesSolver.from_scene(sc, lib_path=lib_path, solverType=1)
    s.setup_scene(sc)
    so, po, io, vo = o.csr("A")
    ss, ps_, is_, vs = s.csr("A")
    assert tuple(so) == tuple(ss)
    assert np.array_equal(po, ps_) and np.array_equal(io, is_), "explicit A: sparsity pattern differs"
    assert rel(vo, vs) <= 1e-8, f"explicit A values rel {rel(vo, vs):.2e}"
    import scipy.sparse as sp
    A = sp.csr_matrix((vs, is_, ps_), shape=ss)
    assert abs(A - A.T).max() <= 1e-12 * abs(A).max()
    x = np.random.default_rng(1).standard_normal(ss[0])
    assert rel(A @ x, s.apply(x)) <= 1e-11, f"explicit A x vs factored apply: {rel(A @ x, s.apply(x)):.2e}"
    if tmpdir is not None and vs.size < 3_000_000:     # exportMatrices with solverType EIGEN writes the explicit matrix (S.cpp:533-541)
        pre = os.path.join(str(tmpdir), "e_")
        s.export(pre, 1)
        o.save_csr("A", pre + "oracle_A.mtx")
        ha, hb = open(pre + "Mat_A.mtx").readlines(), open(pre + "oracle_A.mtx").readlines()
        assert ha[:2] == hb[:2] and len(ha) == len(hb), "Mat_A.mtx header / entry count"
        assert [l.split()[:2] for l in ha[2:200]] == [l.split()[:2] for l in hb[2:200]]
    s.close()


def check_eigen_cg(lib_path=None, warm=1, scene=None):
    """solverType EIGEN (S.cpp:814-862): Eigen's CG with the Jacobi preconditioner, started from guessVector
    (useWarmStart, S.cpp:521-531).  The oracle runs it on the explicit A (S_AS:381-397); the library keeps A factored
    and forms only diag(A).  Gates: guess <= 1e-10, diag(A) <= 1e-10 against the explicit matrix, same result code,
    iterations within max(2, 1 %), Eigen's error estimate within 5 %, velocity within 10 * tol."""
    sc = scene or scenes.blob_scene(32, seed=6, tile=8, pad=1, tolerance=1e-5)
    o = Oracle(sc).setup()
    o.assemble_explicit_A()
    if warm:
        o.construct_guess()
    s = PolyStokesSolver.from_scene(sc, lib_path=lib_path, solverType=1, useWarmStart=warm)
    s.setup_scene(sc)
    n = o.count("nSystemSize")
    og = o.vector("guess") if warm else np.zeros(n)
    assert rel(og, s.vector("guess")) <= 1e-10, f"guess rel {rel(og, s.vector('guess')):.2e}"
    assert (np.abs(og).max() > 0) == bool(warm)
    A = o.scipy_csr("A")
    assert rel(A.diagonal(), s.vector("diagA")) <= 1e-10, f"diag(A) rel {rel(A.diagonal(), s.vector('diagA')):.2e}"
    ro = o.solve_eigen_cg()
    ovel, ovalid = o.writeback()
    rs, vel, valid = s.step_scene(sc)
    assert ro == rs == 1, f"solver result oracle {ro} vs {rs}"
    io, is_ = o.count("iterations"), s.count("iterations")
    assert abs(io - is_) <= max(2, int(0.01 * io)), f"iterations oracle {io} vs {is_}"
    assert abs(o.real("solveError") - s.real("solveError")) <= 0.05 * o.real("solveError"), f"error {o.real('solveError')} vs {s.real('solveError')}"
    tol = max(10 * sc.params["tolerance"], 4e-7)
    for a in range(3):
        assert np.array_equal(ovalid[a], valid[a])
        scale = max(float(np.abs(ovel[a]).max()), 1e-30)
        assert float(np.abs(ovel[a] - vel[a]).max()) <= tol * scale, f"velocity axis {a}: {float(np.abs(ovel[a] - vel[a]).max()) / scale:.2e}"
    s.close()
    return io, is_


def run_case(name, lib_path=None, solve=True):
    sc, ov = SCENE_CASES[name]()
    o = Oracle(sc, **ov).setup()
    s = PolyStokesSolver.from_scene(sc, lib_path=lib_path, **ov)
    s.setup_scene(sc)
    check_classification(o, s)
    check_matrices(o, s)
    check_region_blocks(o, s)
    check_operator(o, s)
    if solve:
        check_solve(sc, o, s, ov)
    s.close()
    return o


_DIST_REF = {}


def dist_reference(case):
    """The oracle set up on a distributed case and its factored scipy apply (the last case asked for is kept, so that the probes written
    before a run and the comparison after it share one setup)."""
    if case not in _DIST_REF:
        _DIST_REF.clear()
        sc, ov = DIST_CASES[case]()
        o = Oracle(sc, **ov).setup()
        _DIST_REF[case] = dict(sc=sc, ov=ov, o=o, apply=scipy_factored(o.csr, sc.dt), probes=None)
    return _DIST_REF[case]


def apply_inputs(n):
    """x1, x2 of the applies of the distributed workers (tests/dist_worker.py)."""
    return np.random.default_rng(0).standard_normal(n), np.random.default_rng(1).standard_normal(n)


PROBE_REGIONS = 8


def write_region_probes(case, outdir):
    """Inputs that isolate single regions: x_r is non-zero only on the DOFs region r couples (the columns of its rows of J), for up to
    PROBE_REGIONS regions spread over the id range (every region of a small scene).  With a random x over many regions, an error in one
    region's sum hides behind the rounding scale of a looser row; A x_r is checked componentwise on its own.  Written to
    <outdir>/probes.npz with the rows where the factored bound of A x_r is non-zero; the workers apply each input and report those rows
    (and how many entries elsewhere are non-zero)."""
    import scipy.sparse as sp
    ref = dist_reference(case)
    o = ref["o"]
    R, n = o.count("regionCount"), o.count("nSystemSize")
    if R == 0:
        return
    J = sp.hstack([o.scipy_csr("JG"), o.scipy_csr("JDt")]).tocsr()
    regions = np.unique(np.linspace(0, R - 1, min(R, PROBE_REGIONS)).round().astype(np.int64))
    rng = np.random.default_rng(2)
    out, probes = {"regions": regions}, []
    for i, r in enumerate(regions):
        cols = np.unique(J[26 * r:26 * (r + 1)].indices)
        x = np.zeros(n)
        x[cols] = rng.standard_normal(cols.size)
        Ax, bound = ref["apply"](x)
        rows = np.nonzero(bound)[0]
        probes.append((int(r), Ax[rows], bound[rows]))
        out.update({f"cols{i}": cols, f"vals{i}": x[cols], f"rows{i}": rows})
    ref["probes"] = probes
    np.savez(os.path.join(str(outdir), "probes.npz"), **out)


def check_distributed(case, ranks):
    """`ranks`: per-rank result dicts written by tests/dist_worker.py (or the GPU twin); merged and compared with the oracle."""
    ref = dist_reference(case)
    _DIST_REF.pop(case)           # the solve below changes the oracle's state
    sc, ov, o = ref["sc"], ref["ov"], ref["o"]
    world = len(ranks)
    cuts = list(ranks[0]["cuts"])
    assert cuts[0] == 0 and cuts[-1] == sc.nz and all(b > a and a % 16 == 0 for a, b in zip(cuts[:-1], cuts[1:]))
    def own(arr, r):      # the layers of a grid field rank r is responsible for: its slab; the last slab takes a slot's extra top layer
        lo, hi = int(r["zlo"]), int(r["zhi"])
        return arr[lo:(hi if hi < sc.nz else arr.shape[0])]
    for r in ranks:
        assert int(r["nranks"]) == world and list(r["cuts"]) == cuts
        # global counts and the global numbering are bit-exact on every rank: on its own slab with slab-local setup (the fields of the other
        # slabs are not computed there), everywhere with replicated setup -- the slabs together cover the grid
        for k in COUNTS:
            assert o.count(k) == int(r["count_" + k]), f"rank {int(r['rank'])} count {k}"
        for slot in range(7):
            for kind, name in ((0, "labels"), (1, "active"), (2, "reduced")):
                assert np.array_equal(own(o.index_field(kind, slot), r), own(r[f"{name}{slot}"].astype(np.int64), r)), f"{name} slot {slot} on rank {int(r['rank'])}"
    # every global vector is the sum of the ranks' shares
    tot = lambda key: sum(r[key] for r in ranks)
    assert rel(o.vector("b"), tot("vec_b")) <= 1e-10, f"b rel {rel(o.vector('b'), tot('vec_b')):.2e}"
    assert rel(o.vector("reducedRHS"), tot("vec_reducedRHS")) <= 1e-8, f"reducedRHS rel {rel(o.vector('reducedRHS'), tot('vec_reducedRHS')):.2e}"
    # the region blocks, region by region and entry by entry (each region is reported by its owner only)
    R = o.count("regionCount")
    blk = region_block_errors(o.vector, lambda v: tot("vec_" + v), R)
    for v, gate in REGION_GATES.items():
        assert blk[v] <= gate, f"{v}: worst per-region error {blk[v]:.2e} > {gate:.0e} on {world} ranks"
    # the operator, componentwise against the factored scipy evaluation; and bit for bit the same apply(x1) on every rank after other
    # applies (an odd and an even number of them, so either parity of the peer moment area) and after the step
    n = o.count("nSystemSize")
    op = probe = 0.0
    if n:
        for key, x in zip(("apply", "apply_x2"), apply_inputs(n)):
            Ax, bound = ref["apply"](x)
            e = operator_error(tot(key), Ax, bound)
            assert e <= OPERATOR_GATE, f"{key}: componentwise error {e:.2e} > {OPERATOR_GATE:.0e} on {world} ranks"
            op = max(op, e)
        for r in ranks:
            assert bool(r["apply_stable"]), f"rank {int(r['rank'])}: apply(x1) is not bit-identical after other applies and after the step"
    if ref["probes"] is not None:
        for i, (region, Ax, bound) in enumerate(ref["probes"]):
            assert int(tot(f"probe{i}_outside")) == 0, f"A x of region {region}'s DOFs is non-zero where the factored bound is 0"
            e = operator_error(tot(f"probe{i}"), Ax, bound)
            assert e <= OPERATOR_GATE, f"A x of region {region}'s DOFs: componentwise error {e:.2e} > {OPERATOR_GATE:.0e} on {world} ranks"
            probe = max(probe, e)
    print(f"{case} on {world} ranks: {R} regions, componentwise apply error {op:.1e}, single-region inputs {probe:.1e}; worst per-region "
          + ", ".join(f"{v} {blk[v]:.1e}" for v in REGION_GATES), flush=True)
    ro = o.solve()
    ovel, ovalid = o.writeback()
    its = [int(r["iterations"]) for r in ranks]
    assert all(int(r["rc"]) == ro for r in ranks) and len(set(its)) == 1, f"results {[int(r['rc']) for r in ranks]} iterations {its} (oracle {ro})"
    io = o.count("iterations")
    assert abs(io - its[0]) <= max(2, int(0.01 * io)), f"iterations oracle {io} vs {its[0]}"
    # the reference's stop rule min(rr, rr / xx) < tol^2 (pcg.h:316-325), recomputed from scratch on the merged solution with the ORACLE's operator
    if n and ro == 1:
        x, b = tot("solution"), o.vector("b")
        e = b - o.apply(x)
        rr, xx = float(e @ e), float(x @ x)
        t2 = dict(sc.params, **ov)["tolerance"] ** 2
        got = min(rr, rr / max(xx, 1e-300))      # slack 1.5: the solver tests its recursively updated residual, this is the true one
        assert got < 1.5 * t2, f"merged solution does not satisfy the stop rule: {got:.3e} >= {t2:.1e}"
    tol = DIST_VEL_GATE.get(case, max(10 * dict(sc.params, **ov)["tolerance"], 4e-7))      # the velocity fields are fp32
    for a in range(3):
        merged = np.empty_like(ovel[a])
        for r in ranks:
            lo, hi = int(r["zlo"]), int(r["zhi"])
            assert np.array_equal(own(r[f"valid{a}"], r), own(ovalid[a], r)), f"valid axis {a} rank {int(r['rank'])}"
            own(merged, r)[...] = own(r[f"vel{a}"], r)       # a rank delivers its slab (the last one the top plane too)
        scale = max(float(np.abs(ovel[a]).max()), 1e-30)
        assert float(np.abs(ovel[a] - merged).max()) <= tol * scale, f"velocity axis {a}: {float(np.abs(ovel[a] - merged).max()) / scale:.2e}"
    assert all(bool(r["repeat_ok"]) for r in ranks), "second step on the same handle differs"
    if case in DIST_NEXT:
        sc2 = DIST_NEXT[case]()
        o2 = Oracle(sc2, **ov).setup()
        ro2 = o2.solve()
        ovel2, ovalid2 = o2.writeback()
        assert o2.count("nSystemSize") != o.count("nSystemSize"), "the second scene must change the system size"
        for r in ranks:
            assert int(r["next_rc"]) == ro2 and int(r["next_nSystemSize"]) == o2.count("nSystemSize") and int(r["next_regionCount"]) == o2.count("regionCount")
            assert abs(int(r["next_iterations"]) - o2.count("iterations")) <= max(2, o2.count("iterations") // 100)
        for a in range(3):
            merged = np.empty_like(ovel2[a])
            for r in ranks:
                assert np.array_equal(own(r[f"next_valid{a}"], r), own(ovalid2[a], r)), f"second scene: valid axis {a} rank {int(r['rank'])}"
                own(merged, r)[...] = own(r[f"next_vel{a}"], r)
            scale = max(float(np.abs(ovel2[a]).max()), 1e-30)
            assert float(np.abs(ovel2[a] - merged).max()) <= tol * scale, f"second scene: velocity axis {a}: {float(np.abs(ovel2[a] - merged).max()) / scale:.2e}"
    return io, its[0]

"""The reference's OWN classifier and matrix-block construction -- exec/HDK_PolyStokesSolver_Classifier.cpp and
exec/HDK_PolyStokesSolver_ConstructMatrixBlocks.cpp compiled unmodified from /root/reference into oracle/_ref/libps_ref_classify.so
(oracle/Makefile `ref`; HDK stand-in oracle/hdk_shim, Eigen facade oracle/eigen_facade, harness oracle/ref_classify.cpp) -- against
(a) the oracle's restatement and (b) the product, on the same integration weights.  Labels, the active (DOF) indices, the reduced
region indices of all 7 sample slots, the counts and the valid-face fields must be BIT-EXACT, and so must the sparsity patterns
(explicit zeros included) of M_c, M_c^-1, mu, mu^-1, G, D^T, JG, JD^T and the three right-hand sides; values bit-equal for the oracle.
This is what pins SURVEY.md section 8a rows C1-C12 and M1-M9 to reference CODE (on the HDK semantics of BASELINE.md section 3) instead
of to a reading of it.
The library is built from a checkout of the reference's sources, which is not part of this repository; without it these tests skip.
The *_matches_oracle tests make the product-side checks against the oracle's classification, blocks and assembly of the same scene, on the
oracle's own weights (bit-equal to the product's: tests/test_ref_full.py): they do not compare with the reference themselves."""
import numpy as np
import pytest

import parity
from oracle import oracle as orc
from oracle import ref_classify
from oracle.oracle import Oracle
from polystokes_b200 import PolyStokesSolver, scenes

needs_reference = pytest.mark.skipif(not ref_classify.available(), reason="oracle/_ref/libps_ref_classify.so not built (needs the reference's sources)")

KINDS = ("labels", "active indices", "reduced indices")
CASES = dict(parity.SCENE_CASES)
CASES.update({
    "S1_uniform_64": lambda: (scenes.scene_s1(), {}),
    "S2_beam_64_tile8_pad1": lambda: (scenes.scene_s2(64), {}),
    "S3_jet_64_tile16_pad2": lambda: (scenes.scene_s3(64), {}),
    "S4_pool_80_tile32_pad3_layers33": lambda: (scenes.scene_s4(80), {}),
    "S5_blob_quarter_tile8_pad3": lambda: (scenes.scene_s5(0.25, tileSize=8), {}),
    "blob48_pad0": lambda: (scenes.blob_scene(48, seed=13, tile=8, pad=0), {}),
    "blob40_layers14": lambda: (scenes.blob_scene(40, seed=17, tile=8, pad=1, liquidLayers=1, solidLayers=4), {}),
})


EMULATED = ["tiles8pad1_box40", "blob40_layers31", "blob_ragged_36x44x52", "blob40_notile", "blob33_uniform", "S2_beam_64_tile8_pad1"]
GPU_CASES = list(CASES) + ["S3_jet_112_tile16_pad2"]


def _gpu_case(case):
    return (scenes.scene_s3(112), {}) if case == "S3_jet_112_tile16_pad2" else CASES[case]()


BLOCKS = ("Mc", "McInv", "u", "uInv", "G", "Dt", "JG", "JDt")
RHS = ("activeRHS", "pressureRHS", "stressRHS")


class _OracleClassifier:
    """The oracle's classification, blocks and assembly of a scene (computed on setup, from its own weights) behind the accessors of
    ref_classify.RefClassifier; construct_blocks / assemble have nothing left to do."""

    def __init__(self, sc, prm, solver_type=0):
        self.o = Oracle(sc, **prm).setup()
        if solver_type:
            self.o.assemble_explicit_A()

    def results(self):
        _, valid = self.o.writeback()        # buildValidFaces only needs the labels: no solve
        fields = [[self.o.index_field(kind, slot) for slot in range(7)] for kind in range(3)]
        return fields, {k: self.o.count(k) for k in ref_classify.COUNT_NAMES}, valid

    def construct_blocks(self, *args):
        pass

    def assemble(self, *args):
        pass

    def csr(self, name):
        return self.o.csr(name)

    def vector(self, name):
        return self.o.vector(name)


def _check(sc, ov, fields_of, weight_field, counts_of, valid_of=None, csr_of=None, vector_of=None, exact_values=BLOCKS, asm_tol=1e-13, oracle=False):
    """The reference code's classifier run on `weight_field`, or with oracle=True the oracle's own classification of the scene, against
    the caller's fields / counts / valid faces / blocks / assembly."""
    prm = dict(sc.params, **ov)
    if oracle:
        R, who = _OracleClassifier(sc, prm), "the oracle's"
    else:
        R, who = ref_classify.RefClassifier(sc.nx, sc.ny, sc.nz, sc.dx, sc.dt, prm, weight_field, density=sc.density), "the reference code's"
    fields, counts, valid = R.results()
    if csr_of is not None and counts["nCenter"] > 0:
        # constructMatrixBlocks of the reference on its own classification; centres of mass and basis evaluation supplied (ref_classify.cpp)
        R.construct_blocks(sc.vel, sc.colvel, sc.viscosity, vector_of("com").reshape(-1, 3), ref_classify.oracle_coeff_fn())
        for m in BLOCKS:
            (sr, pr, ir, vr), (sm, pm, im, vm) = R.csr(m), csr_of(m)
            assert tuple(sr) == tuple(sm), f"{m}: shape {sm} vs {who} {sr}"
            assert np.array_equal(pr, pm) and np.array_equal(ir, im), f"{m}: sparsity pattern differs from {who}"
            if m in exact_values:
                assert np.array_equal(vr, vm), f"{m}: values not bit-equal to {who} (rel {parity.rel(vr, vm):.2e})"
            else:
                assert parity.rel(vr, vm) <= 1e-8, f"{m}: values rel {parity.rel(vr, vm):.2e}"
        for v in RHS:
            assert np.array_equal(R.vector(v), vector_of(v)), f"{v} not bit-equal to {who}"
        # assemble() of the reference (AssembleBlocks.cpp + AssembleSystem.cpp) on the caller's region matrices (D3-D5 are not compiled)
        R.assemble(vector_of("MrDense"), vector_of("ViscDense"), vector_of("bestFit"))
        for m in ("Mr", "B", "BInv"):
            (sr, pr, ir, vr), (sm, pm, im, vm) = R.csr(m), csr_of(m)
            assert tuple(sr) == tuple(sm) and np.array_equal(pr, pm) and np.array_equal(ir, im), f"{m}: pattern differs from {who}"
            assert parity.rel(vr, vm) <= asm_tol, f"{m}: values rel {parity.rel(vr, vm):.2e} vs {who}"
        assert parity.rel(R.vector("reducedRHS"), vector_of("reducedRHS")) <= asm_tol
        assert parity.rel(R.vector("b"), vector_of("b")) <= max(asm_tol, 1e-12), f"b rel {parity.rel(R.vector('b'), vector_of('b')):.2e} vs {who}"
    for kind in range(3):
        for slot in range(7):
            mine = np.asarray(fields_of(kind, slot)).astype(np.int64)
            assert np.array_equal(fields[kind][slot], mine), f"{KINDS[kind]} slot {slot}: {np.count_nonzero(fields[kind][slot] != mine)} of {mine.size} entries differ from {who} classification"
    for k, v in counts.items():
        if k == "regionCount" and not prm["doReduced"]:
            continue
        assert v == counts_of(k), f"{k}: {who} classification {v}, here {counts_of(k)}"
    if valid_of is not None:
        for a in range(3):
            assert np.array_equal(valid[a], np.asarray(valid_of(a), dtype=np.float32)), f"valid faces axis {a}"
    return counts


@needs_reference
@pytest.mark.parametrize("case", list(CASES))
def test_oracle_classification_matches_reference_code(built, case):
    sc, ov = CASES[case]()
    o = Oracle(sc, **ov).setup()
    _, ovalid = o.writeback()        # buildValidFaces only needs the labels: no solve
    counts = _check(sc, ov, o.index_field, o.weight_field, o.count, lambda a: ovalid[a], o.csr, o.vector)
    if case not in ("empty_air",):
        assert counts["nCenter"] > 0


EXPLICIT = {"blob32_tile8": lambda: scenes.blob_scene(32, seed=6, tile=8, pad=1, solverType=1), "box20_uniform": lambda: scenes.box_scene(20, doReduced=0, solverType=1),
            "blob24_notile": lambda: scenes.blob_scene(24, seed=8, doTile=0, solverType=1)}


def _explicit_A(sc, weight_field, csr_of, vector_of, tol, oracle=False):
    """assembleSystemPressureStress (S_AS:351-430, solverType EIGEN): the explicit A from the reference's own sparse triple products
    (with oracle=True: the oracle's explicit A of the scene)."""
    if oracle:
        R, who = _OracleClassifier(sc, sc.params, solver_type=1), "the oracle's"
    else:
        R, who = ref_classify.RefClassifier(sc.nx, sc.ny, sc.nz, sc.dx, sc.dt, sc.params, weight_field, density=sc.density, solver_type=1), "the reference code's"
    R.construct_blocks(sc.vel, sc.colvel, sc.viscosity, vector_of("com").reshape(-1, 3), ref_classify.oracle_coeff_fn())
    R.assemble(vector_of("MrDense"), vector_of("ViscDense"), vector_of("bestFit"))
    (sr, pr, ir, vr), (sm, pm, im, vm) = R.csr("A"), csr_of("A")
    assert tuple(sr) == tuple(sm) and np.array_equal(pr, pm) and np.array_equal(ir, im), f"explicit A: sparsity pattern (explicit zeros included) differs from {who}"
    assert parity.rel(vr, vm) <= tol, f"explicit A values rel {parity.rel(vr, vm):.2e}"
    assert parity.rel(R.vector("b"), vector_of("b")) <= max(tol, 1e-12)


@needs_reference
@pytest.mark.parametrize("case", list(EXPLICIT))
def test_oracle_explicit_A_matches_reference_code(built, case):
    sc = EXPLICIT[case]()
    o = Oracle(sc).setup()
    o.assemble_explicit_A()
    _explicit_A(sc, o.weight_field, o.csr, o.vector, 1e-13)


@needs_reference
@pytest.mark.parametrize("case", list(EXPLICIT))
def test_emulated_explicit_A_matches_reference_code(built, case):
    sc = EXPLICIT[case]()
    s = PolyStokesSolver.from_scene(sc, lib_path=parity.EMUL_LIB)
    s.setup_scene(sc)
    _explicit_A(sc, s.weight_field, s.csr, s.vector, 1e-9)
    s.close()


@needs_reference
@pytest.mark.gpu
@pytest.mark.parametrize("case", list(EXPLICIT))
def test_gpu_explicit_A_matches_reference_code(built, case):
    sc = EXPLICIT[case]()
    s = PolyStokesSolver.from_scene(sc)
    s.setup_scene(sc)
    _explicit_A(sc, s.weight_field, s.csr, s.vector, 1e-9)
    s.close()


@needs_reference
@pytest.mark.parametrize("case", EMULATED)
def test_emulated_classification_matches_reference_code(built, case):
    sc, ov = CASES[case]()
    s = PolyStokesSolver.from_scene(sc, lib_path=parity.EMUL_LIB, **ov)
    rc, vel, valid = s.step_scene(sc)
    _check(sc, ov, s.index_field, s.weight_field, s.count, lambda a: valid[a], s.csr, s.vector, exact_values=parity.BITEXACT_MATS, asm_tol=1e-9)
    s.close()


@needs_reference
@pytest.mark.gpu
@pytest.mark.parametrize("case", GPU_CASES)
def test_gpu_classification_matches_reference_code(built, case):
    """The CUDA classifier on ITS OWN weights against the reference classifier run on those weights."""
    sc, ov = _gpu_case(case)
    s = PolyStokesSolver.from_scene(sc, **ov)
    rc, vel, valid = s.step_scene(sc)
    _check(sc, ov, s.index_field, s.weight_field, s.count, lambda a: valid[a], s.csr, s.vector, exact_values=parity.BITEXACT_MATS, asm_tol=1e-9)
    s.close()


@pytest.mark.parametrize("case", list(EXPLICIT))
def test_emulated_explicit_A_matches_oracle(built, case):
    sc = EXPLICIT[case]()
    s = PolyStokesSolver.from_scene(sc, lib_path=parity.EMUL_LIB)
    s.setup_scene(sc)
    _explicit_A(sc, s.weight_field, s.csr, s.vector, 1e-9, oracle=True)
    s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(EXPLICIT))
def test_gpu_explicit_A_matches_oracle(built, case):
    sc = EXPLICIT[case]()
    s = PolyStokesSolver.from_scene(sc)
    s.setup_scene(sc)
    _explicit_A(sc, s.weight_field, s.csr, s.vector, 1e-9, oracle=True)
    s.close()


@pytest.mark.parametrize("case", EMULATED)
def test_emulated_classification_matches_oracle(built, case):
    sc, ov = CASES[case]()
    s = PolyStokesSolver.from_scene(sc, lib_path=parity.EMUL_LIB, **ov)
    rc, vel, valid = s.step_scene(sc)
    _check(sc, ov, s.index_field, s.weight_field, s.count, lambda a: valid[a], s.csr, s.vector, exact_values=parity.BITEXACT_MATS, asm_tol=1e-9, oracle=True)
    s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", GPU_CASES)
def test_gpu_classification_matches_oracle(built, case):
    """The CUDA classifier, blocks and assembly against the oracle's of the same scene (each on its own, bit-equal, weights)."""
    sc, ov = _gpu_case(case)
    s = PolyStokesSolver.from_scene(sc, **ov)
    rc, vel, valid = s.step_scene(sc)
    _check(sc, ov, s.index_field, s.weight_field, s.count, lambda a: valid[a], s.csr, s.vector, exact_values=parity.BITEXACT_MATS, asm_tol=1e-9, oracle=True)
    s.close()

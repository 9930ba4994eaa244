"""The CG loop iteration by iteration against a plain CG.

The library does not run CG the way pcg.h:268-340 states it (ps_pcg.cu, above cg_rre2): beta and the stop test's r.r come from
|r - alpha Ap|^2 = r.r - 2 alpha r.Ap + alpha^2 Ap.Ap, x.x from the previous update's x.p and p.p, every dot product is a fixed-order
sum of CTA partials finished by the last CTA, and with several ranks the sums are all-reduced inside the kernels.  A wrong alpha or beta
still converges (an inexact line search), so whole solves do not see such a bug; the iterates do.  ps_time_kernel("cg_iteration", k)
runs exactly k iterations from x = 0 with tolerance 0 and no fallback; after it `solution` is x_k, `xmag` the x.x recurrence,
`solveError` sqrt(min(rr, rr / xx)) of the recurrences and `iterations` k.

The reference (`plain_cg`) is pcg.h's loop in its statement order, in numpy on the oracle's factored operator
(parity.scipy_factored) and the library's own b.  Its gates are measured, not guessed.  Two other correct fp64 CGs run beside it, with
every dot product summed in a shuffled order (fixed seed) and an operator that rounds each row as far from the reference as the
library's apply is measured to (perturbed_apply); one of them in pcg.h's form, one in the library's (recurrence_cg).  The farther of
the two at step k (running maximum over the steps <= k) is the yardstick; each gate is GATE_MULT times it (GATE_MULT_LONG at K_LONG),
and never below GATE_FLOOR:
  - x_k against the reference, the pressure part and the stress part separately (max |diff| / max |ref| of each part);
  - x_1 = alpha_0 b: every entry is the library's b times ONE alpha (bit for bit), and that alpha is the reference's;
  - xmag against the reference x_k . x_k, relative;
  - solveError^2 against the reference rre_k, relative to r_{k-1}.r_{k-1} (times rre_k / rr_k when the stop value is rr / xx): the
    recurrence cancels from that scale.
Measured (pytest -s prints the yardsticks and each test's worst error / gate):
  host-emulation twin: x_k yardsticks 2e-16 .. 1e-14 for k <= 21 (6.8e-13 on the 244-unknown scene, which has converged to rounding
  by then), 1e-15 .. 2e-12 at k = 40 (5.6e-10 on the small scene); worst error / gate 0.98 (visc_six_decades), 0.82 on 3 gloo ranks.
  B200 (1000 W power limit): the same yardsticks within a factor of 2 (the apply rounds differently); worst error / gate 0.11 on the
  small scenes, 0.06 on box96_1000_regions (n = 4.5e6, yardstick 3.6e-15 at k = 8), 0.19 on blob64_notile; EIGEN 0.29; fallback
  velocity 0.10.  The multi-GPU cases need >= 2 / 3 devices.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import cg_iterates_worker as W
import edge_cases
import parity
from oracle.oracle import Oracle
from polystokes_b200 import PolyStokesSolver, scenes

HERE = os.path.dirname(os.path.abspath(__file__))

KS = (1, 2, 3, 5, 8, 13, 21)
K_LONG = 40
GATE_MULT = 16.0
GATE_FLOOR = 1e-13
# past k = 21 two correct CGs part as a chaotic function of their rounding (x10 per 5 iterations on blob24_tiled): one sampled
# yardstick is within a small factor of the spread there, so K_LONG has a gate of its own
GATE_MULT_LONG = 64.0

EMUL = pytest.param(parity.EMUL_LIB, id="emul")
CUDA = pytest.param(None, id="cuda", marks=pytest.mark.gpu)

# name -> (scene, what edge of the CG kernels it reaches, predicate on (counts, on the GPU))
SCENES = {
    "blob24_tiled": (lambda: scenes.blob_scene(24, seed=4), "tiled regions; odd nSystemSize (the tail element of the update)",
                     lambda c, gpu: c["regionCount"] > 0 and c["nSystemSize"] % 2 == 1 and (not gpu or c["regionPath"] == 1)),
    "box20_uniform": (lambda: scenes.box_scene(20, doReduced=0), "no reduced rows; odd nSystemSize",
                      lambda c, gpu: c["regionCount"] == 0 and c["nSystemSize"] % 2 == 1),
    "blob24_notile": (lambda: scenes.blob_scene(24, seed=3, doTile=0), "doTile 0: one untiled region; even nSystemSize",
                      lambda c, gpu: c["regionCount"] == 1 and c["nSystemSize"] % 2 == 0),
    "box_10x10x9_tiny": (lambda: scenes.box_scene((10, 10, 9), shell=3, doReduced=0),
                         "fewer than 256 rows in every CG kernel: one CTA, last_block on a grid of 1",
                         lambda c, gpu: c["nSystemSize"] < 256 and c["rows2"] < 256 and c["nRowsExt"] < 256),
    "visc_six_decades": (edge_cases.visc_six_decades, "viscosity over six decades (badly conditioned)", lambda c, gpu: c["regionCount"] > 0),
    "border_blob24": (lambda: edge_cases.border_blob(24, tileSize=8, tilePadding=1), "liquid on the domain faces; even nSystemSize",
                      lambda c, gpu: c["nSystemSize"] % 2 == 0),
}
# the GPU's own scenes: more rows than the resident grids of cg_update_kernel and pass2_kernel hold, > 900 regions (64 lanes), and
# a region of more than 16384 rows (the chunked region kernels)
BIG = {"box96_1000_regions": (lambda: scenes.box_scene(96, liquid_hi_frac=0.95, shell=2, tileSize=8, tilePadding=1),
                              "> 900 regions (reduced_region_kernel with 64 lanes); more rows than the resident grid of the CG kernels",
                              lambda c, gpu: c["regionCount"] > 900 and (not gpu or (c["regionPath"] == 0 and beyond_resident_grid(c)))),
       "blob64_notile": (lambda: scenes.blob_scene(64, seed=3, doTile=0), "doTile 0 with one region of > 16384 rows: the chunked region kernels",
                         lambda c, gpu: c["regionCount"] == 1 and (not gpu or c["regionPath"] == 2))}
BIG_KS = (1, 3, 8)


def beyond_resident_grid(c):
    """The grids of cg_update_kernel and pass2_kernel are the SM count times the resident CTAs of 256 threads per SM (hot_blocks,
    ps_pcg.cu), at most max_threads_per_SM / 256 of them: with more rows than that the grid-stride loops take a second lap and every
    CTA writes a partial."""
    import torch
    p = torch.cuda.get_device_properties(0)
    rows = p.multi_processor_count * (p.max_threads_per_multi_processor // 256) * 256
    return c["nSystemSize"] // 2 > rows and c["rows2"] > rows


# ---- the reference ----------------------------------------------------------------------------------------------------------------
def plain_dot(a, b):
    return float(a @ b)


def shuffled_dot(n, seed=12345):
    perm = np.random.default_rng(seed).permutation(n)
    return lambda a, b: float(np.sum((a * b)[perm]))


def plain_cg(A, b, kmax, dot, keep=()):
    """pcg.h:268-340 with the identity preconditioner from x = 0 for kmax iterations, never stopping.  Returns the lists alpha[k],
    beta[k], rr[k], xx[k], rre[k] (index k = after k iterations; rr[0] = b.b) and the iterates x[k] for k in `keep`."""
    x, r, p = np.zeros_like(b), b.copy(), b.copy()
    rsold = dot(r, r)
    out = dict(alpha=[np.nan], beta=[np.nan], rr=[rsold], xx=[0.0], rre=[np.nan], x={})
    for k in range(1, kmax + 1):
        Ap = A(p)
        alpha = rsold / dot(p, Ap)
        x = x + alpha * p
        r = r - alpha * Ap
        rsnew = dot(r, r)
        xmag = dot(x, x)
        rre = rsnew
        if rsnew / xmag < rre:
            rre = rsnew / xmag
        beta = rsnew / rsold
        p = r + beta * p
        rsold = rsnew
        for key, v in (("alpha", alpha), ("beta", beta), ("rr", rsnew), ("xx", xmag), ("rre", rre)):
            out[key].append(v)
        if k in keep:
            out["x"][k] = x.copy()
    return out


def recurrence_cg(A, b, kmax, dot, keep=()):
    """The same CG in the library's form (ps_pcg.cu, cg_update_kernel): alpha from the summed r.r, the stop test's r.r and beta from
    |r - alpha Ap|^2 = r.r - 2 alpha r.Ap + alpha^2 Ap.Ap, x.x from x.x + 2 alpha x.p + alpha^2 p.p.  Exact in exact arithmetic; in
    fp64 it rounds differently from plain_cg, most where the residual has fallen by orders of magnitude in one step.  Only a yardstick
    here: the library is compared with plain_cg.  Same return value."""
    x, r, p = np.zeros_like(b), b.copy(), b.copy()
    rr = dot(r, r)
    xx, xp, pp = 0.0, 0.0, rr
    out = dict(alpha=[np.nan], beta=[np.nan], rr=[rr], xx=[0.0], rre=[np.nan], x={})
    for k in range(1, kmax + 1):
        Ap = A(p)
        alpha = rr / dot(p, Ap)
        rrNew = (rr - (2.0 * alpha) * dot(r, Ap)) + (alpha * alpha) * dot(Ap, Ap)
        xx = xx + (2.0 * alpha) * xp + (alpha * alpha) * pp
        rre = min(rrNew, rrNew / xx)
        beta = rrNew / rr
        x = x + alpha * p
        r = r - alpha * Ap
        p = r + beta * p
        rr, xp, pp = dot(r, r), dot(x, p), dot(p, p)
        for key, v in (("alpha", alpha), ("beta", beta), ("rr", rrNew), ("xx", xx), ("rre", rre)):
            out[key].append(v)
        if k in keep:
            out["x"][k] = x.copy()
    return out


def jacobi_cg(A, b, x0, k, dot):
    """Eigen's ConjugateGradient with the diagonal preconditioner (ConjugateGradient.h:28-93, as the oracle restates it) for exactly
    k iterations from x0; returns (x_k, sqrt(|r_k|^2 / |b|^2))."""
    d = A.diagonal()
    invdiag = np.where(d != 0, 1.0 / np.where(d != 0, d, 1.0), 1.0)
    x = x0.copy()
    r = b - A @ x
    p = invdiag * r
    absNew = dot(r, p)
    rr = dot(r, r)
    for _ in range(k):
        t = A @ p
        alpha = absNew / dot(p, t)
        x = x + alpha * p
        r = r - alpha * t
        rr = dot(r, r)
        z = invdiag * r
        absOld, absNew = absNew, dot(r, z)
        p = z + (absNew / absOld) * p
    return x, np.sqrt(rr / dot(b, b))


def probe_x(n):
    """The input of the apply whose componentwise error sets the yardstick's operator rounding."""
    return np.random.default_rng(7).standard_normal(n)


def perturbed_apply(apply, amplitude, seed):
    """A x with every entry moved by a random fraction (fixed seed) of `amplitude` times its rounding scale (|A||x|)_i: a second
    correct implementation of the operator that rounds each row differently by up to that much."""
    rng = np.random.default_rng(seed)
    def A(x):
        y, bound = apply(x)
        return y + (amplitude * bound) * rng.uniform(-1.0, 1.0, size=y.size)
    return A


def part_rel(ref, got, nP):
    """(pressure part, stress part) of max |got - ref| / max |ref|."""
    return parity.rel(ref[:nP], got[:nP]), parity.rel(ref[nP:], got[nP:])


def gate(yard, k=1):
    return max((GATE_MULT if k <= max(KS) else GATE_MULT_LONG) * yard, GATE_FLOOR)


class Reference:
    """The oracle set up on one scene; the plain and the shuffled-order CG on its factored operator; per k the gates."""

    def __init__(self, sc, kmax, keep, b, Ax):
        self.sc = sc
        o = self.o = Oracle(sc, threads=1).setup()
        self.n, self.nP = o.count("nSystemSize"), o.count("nPressures")
        # the library's own b: the CG loop is under test here, b is gated against the oracle's elsewhere (parity.check_matrices) and
        # differs from it by a few ulp, which the iteration would amplify like any other perturbation of its start
        assert b.shape == (self.n,) and parity.rel(o.vector("b"), b) <= 1e-10
        self.b = b
        apply = parity.scipy_factored(o.csr, sc.dt)
        A = lambda v: apply(v)[0]
        self.ref = R = plain_cg(A, self.b, kmax, plain_dot, keep)
        # the library's apply of probe_x, componentwise against the factored evaluation (the unit of parity.OPERATOR_GATE)
        self.op_err = parity.operator_error(Ax, *apply(probe_x(self.n)))
        assert self.op_err <= parity.OPERATOR_GATE, f"componentwise apply error {self.op_err:.2e}"
        # two other correct fp64 CGs, with the dot products summed in a shuffled order and an operator that rounds as far from the
        # reference as the library's measured apply does (at least one ulp), one of them in the library's form
        dot, amp = shuffled_dot(self.n), max(self.op_err, np.finfo(np.float64).eps)
        others = [plain_cg(perturbed_apply(apply, amp, 1), self.b, kmax, dot, keep),
                  recurrence_cg(perturbed_apply(apply, amp, 2), self.b, kmax, dot, keep)]
        # yardsticks: the farther of the two, running maxima over the steps so far
        self.yard = {}
        run = np.zeros(5)
        for k in range(1, kmax + 1):
            for S in others:
                now = [abs(R["alpha"][k] - S["alpha"][k]) / abs(R["alpha"][k]), abs(R["xx"][k] - S["xx"][k]) / R["xx"][k],
                       abs(R["rre"][k] - S["rre"][k]) / self.rre_scale(k)]
                now += list(part_rel(R["x"][k], S["x"][k], self.nP)) if k in keep else [0.0, 0.0]
                run = np.maximum(run, now)
            self.yard[k] = dict(zip(("alpha", "xx", "rre", "xP", "xS"), run))

    def rre_scale(self, k):
        R = self.ref
        return R["rr"][k - 1] * R["rre"][k] / R["rr"][k]


_refs = {}


def library_inputs(sc, lib):
    """The library's b and its apply of probe_x."""
    s = PolyStokesSolver.from_scene(sc, lib_path=lib)
    s.setup_scene(sc)
    b = s.vector("b")
    Ax = s.apply(probe_x(b.size))
    s.close()
    return b, Ax


def reference(name, lib, table=None, kmax=K_LONG, keep=KS + (K_LONG,)):
    key = (name, lib, kmax, keep)
    if key not in _refs:
        sc = (table or SCENES)[name][0]()
        _refs[key] = Reference(sc, kmax, keep, *library_inputs(sc, lib))
    return _refs[key]


def hook(s, k):
    s.time_kernel("cg_iteration", k)
    return s.vector("solution"), s.real("xmag"), s.real("solveError"), s.count("iterations")


def check_iterates(where, ref, got, ks, b_lib=None):
    """got: k -> (x_k, xmag, solveError, iterations).  Returns the worst ratio of an error to its gate."""
    R, worst = ref.ref, 0.0
    for k in ks:
        x, xmag, err, its = got[k]
        y = ref.yard[k]
        assert its == k, f"{where}: {its} iterations after asking for {k}"
        for part, e, g in zip(("pressure", "stress"), part_rel(R["x"][k], x, ref.nP), (gate(y["xP"], k), gate(y["xS"], k))):
            assert e <= g, f"{where}: x_{k} {part} part differs from the reference by {e:.2e} (gate {g:.1e})"
            worst = max(worst, e / g)
        e, g = abs(xmag - R["xx"][k]) / R["xx"][k], gate(y["xx"], k)
        assert e <= g, f"{where}: xmag after {k} iterations {xmag!r}, reference x.x {R['xx'][k]!r}: rel {e:.2e} (gate {g:.1e})"
        worst = max(worst, e / g)
        e, g = abs(err * err - R["rre"][k]) / ref.rre_scale(k), gate(y["rre"], k)
        assert e <= g, f"{where}: solveError^2 after {k} iterations {err * err!r}, reference rre {R['rre'][k]!r}: {e:.2e} of r.r (gate {g:.1e})"
        worst = max(worst, e / g)
    if b_lib is not None and 1 in ks:
        worst = max(worst, check_first_iterate(where, ref, got[1][0], b_lib))
    return worst


def check_first_iterate(where, ref, x1, b):
    """x_1 = alpha_0 p_0 with p_0 = b: every entry must be the library's own b times one and the same alpha (pass 2's p.Ap finished
    into ONE value that every CTA of the update read), and that alpha must be the reference's."""
    assert np.array_equal(x1[b == 0], b[b == 0]), f"{where}: x_1 non-zero where b is 0"
    i = int(np.argmax(np.abs(b)))
    a0 = x1[i] / b[i]
    cands = [a0]
    for d in (np.inf, -np.inf):
        a = a0
        for _ in range(3):
            a = np.nextafter(a, d)
            cands.append(a)
    alpha = next((a for a in cands if np.array_equal(a * b, x1)), None)
    assert alpha is not None, (f"{where}: x_1 is not one alpha times b: x_1 / b spans "
                               f"[{np.min(x1[b != 0] / b[b != 0])!r}, {np.max(x1[b != 0] / b[b != 0])!r}]")
    e, g = abs(alpha - ref.ref["alpha"][1]) / abs(ref.ref["alpha"][1]), gate(ref.yard[1]["alpha"])
    assert e <= g, f"{where}: alpha_0 {alpha!r}, reference {ref.ref['alpha'][1]!r}: rel {e:.2e} (gate {g:.1e})"
    return e / g


def _yard_summary(ref, ks):
    return ", ".join(f"k={k}: x {max(ref.yard[k]['xP'], ref.yard[k]['xS']):.1e}" for k in ks)


# ---- fixed-count iterates -----------------------------------------------------------------------------------------------------------
def _run_iterates(lib, name, table, ks):
    ref = reference(name, lib, table, kmax=max(ks), keep=ks) if table is BIG else reference(name, lib)
    sc = ref.sc
    s = PolyStokesSolver.from_scene(sc, lib_path=lib)
    s.setup_scene(sc)
    b_lib = s.vector("b")
    got = {k: hook(s, k) for k in ks}
    worst = check_iterates(f"{name}", ref, got, ks, b_lib)
    # bit for bit: the same calls on a second handle in the opposite order, and the longest run again on the first
    t = PolyStokesSolver.from_scene(sc, lib_path=lib)
    t.setup_scene(sc)
    for k in reversed(ks):
        x, xmag, err, _ = hook(t, k)
        assert np.array_equal(x, got[k][0]) and xmag == got[k][1] and err == got[k][2], f"{name}: x_{k} differs on a second handle"
    t.close()
    x, xmag, err, _ = hook(s, ks[-1])
    assert np.array_equal(x, got[ks[-1]][0]) and xmag == got[ks[-1]][1], f"{name}: x_{ks[-1]} differs when run again"
    # the hook changes P and cgOnly and leaves the tickets mid-count: a step after it equals a fresh handle's step
    rc, vel, valid = s.step_scene(sc)
    f = PolyStokesSolver.from_scene(sc, lib_path=lib)
    rc2, vel2, valid2 = f.step_scene(sc)
    assert rc == rc2 and s.count("iterations") == f.count("iterations") and s.count("usedBiCGStab") == f.count("usedBiCGStab"), \
        f"{name}: the step after the hook: result {rc} / {rc2}, iterations {s.count('iterations')} / {f.count('iterations')}"
    assert np.array_equal(s.vector("solution"), f.vector("solution")), f"{name}: the solution of a step after the hook differs from a fresh handle's"
    for a in range(3):
        assert np.array_equal(vel[a], vel2[a]) and np.array_equal(valid[a], valid2[a]), f"{name}: velocity axis {a} after the hook differs"
    s.close(); f.close()
    print(f"{name}: n {ref.n}, worst error / gate {worst:.2f}; yardsticks {_yard_summary(ref, ks)}")


@pytest.mark.parametrize("lib", [EMUL, CUDA])
@pytest.mark.parametrize("name", list(SCENES))
def test_fixed_count_iterates_match_plain_cg(built, lib, name):
    _run_iterates(lib, name, SCENES, KS + (K_LONG,))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(BIG))
def test_fixed_count_iterates_large_scenes(built, name):
    _run_iterates(None, name, BIG, BIG_KS)


@pytest.mark.parametrize("lib", [EMUL, CUDA])
def test_scenes_reach_the_kernel_edges(built, lib):
    """Each scene must still reach the edge it is here for; a resized scene that stops covering it fails here."""
    gpu = lib is None
    table = dict(SCENES, **BIG) if gpu else SCENES
    for name, (make, what, reaches) in table.items():
        sc = make()
        s = PolyStokesSolver.from_scene(sc, lib_path=lib)
        s.setup_scene(sc)
        c = {k: s.count(k) for k in ("nSystemSize", "regionCount", "nRowsExt", "regionPath", "nCenter", "nEdgeYZ", "nEdgeXZ", "nEdgeXY")}
        c["rows2"] = c["nCenter"] + c["nEdgeYZ"] + c["nEdgeXZ"] + c["nEdgeXY"]
        s.close()
        assert reaches(c, gpu), f"{name} no longer reaches: {what} ({c})"


# ---- the stop test and the poll interval ---------------------------------------------------------------------------------------------
STOP_SCENE = "visc_six_decades"       # its rre_k has a clean new minimum at every target count
FALLBACK_SCENE = "blob24_tiled"
STOP_MAX_IT = 200
STOP_TARGETS = (1, 2, 6, 7, 8, 14, 24, 25, 26, 50)     # near 1, 2, c - 1, c, c + 1, 2 c for c = 7 and the default 25


def stop_tolerances(ref, targets):
    """iteration count -> tolerance: pcg.h stops after iteration m (and reports m) when rre_{m+1} < tol^2 is the first such.  tol^2
    at the geometric midpoint between rre_{m+1} and the smallest rre before it; m moved to the nearest count whose rre_{m+1} is a new
    minimum by more than 1e-6 relative (closer, rounding may decide)."""
    rre = ref.ref["rre"]
    ok = {}
    for m in range(1, len(rre) - 1):
        prev, new = min(rre[1:m + 1]), rre[m + 1]
        if new * (1 + 1e-6) ** 2 < prev:
            ok[m] = np.sqrt(np.sqrt(prev * new))
    out = {}
    for t in targets:
        m = min(ok, key=lambda m: (abs(m - t), m))
        out[m] = ok[m]
    return out


@pytest.mark.parametrize("lib", [EMUL, CUDA])
def test_stop_test_and_poll_interval(built, lib):
    ref = reference(STOP_SCENE, lib, kmax=max(STOP_TARGETS) + 2, keep=())
    sc = ref.sc
    tols = stop_tolerances(ref, STOP_TARGETS)
    assert set(tols) == set(STOP_TARGETS), f"{STOP_SCENE}: the reference's rre_k has no clean crossing at every target: {sorted(tols)}"
    for m, tol in tols.items():
        runs = {}
        for every in (1, 7, 0, 1000):      # 0: the default, 25; 1000 > maxIterations: one poll at the end
            s = PolyStokesSolver.from_scene(sc, lib_path=lib, tolerance=float(tol), checkEvery=every, maxIterations=STOP_MAX_IT)
            rc, vel, valid = s.step_scene(sc)
            its, fb = s.count("iterations"), s.count("usedBiCGStab")
            assert (rc, its, fb) == (1, m, 0), f"tolerance {tol:.6e}, checkEvery {every}: result {rc}, {its} iterations (reference {m}), fallback {fb}"
            runs[every] = (s.vector("solution"), vel, valid)
            s.close()
        x0, v0, w0 = runs[1]
        for every, (x, v, w) in runs.items():
            assert np.array_equal(x, x0), f"tolerance {tol:.6e}: the solution with checkEvery {every} differs from checkEvery 1"
            for a in range(3):
                assert np.array_equal(v[a], v0[a]) and np.array_equal(w[a], w0[a]), f"checkEvery {every}: velocity / valid axis {a} differ"
    print(f"stop test: iteration counts {sorted(tols)} reproduced with checkEvery 1, 7, 25, 1000")


@pytest.mark.parametrize("keep", [1, 0])
@pytest.mark.parametrize("lib", [EMUL, CUDA])
def test_max_iterations_and_the_fallback(built, lib, keep):
    """maxIterations 1, 24, 25, 26 at tolerance 1e-12: CG runs out, BiCGSTAB takes over and runs out as well.  Result, iteration count
    and fallback flag equal the oracle's.  keepNonConvergedResults 1: the written-back velocity of the non-converged fallback iterate
    within check_bicgstab_fallback's gate (the fallback is chaotic, no bit equality); 0: exactly what the oracle's write-back leaves --
    the valid field, and the velocity untouched."""
    sc = SCENES[FALLBACK_SCENE][0]()
    worst = 0.0
    for m in (1, 24, 25, 26):
        o = Oracle(sc, threads=1, maxIterations=m, tolerance=1e-12).setup()
        ro = o.solve()
        ovel, ovalid = o.writeback()
        # yardstick of the chaotic fallback: the oracle with 4 OpenMP threads sums its dot products in another order
        o4 = Oracle(sc, threads=4, maxIterations=m, tolerance=1e-12).setup()
        assert o4.solve() == ro
        ovel4, _ = o4.writeback()
        yard = max(float(np.abs(ovel4[a] - ovel[a]).max()) / max(float(np.abs(ovel[a]).max()), 1e-30) for a in range(3))
        vgate = max(GATE_MULT * yard, 4e-7)       # 4e-7: the fp32 velocity fields (check_bicgstab_fallback)
        s = PolyStokesSolver.from_scene(sc, lib_path=lib, maxIterations=m, tolerance=1e-12, keepNonConvergedResults=keep)
        rc, vel, valid = s.step_scene(sc)
        got, want = (rc, s.count("iterations"), s.count("usedBiCGStab")), (ro, o.count("iterations"), o.count("usedBiCGStab"))
        assert got == want, f"maxIterations {m}: (result, iterations, usedBiCGStab) {got}, oracle {want}"
        for a in range(3):
            assert np.array_equal(valid[a], ovalid[a]), f"maxIterations {m}: valid axis {a}"
            if keep or ro == 1:
                scale = max(float(np.abs(ovel[a]).max()), 1e-30)
                d = float(np.abs(vel[a] - ovel[a]).max()) / scale
                assert d <= vgate, f"maxIterations {m}: velocity axis {a} differs from the oracle's by {d:.2e} (gate {vgate:.1e})"
                worst = max(worst, d / vgate)
            else:
                assert np.array_equal(vel[a], sc.vel[a]), f"maxIterations {m}, keepNonConvergedResults 0: velocity axis {a} was written"
        s.close()
    print(f"maxIterations 1 / 24 / 25 / 26, keepNonConvergedResults {keep}: worst velocity error / gate {worst:.2f}")


def zero_rhs_scene():
    """A blob whose b is exactly 0: no velocity anywhere, solid at rest."""
    sc = scenes.blob_scene(24, seed=4)
    for a in range(3):
        sc.vel[a][...] = 0.0
        sc.colvel[a][...] = 0.0
    return sc


@pytest.mark.parametrize("solver_type", [0, 1])
@pytest.mark.parametrize("lib", [EMUL, CUDA])
def test_zero_rhs(built, lib, solver_type):
    """b == 0: x = 0 after 0 iterations, success.  CG: the reference would divide 0 / 0 (pcg.h:313), DESIGN.md section 4 documents
    the deviation; Eigen's CG returns x = 0 (ConjugateGradient.h:47-53), as the oracle does."""
    sc = zero_rhs_scene()
    o = Oracle(sc, threads=1).setup()
    assert o.count("nSystemSize") > 0 and not np.any(o.vector("b")), "the scene must have unknowns and b exactly 0"
    s = PolyStokesSolver.from_scene(sc, lib_path=lib, solverType=solver_type)
    rc, vel, valid = s.step_scene(sc)
    assert (rc, s.count("iterations"), s.count("usedBiCGStab")) == (1, 0, 0)
    assert not np.any(s.vector("solution")), "x must be 0"
    if solver_type == 1:
        o.assemble_explicit_A()
        o.construct_guess()
        assert o.solve_eigen_cg() == 1 and o.count("iterations") == 0 and not np.any(o.vector("solution"))
    s.close()


# ---- solverType EIGEN ---------------------------------------------------------------------------------------------------------------
EIGEN_KS = (3, 21)


@pytest.mark.parametrize("warm", [0, 1])
@pytest.mark.parametrize("case", list(parity.EXPLICIT_CASES))
@pytest.mark.parametrize("lib", [EMUL, CUDA])
def test_eigen_cg_fixed_count(built, lib, case, warm):
    """solverType EIGEN stopped by maxIterations = k (tolerance 1e-30): x_k, the iteration count and Eigen's error estimate against
    Oracle.solve_eigen_cg on the explicit A.  Yardstick: the same Jacobi CG in numpy with plain and with shuffled dot products."""
    sc = parity.EXPLICIT_CASES[case]()
    worst = 0.0
    for k in EIGEN_KS:
        o = Oracle(sc, threads=1, maxIterations=k, tolerance=1e-30).setup()
        o.assemble_explicit_A()
        n, nP = o.count("nSystemSize"), o.count("nPressures")
        if warm:
            o.construct_guess()
        x0 = o.vector("guess") if warm else np.zeros(n)
        A, b = o.scipy_csr("A"), o.vector("b")
        xr, er = jacobi_cg(A, b, x0, k, plain_dot)
        xs, es = jacobi_cg(A, b, x0, k, shuffled_dot(n))
        ro = o.solve_eigen_cg()
        ox, oerr, oits = o.vector("solution"), o.real("solveError"), o.count("iterations")
        s = PolyStokesSolver.from_scene(sc, lib_path=lib, solverType=1, useWarmStart=warm, maxIterations=k, tolerance=1e-30)
        rc, _, _ = s.step_scene(sc)
        assert (rc, s.count("iterations")) == (ro, oits), f"k {k}: result / iterations {(rc, s.count('iterations'))}, oracle {(ro, oits)}"
        # the oracle itself against the numpy restatement: a check of the yardstick's premise
        for part, yd, e in zip(("pressure", "stress"), part_rel(xr, xs, nP), part_rel(ox, s.vector("solution"), nP)):
            g = gate(yd)
            assert e <= g, f"k {k}: Eigen CG x_k {part} part differs from the oracle's by {e:.2e} (gate {g:.1e})"
            worst = max(worst, e / g)
        e, g = abs(s.real("solveError") - oerr) / oerr, gate(abs(er - es) / er)
        assert e <= g, f"k {k}: Eigen's error {s.real('solveError')!r}, oracle {oerr!r}: rel {e:.2e} (gate {g:.1e})"
        worst = max(worst, e / g)
        s.close()
    print(f"EIGEN {case} warm {warm}: worst error / gate {worst:.2f}")


# ---- several ranks -------------------------------------------------------------------------------------------------------------------
DIST_KS = (1, 2, 5, 13, 21)


def _check_result(where, scene, res, prefix=""):
    """One multi-rank result (its shares already summed): the reference on its b, then the gates of check_iterates."""
    ref = Reference(W.SCENES[scene](), max(DIST_KS), DIST_KS, res[prefix + "b"], res[prefix + "Ax"])
    got = {k: (res[f"{prefix}x{k}"], float(res[f"{prefix}xmag{k}"]), float(res[f"{prefix}err{k}"]), int(res[f"{prefix}its{k}"])) for k in DIST_KS}
    return ref, check_iterates(where, ref, got, DIST_KS)


@pytest.mark.parametrize("scene,world", [("blob48_tile8", 2), ("box48_uniform", 3), ("blob48_tile8", 3)])
def test_distributed_iterates_gloo(built, tmp_path, scene, world):
    """cg_update_kernel's range walk, the two all-reduces per iteration and the halo of p on the host-emulation twin under gloo."""
    port = 29900 + (os.getpid() + world + len(scene)) % 90
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WORLD_SIZE=str(world), OMP_NUM_THREADS="2")
    cmd = [sys.executable, os.path.join(HERE, "cg_iterates_worker.py"), scene, str(tmp_path)] + [str(k) for k in DIST_KS]
    procs = [subprocess.Popen(cmd, env=dict(env, RANK=str(r)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT) for r in range(world)]
    fail = []
    for r, p in enumerate(procs):
        try:
            out, _ = p.communicate(timeout=600)
        except subprocess.TimeoutExpired:
            for q in procs:
                q.kill()
            raise AssertionError(f"rank {r} timed out")
        if p.returncode != 0:
            fail.append(f"rank {r} exit {p.returncode}:\n{out.decode()[-3000:]}")
    assert not fail, "\n".join(fail)
    ranks = [dict(np.load(os.path.join(str(tmp_path), f"rank{r}.npz"))) for r in range(world)]
    assert all(int(r["nranks"]) == world for r in ranks)
    for k in DIST_KS:
        for key in ("xmag", "err", "its"):
            assert len({float(r[f"{key}{k}"]) for r in ranks}) == 1, f"{key} after {k} iterations differs between ranks"
    res = dict(ranks[0])
    for key in ["b", "Ax"] + [f"x{k}" for k in DIST_KS]:       # every global vector is the sum of the ranks' shares
        res[key] = sum(r[key] for r in ranks)
    _, worst = _check_result(f"{scene} on {world} ranks", scene, res)
    print(f"{scene} on {world} gloo ranks: worst error / gate {worst:.2f}")


@pytest.mark.gpu
@pytest.mark.parametrize("scene,ndev", [("blob48_tile8", 2), ("box48_uniform", 3), ("blob48_tile8", 3)])
def test_multi_gpu_iterates(built, tmp_path, scene, ndev):
    """The fused peer all-reduces and the direct p halo of a ps_create_multi handle: x_k (global) against the reference, and against
    the single-GPU handle's x_k (a different summation order only)."""
    import torch
    if torch.cuda.device_count() < ndev:
        pytest.skip(f"needs {ndev} GPUs")
    cmd = [sys.executable, os.path.join(HERE, "cg_iterates_worker.py"), "--devices", str(ndev), scene, str(tmp_path)] + [str(k) for k in DIST_KS]
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=240, env=dict(os.environ, PS_MULTI_WATCHDOG_S="45"))
    except subprocess.TimeoutExpired as e:
        pytest.fail(f"multi-GPU handle hung on {scene} x {ndev}:\n{e.stderr}")
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    res = dict(np.load(os.path.join(str(tmp_path), "multi.npz")))
    assert int(res["nranks"]) == ndev
    ref, worst = _check_result(f"{scene} on {ndev} GPUs", scene, res)
    worst = max(worst, _check_result(f"{scene} on one GPU", scene, res, "one_")[1])
    for k in DIST_KS:
        for part, e, y in zip(("pressure", "stress"), part_rel(res[f"one_x{k}"], res[f"x{k}"], ref.nP), (ref.yard[k]["xP"], ref.yard[k]["xS"])):
            assert e <= 2 * gate(y), f"x_{k} {part} part: {ndev} GPUs vs one GPU {e:.2e} (gate {2 * gate(y):.1e})"
    print(f"{scene} on {ndev} GPUs: worst error / gate {worst:.2f}")

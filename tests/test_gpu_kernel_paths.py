"""Every implementation of the reduced-region term and of the region Gram build, against the oracle with per-entry gates.

Which kernels carry the reduced term of an apply depends on the scene (<= 900 owned regions: reduced_region_kernel with 128 lanes per
axis; more: 64 lanes; a region of more than 16384 coupled rows: the chunked reduced_moments_kernel with per-region tickets, then
reduced_expand_kernel) and on a knob read once per process (PS_REGION_FUSE_MAX).  Each setting runs in a child process
(tests/kernel_path_worker.py) under a time-out; the library's `regionPath` count says which kernels ran, and each test asserts it, so a
moved threshold fails here instead of silently covering another path.

Gates, per setting and scene (the CPU figures are the host-emulation twin against the oracle):
  - operator: |y_i - (A x)_i| <= OPERATOR_GATE bound_i, with A x evaluated by scipy through the oracle's factors and bound the same
    product of their absolute values (parity.scipy_factored); exactly 0 where that bound is 0;
  - region blocks per region and entry: parity.REGION_GATES;
  - apply(x1) bit-identical before, between and after the other apply and the step (a ticket that does not wrap breaks it);
  - the solve: parity.check_solve's gates against the oracle; on the 1000-region scene, which the oracle does not solve here, the
    reference's stop rule recomputed with the oracle's apply and the velocity against the same step solved to tol / 1000.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import kernel_path_worker as W
import parity

HERE = os.path.dirname(os.path.abspath(__file__))

TILED = ["blob40", "blob32_seed5", "blob64_tile32", "box96_tile8"]
ALL = TILED + ["blob64_notile"]

# setting -> (environment, scenes it runs on).  The region knob does nothing on the one-region scene: it takes the chunked kernels.
SETTINGS = {
    "default": ({}, ALL),
    "fuse_max0": ({"PS_REGION_FUSE_MAX": "0"}, TILED),          # the chunked kernels on tiled regions: one chunk per (region, axis)
}


# regionPath: 0 / 1 reduced_region_kernel with 64 / 128 lanes per axis, 2 the chunked kernels
def expected_path(setting, scene, regions):
    if scene == "blob64_notile":
        return 2
    if setting == "fuse_max0":
        return 2
    return 1 if regions <= 900 else 0

# Velocity gates where 10 x tol is not meaningful.  The velocity recovered on these scenes amplifies the CG stopping difference: at its
# tolerance each correct run lands 2-4e-2 from the converged field (blob64_tile32 at 1e-4: the oracle and the emulation twin both, in
# the same 243 iterations, 1.7e-2 apart, their solutions x 4.3e-6 apart; blob64_notile at 1e-4: 5.5e-3 apart; box96_tile8 at 1e-3:
# the twin 3.7e-2 from its run to 1e-6).
# A solve that is wrong in earnest shows up in x (gated at 10 x tol) and in the stop rule recomputed with the oracle's apply.
VEL_GATE = {"blob64_tile32": 0.1, "blob64_notile": 0.1, "box96_tile8": 0.1}

OPERATOR_GATE = parity.OPERATOR_GATE

_results = {}
_refs = {}


def run_worker(setting, tmp_root, lib=None, scenes=None, tight=True, step=True):
    """Run (once per session) the worker for `setting`; returns {scene: npz dict}."""
    key = (setting, lib)
    if key not in _results:
        env_over, names = SETTINGS[setting]
        names = scenes or names
        out = os.path.join(str(tmp_root), setting + ("_emul" if lib else ""))
        env = dict(os.environ, **env_over)
        cmd = [sys.executable, os.path.join(HERE, "kernel_path_worker.py")] + (["--lib", lib] if lib else [])
        cmd += (["--tight"] if tight and setting == "default" else []) + ([] if step else ["--no-step"]) + [out] + names
        try:
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
        except subprocess.TimeoutExpired as e:
            err = e.stderr.decode() if isinstance(e.stderr, bytes) else (e.stderr or "")
            pytest.fail(f"kernel path worker timed out under {setting}:\n{err[-4000:]}")
        assert r.returncode == 0, f"kernel path worker failed under {setting} ({env_over}):\n{r.stdout[-2000:]}{r.stderr[-4000:]}"
        _results[key] = {n: dict(np.load(os.path.join(out, n + ".npz"))) for n in names}
    return _results[key]


class Reference:
    """The oracle on one scene, and A x1, A x2 evaluated by scipy through the oracle's factors."""

    def __init__(self, name):
        from oracle.oracle import Oracle
        self.name = name
        self.sc = W.SCENES[name]()
        self.o = Oracle(self.sc).setup()
        o = self.o
        self.R, self.n = o.count("regionCount"), o.count("nSystemSize")
        self.vec = {v: o.vector(v) for v in ("MrDense", "ViscDense", "BinvDense", "bestFit", "com", "b")}
        apply = parity.scipy_factored(o.csr, self.sc.dt)
        self.Ax, self.bound = zip(*[apply(x) for x in W.vectors(self.n)])
        self.tol = self.sc.params["tolerance"]
        if name in W.TIGHT:
            self.rc = None
        else:
            self.rc = o.solve()
            self.iterations = o.count("iterations")
            self.vel, self.valid = o.writeback()
            self.solution = o.vector("solution")


def reference(name):
    if name not in _refs:
        _refs[name] = Reference(name)
    return _refs[name]


def check_scene(setting, name, res, tight=None, path=None):
    """The oracle gates on one worker result; returns (worst componentwise apply error, worst region-block error / its gate)."""
    ref = reference(name)
    where = f"{setting} on {name}"
    assert int(res["count_regionCount"]) == ref.R and int(res["count_nSystemSize"]) == ref.n, where
    want = expected_path(setting, name, ref.R) if path is None else path
    path = int(res["count_regionPath"])
    assert path == want, f"{where}: regionPath {path}, expected {want}"
    assert np.array_equal(res["com"], ref.vec["com"]), f"{where}: centres of mass not bit-equal"
    assert parity.rel(ref.vec["b"], res["b"]) <= 1e-10, f"{where}: b rel {parity.rel(ref.vec['b'], res['b']):.2e}"
    blocks = parity.region_block_errors(ref.vec.get, res.get, ref.R)
    for v, gate in parity.REGION_GATES.items():
        assert blocks[v] <= gate, f"{where} (regionPath {path}): {v} worst per-region error {blocks[v]:.2e} > {gate:.0e}"
    op = 0.0
    for y, Ax, bound in ((res["y1_first"], ref.Ax[0], ref.bound[0]), (res["y2"], ref.Ax[1], ref.bound[1])):
        e = parity.operator_error(y, Ax, bound)
        assert e <= OPERATOR_GATE, f"{where} (regionPath {path}): componentwise apply error {e:.2e} > {OPERATOR_GATE:.0e}"
        op = max(op, e)
    for v in ("MrDense", "ViscDense", "BinvDense", "bestFit"):
        assert np.array_equal(res[v], res[v + "_second_handle"]), f"{where}: {v} of a second handle differs"
    assert np.array_equal(res["y1_first"], res["y1_second"]), f"{where} (regionPath {path}): apply(x1) changed after apply(x2)"
    if "y1_after_step" in res:
        assert np.array_equal(res["y1_first"], res["y1_after_step"]), f"{where} (regionPath {path}): apply(x1) changed after the solve"
        check_solve(where, ref, res, tight)
    return op, max(blocks[v] / g for v, g in parity.REGION_GATES.items())


def check_solve(where, ref, res, tight):
    rc, its = int(res["rc"]), int(res["iterations"])
    vtol = VEL_GATE.get(ref.name, max(10 * ref.tol, 4e-7))      # the velocity fields are fp32
    if ref.rc is not None:
        assert rc == ref.rc, f"{where}: solver result {rc}, oracle {ref.rc}"
        assert abs(its - ref.iterations) <= max(2, int(0.01 * ref.iterations)), f"{where}: iterations {its}, oracle {ref.iterations}"
        d = parity.rel(ref.solution, res["solution"])
        assert d <= 10 * ref.tol, f"{where}: solution differs from the oracle's by {d:.2e}"
        vel, valid = ref.vel, ref.valid
    else:
        # the reference's stop rule min(rr, rr / xx) < tol^2 (pcg.h:316-325), recomputed on the returned x with the oracle's apply
        assert rc == 1, f"{where}: solver result {rc}"
        x = res["solution"]
        e = ref.vec["b"] - ref.o.apply(x)
        rr, xx = float(e @ e), float(x @ x)
        got = min(rr, rr / max(xx, 1e-300))      # slack 1.5: the loop tests its recursively updated residual, this is the true one
        assert got < 1.5 * ref.tol ** 2, f"{where}: returned x does not satisfy the stop rule: {got:.3e} >= {ref.tol ** 2:.1e}"
        if tight is None:
            return
        assert int(tight["tight_rc"]) == 1
        vel, valid = [tight[f"tight_vel{a}"] for a in range(3)], [tight[f"tight_valid{a}"] for a in range(3)]
    for a in range(3):
        assert np.array_equal(valid[a], res[f"valid{a}"]), f"{where}: valid field axis {a}"
        scale = max(float(np.abs(vel[a]).max()), 1e-30)
        d = float(np.abs(vel[a] - res[f"vel{a}"]).max()) / scale
        assert d <= vtol, f"{where}: velocity axis {a} differs by {d:.2e} (gate {vtol:.1e})"
    if int(res["usedBiCGStab"]) == 0:
        x = res["solution"]
        xx = float(x @ x)
        assert abs(float(res["xmag"]) - xx) <= 1e-11 * max(xx, 1e-300), f"{where}: x.x recurrence drift"


@pytest.mark.gpu
@pytest.mark.parametrize("setting", list(SETTINGS))
def test_gpu_kernel_path_matches_oracle(built, setting, tmp_path_factory):
    res = run_worker(setting, tmp_path_factory.getbasetemp())
    tight = run_worker("default", tmp_path_factory.getbasetemp())["box96_tile8"]
    for name, r in res.items():
        op, blk = check_scene(setting, name, r, tight)
        print(f"{setting:12s} {name:14s} regionPath {int(r['count_regionPath'])}: worst componentwise apply error {op:.2e}, "
              f"worst region-block error {blk:.2e} of its gate")


@pytest.mark.gpu
def test_gpu_kernel_path_scenes_cover_the_edges(built, tmp_path_factory):
    """The scenes reach what each kernel does differently at its edges: > 1024 rows on one (region, axis) (the tail loop of
    reduced_region_kernel<128, 8, .> past 8 x 128 rows), a region spanning several 256-cell Gram chunks, one whose last chunk is
    partial, one with fewer than 32 cells, and more than 900 regions (the default 64-lane path)."""
    res = run_worker("default", tmp_path_factory.getbasetemp())
    assert int(res["blob64_tile32"]["count_maxRegionAxisRows"]) > 1024
    assert int(res["blob64_notile"]["count_maxRegionRows"]) > 16384
    cells = [int(r["count_maxRegionCells"]) for r in res.values()]
    assert any(c > 2 * 256 for c in cells) and any(c % 256 for c in cells)
    assert min(int(r["count_minRegionCells"]) for r in res.values()) < 32
    assert int(res["box96_tile8"]["count_regionCount"]) > 900


def test_emulated_kernel_path_worker(built, tmp_path_factory):
    """The harness and the gates above without a GPU: the worker on the host-emulation twin (which has the chunked kernels only,
    regionPath 2), default setting, every scene; the 1000-region scene is checked by its stop rule."""
    res = run_worker("default", tmp_path_factory.getbasetemp(), lib=parity.EMUL_LIB, tight=False)
    for name, r in res.items():
        op, blk = check_scene("default", name, r, path=2)
        print(f"emulated {name:14s}: worst componentwise apply error {op:.2e}, worst region-block error {blk:.2e} of its gate")
    assert int(res["blob64_tile32"]["count_maxRegionAxisRows"]) > 1024
    assert int(res["blob64_notile"]["count_maxRegionRows"]) > 16384
    assert int(res["box96_tile8"]["count_regionCount"]) > 900
    assert min(int(r["count_minRegionCells"]) for r in res.values()) < 32

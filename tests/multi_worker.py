"""Child process of tests/test_gpu_multi.py: one case of the ps_create_multi parity check (a hang in the multi-GPU handle must
cost one test its time-out, not the whole GPU session).  usage: python multi_worker.py <case> <ndev>"""
import os
import sys
import threading

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import edge_cases  # noqa: E402
import parity  # noqa: E402
from polystokes_b200 import PolyStokesSolver, scenes  # noqa: E402

CASES = {
    "blob64_tile16_pad2": lambda: scenes.blob_scene(64, seed=13, tile=16, pad=2),                       # slab-local setup
    "blob48_tile8_pad1": lambda: scenes.blob_scene(48, seed=21, tile=8, pad=1),                         # replicated setup (boundary fix-up)
    "box64_uniform": lambda: scenes.box_scene(64, doReduced=0, tolerance=1e-6),
    "s3_128": lambda: scenes.scene_s3(128),
    # liquid on the domain faces (tests/test_input_edges.py)
    **{name: (lambda c: lambda: c()[0])(case) for name, case in edge_cases.DIST.items()},
}


def main(case, ndev):
    sc = CASES[case]()
    one = PolyStokesSolver.from_scene(sc)
    rc1, vel1, valid1 = one.step_scene(sc)
    many = PolyStokesSolver.from_scene(sc, devices=list(range(ndev)))
    rcN, velN, validN = many.step_scene(sc)
    assert rc1 == rcN == 1, (rc1, rcN)
    for k in parity.COUNTS:
        assert one.count(k) == many.count(k), f"count {k}"
    assert abs(one.count("iterations") - many.count("iterations")) <= max(2, one.count("iterations") // 100)
    tol = max(10 * sc.params["tolerance"], 4e-7)
    for a in range(3):
        assert np.array_equal(valid1[a], validN[a]), f"valid axis {a}"
        scale = max(float(np.abs(vel1[a]).max()), 1e-30)
        assert float(np.abs(vel1[a] - velN[a]).max()) <= tol * scale, f"velocity axis {a}: {float(np.abs(vel1[a] - velN[a]).max()) / scale:.2e}"
    # a second step on the same handle reproduces the first bit for bit; the handle on a different calling thread works too
    res = {}
    th = threading.Thread(target=lambda: res.update(r=many.step_scene(sc)))
    th.start(); th.join()
    rc2, vel2, _ = res["r"]
    assert rc2 == rcN and all(np.array_equal(velN[a], vel2[a]) for a in range(3))
    # new per-step parameters on the same handle (ps_set_params: a DOP substep with another dt), against a fresh single-GPU handle
    P = many._P
    P.dt = float(sc.dt) * 0.5
    assert many.lib.ps_set_params(many.h, P) == 1, many.last_error()
    rc3, vel3, valid3 = many.step_scene(sc)
    half = PolyStokesSolver(sc.nx, sc.ny, sc.nz, sc.dx, float(sc.dt) * 0.5, sc.density, **sc.params)
    rc4, vel4, valid4 = half.step_scene(sc)
    assert rc3 == rc4 == 1
    its3, its4 = many.count("iterations"), half.count("iterations")
    worst = 0.0
    for a in range(3):
        assert np.array_equal(valid3[a], valid4[a])
        scale = max(float(np.abs(vel4[a]).max()), 1e-30)
        worst = max(worst, float(np.abs(vel3[a] - vel4[a]).max()) / scale)
    print(f"dt/2 on the same handle: iterations {its3} (multi) vs {its4} (fresh single-GPU handle), velocity max rel diff {worst:.3e} (gate {tol:.1e})")
    assert abs(its3 - its4) <= max(2, its4 // 100) and worst <= tol, "dt/2 step differs from a fresh handle's"
    its = many.count("iterations")
    one.close(); many.close(); half.close()
    print(f"multi ok: {case} on {ndev} GPUs, {its} iterations")


if __name__ == "__main__":
    main(sys.argv[1], int(sys.argv[2]))

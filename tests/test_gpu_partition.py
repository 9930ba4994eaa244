"""Work-balanced z cuts on real GPUs (tests/partition_worker.py, mode "steps"): a step, ps_rebalance, and a step on the new cuts, on small
S5- and S4-shaped scenes at 2 / 4 / 8 GPUs -- one process per GPU with the NVLink peer transport or with NCCL alone, and one
ps_create_multi handle -- against a single-GPU handle: counts and index fields (or, on the multi handle, the G / Dt / JG blocks) bit for
bit, unitLoad identical, iterations within max(2, 1 %), velocity within 10 x tol.  A case skips when there are too few GPUs."""
import os
import subprocess
import sys

import numpy as np
import pytest

import parity
import partition_worker
from test_partition_emul import launch

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
partition_worker.register()
NZ = {"s5_half_tile16": 128, "s4_128_tile32": 128}
UNIT = {"s5_half_tile16": 16, "s4_128_tile32": 32}


def _need(ndev, case):
    import torch
    if torch.cuda.device_count() < ndev:
        pytest.skip(f"needs {ndev} GPUs")
    if NZ[case] < UNIT[case] * ndev:
        pytest.skip("fewer z-units than devices")


def _run(args, env=None, timeout=600):
    r = subprocess.run([sys.executable, os.path.join(HERE, "partition_worker.py")] + args, capture_output=True, text=True, timeout=timeout,
                       env=dict(os.environ, OMP_NUM_THREADS="2", PS_MULTI_WATCHDOG_S="60", **(env or {})))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]


def _single(case, tmp_path):
    _run(["steps", case, str(tmp_path), "1"])
    return dict(np.load(os.path.join(tmp_path, "single.npz")))


def _compare_solve(case, one, its, vel_of):
    sc, ov = parity.DIST_CASES[case]()
    assert abs(its - int(one["iterations"])) <= max(2, int(0.01 * int(one["iterations"]))), f"iterations {its} vs {int(one['iterations'])} on one GPU"
    tol = max(10 * dict(sc.params, **ov)["tolerance"], 4e-7)
    for a in range(3):
        ref, got = one[f"vel{a}"], vel_of(a)
        scale = max(float(np.abs(ref).max()), 1e-30)
        assert float(np.abs(ref - got).max()) <= tol * scale, f"velocity axis {a}: {float(np.abs(ref - got).max()) / scale:.2e}"


def test_unit_table_on_one_gpu(built):
    """The CUDA library's unit table of one GPU against the oracle's model, its sum against ps_kernel_bytes, ps_rebalance a no-op."""
    from oracle.oracle import Oracle
    from polystokes_b200 import PolyStokesSolver
    from polystokes_b200._capi import PS_NOCHANGE
    from test_partition_emul import unit_model
    for case, unit in (("offz_blob_tile16", 16), ("blob_40x36x96_tile32_pad3", 32), ("span_bodies_notile", 16)):
        sc, ov = parity.DIST_CASES[case]()
        s = PolyStokesSolver.from_scene(sc, **ov)
        s.setup_scene(sc)
        T = unit_model(Oracle(sc, **ov).setup(), sc.nz, unit)
        assert np.array_equal(s.vector("unitCounts").reshape(-1, 9).astype(np.int64), T), case
        assert float(s.vector("unitLoad").sum()) == s.kernel_bytes("cg_iteration"), case
        assert s.rebalance() == (PS_NOCHANGE, [0, sc.nz])
        s.close()


CASES = [("s5_half_tile16", n) for n in (2, 4, 8)] + [("s4_128_tile32", n) for n in (2, 4)]


@pytest.mark.parametrize("transport", ["peer", "nccl"])
@pytest.mark.parametrize("case,ndev", CASES)
def test_rebalanced_one_process_per_gpu(built, tmp_path, case, ndev, transport):
    _need(ndev, case)
    one = _single(case, tmp_path)
    port = 30200 + (os.getpid() + hash((case, ndev, transport))) % 500
    ranks = launch("steps", case, ndev, tmp_path, port, gpu=True, timeout=600, extra_env={"PS_COMM": "nccl" if transport == "nccl" else ""})
    nz = NZ[case]
    cuts = [int(c) for c in ranks[0]["cuts"]]
    assert all(int(r["peer"]) == (1 if transport == "peer" else 0) for r in ranks)
    print(f"{case} on {ndev} GPUs ({transport}): even {list(ranks[0]['even_cuts'])} -> {cuts} (rc {int(ranks[0]['rb_rc'])})", flush=True)
    for r in ranks:
        assert int(r["rc1"]) == int(r["rc"]) == int(one["rc"]) == 1
        assert list(r["rb_cuts"]) == cuts == [int(c) for c in r["cuts"]]
        assert np.array_equal(r["unitLoad"], one["unitLoad"]) and np.array_equal(r["unitLoad_after"], one["unitLoad"]), "unitLoad differs from one GPU"
        for k in parity.COUNTS:
            assert int(r["count_" + k]) == int(one["count_" + k]), f"count {k} on rank {int(r['rank'])}"
        lo, hi = int(r["zlo"]), int(r["zhi"])
        own = lambda f: f[lo:(hi if hi < nz else f.shape[0])]
        for slot in range(7):
            for name in ("labels", "active", "reduced"):
                assert np.array_equal(own(r[f"{name}{slot}"]), own(one[f"{name}{slot}"])), f"{name} slot {slot} on rank {int(r['rank'])}"
    assert len({int(r["iterations"]) for r in ranks}) == 1

    def merged(a):
        m = np.empty_like(one[f"vel{a}"])
        for r in ranks:
            lo, hi = int(r["zlo"]), int(r["zhi"])
            sl = slice(lo, hi if hi < nz else m.shape[0])
            m[sl] = r[f"vel{a}"][sl]
            assert np.array_equal(r[f"valid{a}"][sl], one[f"valid{a}"][sl]), f"valid axis {a} on rank {int(r['rank'])}"
        return m
    _compare_solve(case, one, int(ranks[0]["iterations"]), merged)


@pytest.mark.parametrize("case,ndev", [("s5_half_tile16", 8), ("s5_half_tile16", 4), ("s4_128_tile32", 2)])
def test_rebalanced_multi_handle(built, tmp_path, case, ndev):
    _need(ndev, case)
    one = _single(case, tmp_path)
    _run(["steps", case, str(tmp_path), str(ndev)])
    m = dict(np.load(os.path.join(tmp_path, "multi.npz")))
    print(f"{case} on a {ndev}-GPU multi handle: -> {list(m['cuts'])} (rc {int(m['rb_rc'])})", flush=True)
    assert int(m["rc1"]) == int(m["rc"]) == 1 and list(m["rb_cuts"]) == list(m["cuts"])
    assert np.array_equal(m["unitLoad"], one["unitLoad"]), "unitLoad differs from one GPU"
    for k in parity.COUNTS:
        assert int(m["count_" + k]) == int(one["count_" + k]), f"count {k}"
    for key in [k for k in one if k.startswith("csr_G_") or k.startswith("csr_Dt_")]:
        assert np.array_equal(m[key], one[key]), f"{key} differs from one GPU"
    for i in (0, 1):       # JG: the pattern bit for bit (values are sums in another order across shared rows)
        assert np.array_equal(m[f"csr_JG_{i}"], one[f"csr_JG_{i}"]), "JG pattern differs from one GPU"
    for a in range(3):
        assert np.array_equal(m[f"valid{a}"], one[f"valid{a}"])
    _compare_solve(case, one, int(m["iterations"]), lambda a: m[f"vel{a}"])

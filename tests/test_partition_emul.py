"""Work-balanced z cuts on CPU: world_size-N gloo jobs drive the host-emulation twin (tests/partition_worker.py).

The unit table of a setup (ps_get_vector "unitLoad" / "unitCounts") against a numpy model built from the oracle's index fields, labels
and weights; ps_rebalance against a brute-force search over every cut vector; ps_set_partition's rules; and after the cuts move,
everything parity.check_distributed checks against the oracle."""
import itertools
import os
import subprocess
import sys

import numpy as np
import pytest

import parity
import partition_worker
from oracle.oracle import Oracle
from polystokes_b200 import PolyStokesSolver
from polystokes_b200._capi import PS_SUCCESS, PS_INVALID, PS_NOCHANGE

HERE = os.path.dirname(os.path.abspath(__file__))
partition_worker.register()

L_REDUCED = -6
ACTIVE = (-4, -9)        # L_ACTIVEFLUID, L_BOUNDARY


def launch(mode, case, world, outdir, port, cuts=None, gpu=False, timeout=1200, extra_env=None):
    env = dict(os.environ, **(extra_env or {}))
    env = dict(env, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WORLD_SIZE=str(world), OMP_NUM_THREADS="2")
    args = [sys.executable, os.path.join(HERE, "partition_worker.py"), mode, case, str(outdir)] + ([",".join(map(str, cuts))] if cuts else []) + (["gpu"] if gpu else [])
    procs = [subprocess.Popen(args, env=dict(env, RANK=str(r), LOCAL_RANK=str(r)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT) for r in range(world)]
    fail = []
    for r, p in enumerate(procs):
        try:
            out, _ = p.communicate(timeout=timeout)
        except subprocess.TimeoutExpired:
            for q in procs:
                q.kill()
            raise AssertionError(f"rank {r} timed out")
        if p.returncode != 0:
            fail.append(f"rank {r} exit {p.returncode}:\n{out.decode()[-3000:]}")
    assert not fail, "\n".join(fail)
    return [dict(np.load(os.path.join(outdir, f"rank{r}.npz"))) for r in range(world)]


def unit_of(params):
    """lcm(16, tileSize) layers with tiles, 16 without."""
    p = dict(params)
    if p.get("doReduced", 1) and p.get("doTile", 1) and p.get("tileSize", 16) >= 1:
        return int(np.lcm(16, p["tileSize"]))
    return 16


def unit_model(o, nz, unit):
    """[units][9]: active voxels of the 7 slots, coupled reduced rows (by the z of the face), regions (by the z of their first cell),
    counted from the oracle; the slots' top layer goes to the last unit."""
    nU = -(-nz // unit)
    T = np.zeros((nU, 9), dtype=np.int64)
    per_unit = lambda per_z: np.bincount(np.minimum(np.arange(per_z.size) // unit, nU - 1), weights=per_z, minlength=nU).astype(np.int64)
    for slot in range(7):
        T[:, slot] = per_unit((o.index_field(1, slot) >= 0).sum(axis=(1, 2)))
    cell_ok = (o.index_field(1, 0) >= 0) & (o.weight_field(1, 0) > 0)
    for a in range(3):
        ax = 2 - a                                    # numpy axis of coordinate a
        lab, ridx = o.index_field(0, 1 + a), o.index_field(2, 1 + a)
        f = (lab == L_REDUCED) & (o.weight_field(0, 1 + a) > 0) & (ridx >= 0)
        pad = [(0, 0)] * 3
        pad[ax] = (1, 1)
        P = np.pad(cell_ok, pad)
        n = cell_ok.shape[ax]
        near = np.take(P, np.arange(0, n + 1), axis=ax) | np.take(P, np.arange(1, n + 2), axis=ax)
        for e in ((1 if a == 0 else 0), (1 if a == 2 else 2)):
            t = 3 - a - e                             # the third axis: dir 1 is the edge one step along it
            E = np.isin(o.index_field(0, 4 + e), ACTIVE) & (o.weight_field(1, 4 + e) > 0)
            m = f.shape[2 - t]
            near |= np.take(E, np.arange(0, m), axis=2 - t) | np.take(E, np.arange(1, m + 1), axis=2 - t)
        T[:, 7] += per_unit((f & near).sum(axis=(1, 2)))
    cells, lab = o.index_field(2, 0), o.index_field(0, 0)
    R = o.count("regionCount")
    zmin = np.full(R, nz, dtype=np.int64)
    z, _, _ = np.nonzero((lab == L_REDUCED) & (cells >= 0))
    np.minimum.at(zmin, cells[(lab == L_REDUCED) & (cells >= 0)], z)
    T[:, 8] = np.bincount(np.minimum(zmin // unit, nU - 1), minlength=nU)
    return T


def loads(T, bytes_of):
    return np.array([bytes_of(t) for t in T])


def cg_bytes(t):
    """ps_kernel_bytes("cg_iteration") of a count row (DESIGN.md section 5)."""
    nC, nA, nE, nRed, R = int(t[0]), int(t[1] + t[2] + t[3]), int(t[4] + t[5] + t[6]), int(t[7]), int(t[8])
    n, rows = 4 * nC + nE, nA + nRed
    pass1 = 32 * rows + nA + 8 * n + 8 * rows + 24 * nRed + R * (26 * 26 + 52 + 30) * 8
    pass2dots = 32 * nC + 20 * nE + 8 * rows + 8 * (nC + nE) + 24 * n
    return float(pass1 + pass2dots + 56 * n)


def brute_force(load, nranks):
    """Lexicographically smallest cut vector (in units) that minimises the largest slab load, every slab at least one unit."""
    n = len(load)
    pre = np.concatenate([[0.0], np.cumsum(load)])
    best, arg = None, None
    for inner in itertools.combinations(range(1, n), nranks - 1):
        c = (0,) + inner + (n,)
        m = max(pre[c[k + 1]] - pre[c[k]] for k in range(nranks))
        if best is None or m < best:
            best, arg = m, c
    return list(arg), best


def slab_max(load, cuts_units):
    pre = np.concatenate([[0.0], np.cumsum(load)])
    return max(pre[b] - pre[a] for a, b in zip(cuts_units[:-1], cuts_units[1:]))


def even_cuts(nz, unit, world):
    nU = -(-nz // unit)
    c = [min(nz, ((k * nU + world // 2) // world) * unit) for k in range(world + 1)]
    c[0], c[-1] = 0, nz
    return c


def port_of(*key):
    return 31000 + (os.getpid() + hash(key)) % 900


def check_unit_table(case, ranks):
    sc, ov = parity.DIST_CASES[case]()
    unit = unit_of(dict(sc.params, **ov))
    o = Oracle(sc, **ov).setup()
    T = unit_model(o, sc.nz, unit)
    world = len(ranks)
    for r in ranks:
        got = r["unitCounts"].reshape(-1, 9).astype(np.int64)
        assert np.array_equal(got, T), f"unitCounts on rank {int(r['rank'])} differ from the model in {np.argwhere(got != T).tolist()[:8]}"
        assert np.array_equal(r["unitLoad"], loads(T, cg_bytes)), "unitLoad differs from the model"
        assert float(r["unitLoad"].sum()) == float(r["cg_bytes"]), f"sum(unitLoad) {r['unitLoad'].sum()} != cg_iteration bytes {r['cg_bytes']}"
    # a rank's units hold exactly its slotCut ranges (even cuts): the active indices of its slab
    cuts = list(ranks[0]["even_cuts"])
    for k in range(world):
        u0, u1 = cuts[k] // unit, -(-cuts[k + 1] // unit)
        for slot in range(7):
            a = o.index_field(1, slot)
            own = a[cuts[k]:(cuts[k + 1] if k + 1 < world else a.shape[0])]
            own = own[own >= 0]
            lo = int(own.min()) if own.size else None
            assert T[u0:u1, slot].sum() == own.size, f"slot {slot} rank {k}: units hold {T[u0:u1, slot].sum()}, the slab {own.size}"
            if own.size:
                assert int(own.max()) - lo + 1 == own.size and lo == T[:u0, slot].sum(), f"slot {slot} rank {k}: not the contiguous range after the units below"
    return T, unit, o


REBALANCE = [("offz_blob_tile16", 2), ("offz_blob_tile16", 3), ("offz_blob_tile16", 4),
             ("blob_40x36x96_tile32_pad3", 2),                  # tile 32: even cuts 64 / 32
             ("span_bodies_notile", 3)]                         # untiled: shared regions across the cuts


@pytest.mark.parametrize("case,world", REBALANCE)
def test_rebalance_matches_brute_force_and_oracle(built, tmp_path, case, world):
    parity.write_region_probes(case, tmp_path)
    ranks = launch("rebalance", case, world, tmp_path, port_of(case, world))
    T, unit, _ = check_unit_table(case, ranks)
    load = loads(T, cg_bytes)
    nz = parity.DIST_CASES[case]()[0].nz
    even = [int(c) for c in ranks[0]["even_cuts"]]
    cur = [-(-c // unit) for c in even]
    best, m = brute_force(load, world)
    want = [c * unit for c in best[:-1]] + [nz] if m < slab_max(load, cur) else even
    for r in ranks:
        assert int(r["rb0_rc"]) == PS_INVALID, "ps_rebalance before any setup"
        assert int(r["rb1_rc"]) == (PS_SUCCESS if want != even else PS_NOCHANGE)
        assert list(r["rb1_cuts"]) == want, f"rebalanced cuts {list(r['rb1_cuts'])}, brute force {want} (even {even})"
        assert int(r["rb2_rc"]) == PS_NOCHANGE and list(r["rb2_cuts"]) == want
        assert np.array_equal(r["unitLoad_after"], load), "the unit loads depend on the cuts"
    print(f"{case} on {world} ranks: even {even} (largest slab {slab_max(load, cur):.0f} B) -> {want} ({m:.0f} B)", flush=True)
    if case == "offz_blob_tile16":
        assert want != even
    parity.check_distributed(case, ranks)


def test_set_partition_rules_and_persistence(built, tmp_path):
    case, world, cuts = "offz_blob_tile16", 2, [0, 80, 96]
    parity.write_region_probes(case, tmp_path)
    ranks = launch("set", case, world, tmp_path, port_of("set"), cuts=cuts)
    even = [int(c) for c in ranks[0]["even_cuts"]]
    for r in ranks:
        assert int(r["set_rc"]) == PS_SUCCESS and list(r["cuts"]) == cuts
        for name in ("first", "last", "order", "empty", "unit", "disagree"):
            assert int(r[f"bad_{name}_rc"]) == PS_INVALID, f"broken rule {name}: rc {int(r[f'bad_{name}_rc'])} on rank {int(r['rank'])}"
            assert list(r[f"bad_{name}_cuts"]) == cuts, f"broken rule {name} moved the cuts"
        assert bool(r["kept_step_ok"]), "a step after the refused calls differs from the step before them"
        assert int(r["null_rc"]) == PS_SUCCESS and list(r["null_cuts"]) == even
        assert list(r["dt_cuts"]) == cuts, "ps_set_params with a new dt moved the cuts"
        assert list(r["tile32_cuts"]) == even_cuts(96, 32, world), "tileSize 32 (80 is no multiple of 32) must give the even cuts"
    parity.check_distributed(case, ranks)


def test_cuts_survive_the_replicated_restart(built, tmp_path):
    case, world, cuts = "fixup_blob_32x32x48_tile16", 2, [0, 16, 48]
    ranks = launch("restart", case, world, tmp_path, port_of("restart"), cuts=cuts)
    for r in ranks:
        assert int(r["set_rc"]) == PS_SUCCESS and list(r["cuts"]) == cuts
        assert int(r["local"]) == 0, "the boundary fix-up has work: the setup must have restarted replicated"
    parity.check_distributed(case, ranks)


def test_scene_moving_along_z(built, tmp_path):
    ranks = launch("move", "offz_blob_tile16", 2, tmp_path, port_of("move"))
    for r in ranks:
        for name in ("low", "high"):
            assert int(r[f"{name}_rb"]) == PS_SUCCESS, f"{name}: the first step's loads must move the cuts"
            assert list(r[f"{name}_rebalanced_cuts"]) != list(r[f"{name}_first_cuts"])
            for phase in ("first", "rebalanced"):
                assert int(r[f"{name}_{phase}_set"]) == PS_SUCCESS
                assert bool(r[f"{name}_{phase}_same"]), f"{name} scene, {phase} step: not the fresh handle's result on the same cuts"
    lo, hi = list(ranks[0]["low_rebalanced_cuts"]), list(ranks[0]["high_rebalanced_cuts"])
    assert lo[1] < 48 < hi[1], f"cuts {lo} for the low scene, {hi} for the high one"


def test_one_rank(built):
    sc, ov = parity.DIST_CASES["offz_blob_tile16"]()
    s = PolyStokesSolver.from_scene(sc, lib_path=parity.EMUL_LIB, **ov)
    assert s.rebalance()[0] == PS_INVALID
    s.setup_scene(sc)
    T = unit_model(Oracle(sc, **ov).setup(), sc.nz, 16)
    assert np.array_equal(s.vector("unitCounts").reshape(-1, 9).astype(np.int64), T)
    assert float(s.vector("unitLoad").sum()) == s.kernel_bytes("cg_iteration")
    assert s.rebalance() == (PS_NOCHANGE, [0, sc.nz])
    assert s.set_partition([0, sc.nz]) == PS_SUCCESS and s.set_partition(None) == PS_SUCCESS
    assert s.set_partition([0, 16]) == PS_INVALID
    assert s.partition()[4] == [0, sc.nz]
    s.close()

"""Reduced regions that cross the slab cuts (doTile off, tilePadding 0) on N > 1 ranks, on CPU: world_size-2 / -3 / -4 gloo jobs
drive the host-emulation twin (tests/spanning_worker.py); the merged result is compared with the single-process oracle through
parity.check_distributed, with the gates of the other distributed cases.  A region whose reduced faces lie in several slabs is
shared: its rows follow the slab of the face, and every apply sums its moments over the ranks."""
import os
import subprocess
import sys

import numpy as np
import pytest

import parity
import spanning_cases

HERE = os.path.dirname(os.path.abspath(__file__))


def launch(case, world, outdir, port, gpu=False, extra_env=None, timeout=600):
    env = dict(os.environ, **(extra_env or {}))
    env = dict(env, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WORLD_SIZE=str(world), OMP_NUM_THREADS="2")
    procs = [subprocess.Popen([sys.executable, os.path.join(HERE, "spanning_worker.py"), case, str(outdir)] + (["gpu"] if gpu else []),
                              env=dict(env, RANK=str(r), LOCAL_RANK=str(r)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT) for r in range(world)]
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
    return [np.load(os.path.join(outdir, f"rank{r}.npz")) for r in range(world)]


def run(case, world, outdir, port, **kw):
    """launch() with the single-region inputs of parity.write_region_probes."""
    spanning_cases.register()
    parity.write_region_probes(case, outdir)
    return launch(case, world, outdir, port, **kw)


def check(case, ranks):
    """The oracle comparison plus what is particular to shared regions."""
    spanning_cases.register()
    world = len(ranks)
    shared = [int(r["shared"]) for r in ranks]
    assert len(set(shared)) == 1, f"ranks disagree on the shared regions: {shared}"
    R = int(ranks[0]["count_regionCount"])
    print(f"{case} on {world} ranks: cuts {[int(c) for c in ranks[0]['cuts']]}, regionCount {R}, sharedRegions {shared[0]}; per rank regionPath "
          f"{[int(r['count_regionPath']) for r in ranks]}, maxRegionRows {[int(r['count_maxRegionRows']) for r in ranks]}", flush=True)
    min_regions, min_shared = spanning_cases.MIN_COUNTS[case][world]
    assert R >= min_regions and shared[0] >= min_shared, f"{R} regions, {shared[0]} shared: the case needs >= {min_regions} / {min_shared}"
    if case not in spanning_cases.NO_SHARED:      # padded tiles keep the slab rules of regions that never cross a cut
        # the same number of shared regions as the rule applied to the oracle's classification
        expect = spanning_cases.shared_regions(parity.dist_reference(case)["o"], ranks[0]["cuts"])
        assert shared[0] == len(expect), f"{shared[0]} shared regions, the oracle's classification gives {len(expect)}"
    if case in spanning_cases.NO_SHARED:
        assert shared[0] == 0, f"{shared[0]} shared regions with padded tiles"
    else:
        assert shared[0] > 0, "no region crosses a cut: the case does not test what it should"
    assert all(int(r["local"]) == 0 for r in ranks), "regions crossing cuts need the replicated setup"
    if shared[0] > 0:     # every apply of the step sums the moments once: CG + recovery at least
        assert all(int(r["peerExchanges"]) + int(r["commExchanges"]) >= int(r["iterations"]) + 1 for r in ranks)
    if case in spanning_cases.SWITCH:
        assert all(list(r["first_cuts"]) != list(r["cuts"]) for r in ranks), "the cuts must move when doTile changes"
        assert all(int(r["first_shared"]) == 0 and int(r["first_rc"]) == 1 for r in ranks)
        assert all(bool(r["back_ok"]) for r in ranks), "switching back to the first tiling does not reproduce its step"
    io, its = parity.check_distributed(case, ranks)
    # velSolution: every region reported once, by its owner -- the sum over the ranks is the global vector
    vs = sum(r["velSolution"] for r in ranks)
    assert np.all(np.isfinite(vs))
    return io, its


CASES = ["span_blob64_notile", "span_blob64_tile8_pad0", "span_blob64_tile16_pad0", "span_blob64_notile_bicgstab6", "span_bodies_notile"]


@pytest.mark.parametrize("world", [2, 3, 4])
@pytest.mark.parametrize("case", CASES)
def test_spanning_regions_match_oracle(built, tmp_path, case, world):
    port = 29300 + (os.getpid() + hash(case) + 17 * world) % 300
    ranks = run(case, world, tmp_path, port)
    assert all(int(r["peerExchanges"]) == 0 for r in ranks)        # no peer memory in the emulation twin: the communicator sums
    check(case, ranks)


def test_switch_between_tiled_and_untiled_moves_the_cuts(built, tmp_path):
    """24^3 tiles cut at multiples of 48, no tiles at multiples of 16: 2 ranks are the only world size where both fit 64 layers."""
    port = 29200 + os.getpid() % 50
    check("span_blob64_switch_tile_notile", run("span_blob64_switch_tile_notile", 2, tmp_path, port))


def test_unpadded_tile8_gate_reflects_the_single_rank_difference(built):
    """The 1e-3 velocity gate of span_blob64_tile8_pad0 (spanning_cases.VEL_GATE) is needed on ONE rank already: the twin and the
    oracle, two correct CG runs, stop at velocities further apart than 10 x tol, and well inside the gate."""
    from oracle.oracle import Oracle
    from polystokes_b200 import PolyStokesSolver
    sc, ov = spanning_cases.CASES["span_blob64_tile8_pad0"]()
    o = Oracle(sc, **ov).setup()
    assert o.solve() == 1
    ovel, _ = o.writeback()
    s = PolyStokesSolver.from_scene(sc, lib_path=parity.EMUL_LIB, **ov)
    rc, vel, _ = s.step_scene(sc)
    s.close()
    assert rc == 1
    worst = max(float(np.abs(ovel[a] - vel[a]).max()) / max(float(np.abs(ovel[a]).max()), 1e-30) for a in range(3))
    tol = sc.params["tolerance"]
    assert 10 * tol < worst <= 0.5 * spanning_cases.VEL_GATE["span_blob64_tile8_pad0"], f"single-rank difference {worst:.2e}"


def test_padded_tiles_share_nothing(built, tmp_path):
    port = 29250 + os.getpid() % 50
    check("span_blob64_tile8_pad1", run("span_blob64_tile8_pad1", 3, tmp_path, port))


def test_bodies_scene_covers_the_sharing_cases():
    """span_bodies_notile at 4 ranks (cuts 16 / 32 / 48), by the sharing rule applied to the oracle's classification: what its
    comment in spanning_cases claims, so that a change of the scene cannot quietly drop a case."""
    from oracle.oracle import Oracle
    sc, ov = spanning_cases.CASES["span_bodies_notile"]()
    o = Oracle(sc, **ov).setup()
    cuts = [0, 16, 32, 48, 64]
    sh = spanning_cases.shared_regions(o, cuts)
    cells = o.index_field(2, 0)
    R = o.count("regionCount")
    zr = [np.nonzero((cells == r).any(axis=(1, 2)))[0] for r in range(R)]
    owner = [int(np.searchsorted(cuts, z[0], side="right") - 1) for z in zr]
    assert R == 6 and sorted(sh) == [0, 3, 4], (R, sh)
    assert sh[0] == (0, [0, 1, 2, 3]), "region 0 crosses every cut, owned by rank 0"
    assert owner[2] == 1 and 2 not in sh and zr[2][0] >= 16 and zr[2][-1] < 32, "region 2 lies inside slab 1, unshared"
    assert owner[4] == 2 and min(r for r in sh if 2 in sh[r][1]) < 2 < 4, "rank 2 builds region 2 (between shared region 0 and its own 4)"
    assert zr[4][-1] == 47 and sh[4] == (2, [2, 3]), "region 4: cells below z = 48, shared through its z-faces on that plane"
    assert sh[3] == (1, [1, 2, 3]), "region 3 crosses z = 32 and 48, not 16"
    assert 1 in (owner[r] for r in range(R) if r not in sh) and any(owner[r] == 1 for r in sh) and any(owner[r] < 1 and 1 in sh[r][1] for r in sh), \
        "rank 1: own unshared, own shared and lower rank's shared regions"

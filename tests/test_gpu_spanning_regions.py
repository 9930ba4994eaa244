"""Reduced regions that cross the slab cuts on real GPUs: one process per GPU (the NVLink peer transport, whose symmetric blocks
also carry the shared-region moments, or NCCL), merged result against the oracle,
and the ps_create_multi handle against the single-GPU handle.  Every case runs in child processes under a time-out."""
import os
import subprocess
import sys

import pytest

from test_distributed_spanning_emul import check, run

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _ngpu():
    import torch
    return torch.cuda.device_count()


# every case at 2 and 4 ranks on both transports (64-layer grids hold at most four 16-layer slabs); 8 ranks on S3 128^3 untiled;
# the doTile switch at 2 ranks, the only world size where both of its cut units (48 and 16) fit 64 layers; the multi-region scene at
# 2, 3 and 4 ranks
CASES = ["span_blob64_notile", "span_blob64_tile8_pad0", "span_blob64_tile16_pad0", "span_blob64_notile_bicgstab6"]
RUNS = ([(c, w) for c in CASES for w in (2, 4)] + [("span_blob64_switch_tile_notile", 2), ("span_blob64_tile8_pad1", 4), ("span_s3_128_notile", 8)]
        + [("span_bodies_notile", w) for w in (2, 3, 4)])


@pytest.mark.parametrize("transport", ["peer", "nccl"])
@pytest.mark.parametrize("case,world", RUNS)
def test_gpu_spanning_regions_match_oracle(built, tmp_path, case, world, transport):
    if _ngpu() < world:
        pytest.skip(f"needs {world} GPUs")
    port = 29500 + (os.getpid() + hash(case) + world + (7 if transport == "nccl" else 0)) % 90
    ranks = run(case, world, tmp_path, port, gpu=True, extra_env={"PS_COMM": "nccl" if transport == "nccl" else ""}, timeout=300)
    assert all(int(r["peer"]) == (1 if transport == "peer" else 0) for r in ranks), "requested transport not in use"
    if int(ranks[0]["shared"]) > 0:
        # the shared-region moments took the requested transport too: peer memory, or the communicator's all-reduce
        if transport == "peer":
            assert all(int(r["peerExchanges"]) > 0 and int(r["commExchanges"]) == 0 for r in ranks), "shared moments did not travel by peer memory"
        else:
            assert all(int(r["peerExchanges"]) == 0 and int(r["commExchanges"]) > 0 for r in ranks)
    if case == "span_bodies_notile":
        # the unshared regions on the one-CTA reduced_region_kernel (shared rows do not count towards maxRegionRows), next to the shared
        # regions on the chunked kernels: every rank holds rows of region 0, which crosses every cut
        paths = [int(r["count_regionPath"]) for r in ranks]
        assert all(p in (0, 1) for p in paths), f"regionPath per rank {paths}: expected the one-CTA region kernel (0 or 1)"
    check(case, ranks)


@pytest.mark.parametrize("case", ["span_pillars_over_cap", "span_pillars_under_cap"])
def test_gpu_shared_moments_beyond_the_peer_area(built, tmp_path, case):
    """More shared regions than the peer moment area holds: under the peer transport the communicator's all-reduce sums them; just
    fewer: peer memory.  Then the whole oracle comparison."""
    if _ngpu() < 2:
        pytest.skip("needs 2 GPUs")
    port = 29600 + (os.getpid() + hash(case)) % 90
    ranks = run(case, 2, tmp_path, port, gpu=True, extra_env={"PS_COMM": ""}, timeout=600)
    assert all(int(r["peer"]) == 1 for r in ranks), "peer transport not in use"
    shared, cap = int(ranks[0]["shared"]), int(ranks[0]["count_peerSharedCap"])
    print(f"{case}: sharedRegions {shared}, peer capacity {cap}, exchanges by peer memory {[int(r['peerExchanges']) for r in ranks]}, "
          f"by the communicator {[int(r['commExchanges']) for r in ranks]}", flush=True)
    if case == "span_pillars_over_cap":
        assert shared > cap
        assert all(int(r["commExchanges"]) > 0 and int(r["peerExchanges"]) == 0 for r in ranks), "the communicator must sum them"
    else:
        assert 0 < shared <= cap
        assert all(int(r["peerExchanges"]) > 0 and int(r["commExchanges"]) == 0 for r in ranks), "shared moments did not travel by peer memory"
    check(case, ranks)


@pytest.mark.parametrize("case,ndev", [("span_blob64_notile", 2), ("span_blob64_tile8_pad0", 4), ("span_s3_128_notile", 8), ("span_bodies_notile", 4)])
def test_gpu_multi_handle_spanning_matches_single_gpu(built, case, ndev):
    if _ngpu() < ndev:
        pytest.skip(f"needs {ndev} GPUs")
    env = dict(os.environ, PS_MULTI_WATCHDOG_S="45")
    try:
        r = subprocess.run([sys.executable, os.path.join(HERE, "spanning_multi_worker.py"), case, str(ndev)], capture_output=True, text=True, timeout=300, env=env)
    except subprocess.TimeoutExpired as e:
        pytest.fail(f"multi-GPU handle hung on {case} x {ndev}:\n{e.stderr}")
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]

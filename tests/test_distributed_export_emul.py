"""ps_export on a slab-decomposed handle, on CPU: world_size-N gloo jobs drive the host-emulation twin (tests/export_worker.py).  Every rank
calls ps_export, rank 0 writes the file set of one rank, and that set must equal the export of a plain handle on the same scene: the
component matrices and vectors, Mat_A, Vec_b and Vec_guess byte for byte, dimData except the thread count, the guess against the oracle,
the solution by the reference's stop rule.  A write that fails on rank 0 fails on every rank and leaves the handles usable."""
import json
import os
import subprocess
import sys

import pytest

import export_worker

HERE = os.path.dirname(os.path.abspath(__file__))

# (case, world, export through ps_step's toggles)
RUNS = [("blob48_tile8", 2, False),                 # replicated setup, tiles padded by 1
        ("blob64_tile16", 2, False), ("blob64_tile16", 4, True),      # slab-local setup
        ("blob_36x40x64_tile16", 3, False),
        ("box48_uniform", 2, False),                # no reduced regions
        ("span_bodies_notile", 2, True), ("span_bodies_notile", 3, False), ("span_bodies_notile", 4, False),   # shared and unshared regions
        ("span_blob64_tile8_pad0", 3, False)]       # unpadded tiles crossing the cuts


def run(args, env=None, timeout=900):
    r = subprocess.run([sys.executable, os.path.join(HERE, "export_worker.py")] + args, capture_output=True, text=True, timeout=timeout,
                       env=dict(os.environ, OMP_NUM_THREADS="2", **(env or {})))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]


def launch(case, world, outdir, port, auto, gpu=False, timeout=900, extra_env=None):
    env = dict(os.environ, **(extra_env or {}))
    env = dict(env, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WORLD_SIZE=str(world), OMP_NUM_THREADS="2", EXPORT_AUTO="1" if auto else "0")
    procs = [subprocess.Popen([sys.executable, os.path.join(HERE, "export_worker.py"), "rank", case, str(outdir)] + (["gpu"] if gpu else []),
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
    return [json.load(open(os.path.join(outdir, f"rank{r}.json"))) for r in range(world)]


def check_records(ranks, ref):
    """Every rank: the step's result, the failing export (PS_FAILED naming the prefix) and the step + export after it."""
    for k, r in enumerate(ranks):
        assert r["rc"] == ref["rc"] == 1, f"rank {k}: step result {r['rc']} (one rank: {ref['rc']})"
        assert r["bad_rc"] == -1, f"rank {k}: export into a missing directory returned {r['bad_rc']}"
        assert r["bad_prefix"] in r["bad_error"], f"rank {k}: ps_last_error {r['bad_error']!r} does not name the prefix"
        assert r["again_rc"] == 1 and r["again_export"] == 1, f"rank {k}: step / export after the failed write: {r['again_rc']} / {r['again_export']}"
    assert len({r["iterations"] for r in ranks}) == 1
    n_again = [len(os.listdir(os.path.join(os.path.dirname(os.path.dirname(r["bad_prefix"])), "again", f"rank{k}"))) for k, r in enumerate(ranks)]
    assert n_again == [len(export_worker.FILES)] + [0] * (len(ranks) - 1), f"files of the export after the failed write: {n_again}"


@pytest.mark.parametrize("case,world,auto", RUNS)
def test_distributed_export_matches_one_rank(built, tmp_path, case, world, auto):
    port = 29600 + (os.getpid() + hash(case) + 17 * world) % 300
    run(["ref", case, str(tmp_path)])
    ranks = launch(case, world, tmp_path, port, auto)
    ref = json.load(open(os.path.join(tmp_path, "ref", "ref.json")))
    check_records(ranks, ref)
    export_worker.compare(case, str(tmp_path), world)

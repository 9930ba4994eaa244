"""ps_export and the global views on real GPUs (tests/export_worker.py): the ps_create_multi handle at 2, 4 and 8 GPUs and one process per
GPU at 2 ranks (NVLink peer transport, or NCCL alone) export the file set of a single-GPU handle; the multi handle passes the oracle
checks of parity as `s`, its ps_get_csr blocks equal the single-GPU handle's, and ps_step's automatic export changes nothing in the step.
Every case runs in child processes under a time-out; a case skips when there are too few GPUs."""
import json
import os

import pytest

import export_worker
from test_distributed_export_emul import check_records, launch, run

pytestmark = pytest.mark.gpu
CASES = ["blob64_tile16", "blob48_tile8", "span_bodies_notile"]      # slab-local (tilePadding 2), replicated (tilePadding 1), shared regions
NZ = {"blob64_tile16": 64, "blob48_tile8": 48, "span_bodies_notile": 64, "s3_128": 128}


def _ngpu():
    import torch
    return torch.cuda.device_count()


def _need(ndev, case):
    if _ngpu() < ndev:
        pytest.skip(f"needs {ndev} GPUs")
    if NZ[case] < 16 * ndev:
        pytest.skip("fewer 16-layer slabs than devices")


@pytest.mark.parametrize("ndev", [2, 4, 8])
@pytest.mark.parametrize("case", CASES)
def test_multi_handle_export_matches_single_gpu(built, tmp_path, case, ndev):
    _need(ndev, case)
    run(["ref", case, str(tmp_path), "gpu"], env={"PS_MULTI_WATCHDOG_S": "45"}, timeout=300)
    run(["multi", case, str(tmp_path), str(ndev)], env={"PS_MULTI_WATCHDOG_S": "45"}, timeout=300)
    ref = json.load(open(os.path.join(tmp_path, "ref", "ref.json")))
    check_records([json.load(open(os.path.join(tmp_path, "rank0.json")))], ref)
    export_worker.compare(case, str(tmp_path), ndev)


@pytest.mark.parametrize("transport", ["peer", "nccl"])
@pytest.mark.parametrize("case", CASES)
def test_one_process_per_gpu_export_matches_single_gpu(built, tmp_path, case, transport):
    _need(2, case)
    run(["ref", case, str(tmp_path), "gpu"], timeout=300)
    port = 29800 + (os.getpid() + hash(case) + (7 if transport == "nccl" else 0)) % 150
    ranks = launch(case, 2, tmp_path, port, auto=False, gpu=True, timeout=300, extra_env={"PS_COMM": "nccl" if transport == "nccl" else ""})
    check_records(ranks, json.load(open(os.path.join(tmp_path, "ref", "ref.json"))))
    export_worker.compare(case, str(tmp_path), 2)


@pytest.mark.parametrize("case,ndev", [(c, n) for c in CASES for n in (2, 4)] + [("s3_128", 8)])
def test_multi_handle_views_match_oracle(built, case, ndev):
    _need(ndev, case)
    run(["views", case, "-", str(ndev)], env={"PS_MULTI_WATCHDOG_S": "45"}, timeout=600)


@pytest.mark.parametrize("case", ["span_bodies_notile", "blob64_tile16"])
def test_multi_handle_automatic_export(built, tmp_path, case):
    _need(2, case)
    run(["auto", case, str(tmp_path), "2"], env={"PS_MULTI_WATCHDOG_S": "45"}, timeout=300)

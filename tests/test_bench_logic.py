"""Host logic of bench.py that runs without a GPU: the choice of the reference arm's grid (a measured, unscaled run of the compiled reference at
the largest S3 grid that fits the time / memory budget -- 256^3, the metric's own configuration, on the GPU box's host) and the per-machine cache
that lets the N > 1 lines of a scaling run reuse the N = 1 measurement; the --dump-outputs writer."""
import importlib.util
import json
import os
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_reference_grid_follows_the_budget(monkeypatch):
    b = _bench()
    monkeypatch.setattr(b, "mem_available_gb", lambda: 196.0)
    cal = {"n": 64, "seconds": 3.1, "cg_s": 1.2, "maxrss_gb": 1.6}        # the calibration run of profiles/r02_bench_ref_n1_v8_measured_256.json
    n, pred_s, pred_gb = b.choose_ref_grid(1500.0, cal)
    assert n == 256 and 600 < pred_s < 1100 and pred_gb < 0.7 * 196       # measured there: 917 s, 92 GB
    assert b.choose_ref_grid(600.0, cal)[0] == 192
    assert b.choose_ref_grid(100.0, cal)[0] == 128
    monkeypatch.setattr(b, "mem_available_gb", lambda: 62.0)               # a small host: memory, not time, decides
    assert b.choose_ref_grid(1500.0, cal)[0] < 256


def test_reference_run_cache_is_per_boot_and_expires(tmp_path, monkeypatch):
    b = _bench()
    monkeypatch.setattr(b, "REF_CACHES", [str(tmp_path / "a" / "run.json"), str(tmp_path / "b" / "run.json")])
    assert b.ref_cache_load() is None
    b.ref_cache_store({"scene": "S3", "kind": "reference", "n": 256, "seconds": 916.9, "cores": 16})
    got = b.ref_cache_load()
    assert got["n"] == 256 and got["seconds"] == 916.9
    os.remove(b.REF_CACHES[0])                                             # the second location alone is enough
    assert b.ref_cache_load()["n"] == 256
    stale = json.load(open(b.REF_CACHES[1]))
    json.dump(dict(stale, boot_id="another-machine"), open(b.REF_CACHES[1], "w"))
    assert b.ref_cache_load() is None
    json.dump(dict(stale, time=time.time() - 13 * 3600), open(b.REF_CACHES[1], "w"))
    assert b.ref_cache_load() is None


def test_dump_outputs_writes_fp32_fields_and_a_fixed_sample_of_large_ones(tmp_path, monkeypatch):
    import numpy as np
    b = _bench()
    monkeypatch.setattr(b, "DUMP_MAX_ENTRIES", 1000)
    rng = np.random.default_rng(1)
    small = [rng.standard_normal((4, 5, 6)).astype(np.float32) for _ in range(3)]
    large = [rng.standard_normal((20, 10, 10)).astype(np.float32) for _ in range(3)]
    for run in ("a", "b"):
        b.dump_outputs(str(tmp_path / run), small, large)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == [f"{k}{ax}.npy" for k in ("valid", "vel") for ax in range(3)]
    for ax in range(3):
        vel = np.load(tmp_path / "a" / f"vel{ax}.npy")
        assert vel.dtype == np.float32 and np.array_equal(vel, small[ax])               # small enough: the whole field, shape kept
        valid = np.load(tmp_path / "a" / f"valid{ax}.npy")
        assert valid.dtype == np.float32 and valid.shape == (1000,)
        assert np.isin(valid, large[ax]).all()                                             # a sample of the field's own entries ...
        assert np.array_equal(valid, np.load(tmp_path / "b" / f"valid{ax}.npy"))          # ... at the same positions on every run

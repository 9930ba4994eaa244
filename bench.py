#!/usr/bin/env python
"""bench.py -- Stokes steps/sec (classify + assemble + PCG + write-back) at 256^3 on N B200s.

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, through the C ABI)
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU path (oracle restatement)
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's output fields to DIR/*.npy

A *step* is one full solveGasSubclass body (exec/HDK_PolyStokes.C:344-584) on the synthetic scene S3
(SURVEY.md section 8d; BASELINE.json configs[2], the single-GPU 256^3 configuration the metric is quoted on).
Prints ONE JSON line (rank 0).  See DESIGN.md section 6 for how every number is obtained.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the tree it runs from as it found it (it may be read-only)

METRIC = "stokes_steps_per_sec_256cubed"
UNIT = "steps/s"
SCENE_N = 256


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


# The reference arm's measured run is remembered on THIS machine (same boot, at most 12 h old) so that the N > 1 lines of a scaling run reuse
# the N = 1 measurement instead of spending another quarter of an hour of host time each: the CPU path does not depend on N.
REF_CACHES = [os.path.join(tempfile.gettempdir(), "polystokes_b200_reference_run.json")]


def _boot_id():
    try:
        with open("/proc/sys/kernel/random/boot_id") as f:
            return f.read().strip()
    except Exception:
        return "unknown"


def ref_cache_load():
    for path in REF_CACHES:
        try:
            with open(path) as f:
                res = json.load(f)
            if res.get("scene") == "S3" and res.get("kind") is not None and res.get("boot_id") == _boot_id() and time.time() - float(res.get("time", 0)) < 12 * 3600:
                return res
        except Exception:
            continue
    return None


def ref_cache_store(res):
    res = dict(res, boot_id=_boot_id(), time=time.time())
    for path in REF_CACHES:
        try:
            os.makedirs(os.path.dirname(path), exist_ok=True)
            with open(path, "w") as f:
                json.dump(res, f)
        except Exception:
            pass


def reference_available():
    try:
        from oracle import ref_full
        return ref_full.available()
    except Exception:
        return False


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def mem_available_gb():
    try:
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable:"):
                return float(ln.split()[1]) / 1e6
    except Exception:
        pass
    return 0.0


def _ref_verify(R, sc, res):
    """Item by item against the committed digest of this configuration (tests/golden/fullsize_S3.json, made from the oracle): the compiled
    reference at FULL size must give the same counts, label / index / weight fields (SHA-256), G and D^T (pattern + values), |b|, iteration count
    (within 1 %: the setup sums are accumulated per job), valid masks and -- within 10 x tol -- the velocity sample."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import make_fullsize as mf
    path = os.path.join(ROOT, "tests", "golden", "fullsize_S3.json")
    if sc.nx != SCENE_N or not os.path.exists(path):
        return None
    with open(path) as f:
        g = json.load(f)
    bad = [k for k in mf.COUNTS if R.count(k) != g["counts"][k]]
    fields = mf.field_digests(R.index_field, R.weight_field)
    bad += [k for k in fields if fields[k] != g["fields"][k]]
    csr = mf.csr_digests(R.csr)
    bad += [f"csr {m} {qq}" for m in csr for qq in ("shape", "nnz", "pattern", "values") if csr[m][qq] != g["csr"][m][qq]]
    b = R.vector("b")
    bn = float(np.sqrt(np.dot(b, b)))
    if abs(bn - g["b_norm"]) > 1e-10 * g["b_norm"]:
        bad.append(f"b_norm {bn} vs {g['b_norm']}")
    if abs(res["iterations"] - g["iterations"]) > max(2, g["iterations"] // 100):
        bad.append(f"iterations {res['iterations']} vs {g['iterations']}")
    vel = [R.face_field(0, a) for a in range(3)]; valid = [R.face_field(1, a) for a in range(3)]
    got = mf.velocity_sample(vel, valid)
    worst = max(float(np.abs(np.array(g[f"vel{a}_sample"]) - np.array(got[f"vel{a}_sample"])).max()) / g[f"vel{a}_absmax"] for a in range(3))
    if worst > 10 * sc.params["tolerance"]:
        bad.append(f"velocity sample rel diff {worst:.2e}")
    bad += [f"valid{a}" for a in range(3) if got[f"valid{a}"] != g[f"valid{a}"]]
    return {"equal": not bad, "mismatches": bad, "velocity_sample_max_rel_diff": worst,
            "checked": "14 counts, 35 field hashes, G / D^T patterns + values, |b|, iterations, valid masks, velocity sample (10 x tol)"}


def _ref_worker(n, threads, q):
    """One COMPLETE step of the REFERENCE'S OWN solver on S3 at n^3 (child process, so its memory goes back to the OS).

    The solver is all of exec/HDK_PolyStokesSolver*.cpp + lib/, compiled unmodified into oracle/_ref/libps_ref_full.so on the HDK stand-in /
    Eigen facade, driven in the stage order of exec/HDK_PolyStokes.C:344-584.  Threads: `threads` jobs behind UT_ThreadedAlgorithm /
    UTparallelFor / tbb::parallel_for (setup sweeps), OpenMP for Eigen's row-parallel SpMV and the 3 `omp sections` of the operator apply
    (lib/include/ApplyPressureStressMatrix.h:122-164; nested regions are serial, as in the real plugin)."""
    import resource
    from polystokes_b200 import scenes
    from oracle import ref_full
    os.environ.setdefault("OMP_NUM_THREADS", str(threads))
    L = ref_full.lib()
    jobs = L.reffull_set_threads(int(threads))
    sc = scenes.scene_s3(n)
    devnull = os.open(os.devnull, os.O_WRONLY); saved = os.dup(1); os.dup2(devnull, 1)      # the reference chats on stdout
    try:
        t0 = time.perf_counter()
        R = ref_full.RefFull(sc).setup()
        t_setup = time.perf_counter() - t0
        t0 = time.perf_counter()
        rc = R.solve()
        t_solve = time.perf_counter() - t0
    finally:
        os.dup2(saved, 1); os.close(saved); os.close(devnull)
    out = dict(n=n, seconds=t_setup + t_solve, setup_s=t_setup, solve_s=t_solve, cg_s=R.real("solveWallclockMs") * 1e-3, iterations=int(R.count("iterations")),
               nSystemSize=int(R.count("nSystemSize")), result=int(rc), jobs=int(jobs), cores=int(threads),
               maxrss_gb=resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 1e6)
    if os.environ.get("PS_REF_VERIFY", "1") != "0":
        try:
            out["digest_check"] = _ref_verify(R, sc, out)
        except Exception as e:          # the measurement stands even if the check cannot run
            out["digest_check"] = {"equal": None, "error": repr(e)}
    R.close()
    q.put(out)


def run_ref_full(n, threads=None):
    """Measured, unscaled: one full step of the compiled reference at n^3 with all host cores."""
    import multiprocessing as mp
    threads = threads or host_cores()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    pr = ctx.Process(target=_ref_worker, args=(n, threads, q))
    pr.start()
    res = None
    while res is None:
        try:
            res = q.get(timeout=1.0)
        except Exception:
            if not pr.is_alive():
                raise RuntimeError(f"reference run at {n}^3 died (exit code {pr.exitcode}; out of memory?)")
    pr.join()
    return res


def choose_ref_grid(budget_s, cal):
    """Largest S3 grid whose predicted reference time fits `budget_s` and whose predicted memory fits the host.  `cal` is a measured run at a small
    grid; setup scales with the voxel count, CG with rows x iterations (iterations ~ n on S3: 63 / 97 / 129 / 258 at 64 / 96 / 128 / 256) times a
    cache factor: the 64^3 system (0.3 M rows) iterates out of the host's caches, the larger ones from DRAM -- measured on the GPU box's 16-core host
    (profiles/r02_bench_ref_n1_v8.json): 120 ns per row and iteration at 96^3, 190 ns at 256^3, i.e. ~2 x the calibration's rate."""
    avail = mem_available_gb()
    for n in (256, 192, 128, 96):
        f3 = (n / cal["n"]) ** 3
        dram = 2.0 if n >= 160 else 1.5 if n >= 96 else 1.0
        pred_s = (cal["seconds"] - cal["cg_s"]) * f3 + cal["cg_s"] * f3 * (n / cal["n"]) * dram
        pred_gb = cal["maxrss_gb"] * f3 * 1.15
        if pred_s <= budget_s and pred_gb <= 0.7 * avail:
            return n, pred_s, pred_gb
    return cal["n"], cal["seconds"], cal["maxrss_gb"]


def run_cpu_sample(n, threads=0):
    """One full step of the oracle (CPU restatement, OpenMP) on S3 at n^3; measured seconds, no scaling."""
    from polystokes_b200 import scenes
    from oracle.oracle import Oracle, lib
    sc = scenes.scene_s3(n)
    t0 = time.perf_counter()
    o = Oracle(sc, threads=threads).setup()
    t_setup = time.perf_counter() - t0
    t0 = time.perf_counter()
    o.solve()
    o.writeback()
    t_solve = time.perf_counter() - t0
    return dict(n=n, seconds=t_setup + t_solve, setup_s=t_setup, solve_s=t_solve, iterations=int(o.count("iterations")), nSystemSize=int(o.count("nSystemSize")),
                cores=lib().orc_num_threads())


def bench_multi(a, sc, config, metric):
    """ONE process, a.gpus devices behind one ps_create_multi handle (the way a single cook thread would drive several GPUs): e2e only -- the
    handle takes the caller's full-grid HOST arrays, every rank uploads / downloads its slab."""
    import numpy as np
    import torch
    from polystokes_b200 import PolyStokesSolver, PS_SUCCESS
    solver = PolyStokesSolver.from_scene(sc, devices=list(range(a.gpus)))
    pin = lambda x: torch.from_numpy(np.ascontiguousarray(x)).pin_memory()
    h_in = [pin(sc.surface), pin(sc.collision), pin(sc.viscosity)]
    h_vel = [pin(v) for v in sc.vel]; h_cvel = [pin(v) for v in sc.colvel]
    h_out = [torch.empty_like(v).pin_memory() for v in h_vel]; h_valid = [torch.empty_like(v).pin_memory() for v in h_vel]
    npv = lambda ts: [t.numpy() for t in ts]

    def step():
        rc = solver.step(h_in[0].numpy(), h_in[1].numpy(), h_in[2].numpy(), npv(h_vel), npv(h_cvel), npv(h_out), npv(h_valid))
        if rc != PS_SUCCESS:
            raise SystemExit(f"bench.py: solver returned {rc}")
    for _ in range(max(a.warmup, 1)):
        step()
    sampler = ClockSampler(0)
    sampler.start()
    t0 = time.perf_counter()
    launches = 0
    for _ in range(a.steps):
        step()
        launches += int(solver.stats.gpu_launches)
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, h_out, h_valid)
    value = a.steps / wall
    counts = {k: solver.count(k) for k in ["nCenter", "nActiveVs", "nSystemSize", "regionCount", "nRowsExt", "nTotalDOFs", "iterations"]}
    h2d = sum(t.numel() * 4 for t in h_in + h_vel + h_cvel); d2h = sum(t.numel() * 4 for t in h_out + h_valid)
    emit({"metric": metric, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": wall / a.steps * 1e3, "higher_is_better": True,
          "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
          "config": dict(config, parallelism=f"ONE process, one ps_create_multi handle over {a.gpus} GPUs (one host thread per GPU, slab-local upload / download of the caller's host arrays)",
                         counts=counts, timing="host clock around K calls of ps_step with pinned host arrays"),
          "stage_ms": {k: round(v, 3) for k, v in solver.stage_ms().items()}, "cg_iterations": counts["iterations"], "clocks": clocks,
          "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": wall / a.steps * 1e3}, "gpu_launches": launches,
          "roofline": None, "cpu_baseline": None})
    solver.close()


def emit(obj):
    """The ONE JSON line of the contract, on the real stdout (see main: fd 1 is pointed at stderr while the bench runs)."""
    os.write(_REAL_STDOUT, (json.dumps(obj) + "\n").encode())


_REAL_STDOUT = 1

# --dump-outputs: at most 2^21 entries (8 MB of fp32) per array, i.e. 48 MB for the 3 velocity + 3 valid face fields
DUMP_MAX_ENTRIES = 1 << 21


def dump_outputs(path, vel, valid):
    """Write what one step handed back to its caller -- the velocity and valid face fields, 3 axes each -- as <path>/vel<axis>.npy and
    <path>/valid<axis>.npy (float32), so that the outputs of two builds can be compared entry for entry.  A field of more than
    DUMP_MAX_ENTRIES entries is written as a sample of its flattened entries at fixed positions: sorted indices drawn without replacement
    by PCG64(0), the same on every run for the same grid."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    for name, t in [(f"vel{ax}", vel[ax]) for ax in range(3)] + [(f"valid{ax}", valid[ax]) for ax in range(3)]:
        t = torch.as_tensor(t)
        if t.numel() > DUMP_MAX_ENTRIES:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_MAX_ENTRIES, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy().astype(np.float32, copy=False))


def main():
    # Libraries chat on stdout (NCCL prints its version banner there when the first communicator is created): keep the
    # real stdout for the result line only and send everything else to stderr.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=SCENE_N, help="grid resolution of S3 (the metric is quoted at 256)")
    ap.add_argument("--scene", default="S3", choices=["S3", "S4", "S5"], help="S3 = BASELINE.json configs[2] (the metric's), S4 = configs[3] (384^3), S5 = configs[4] (512x256x256)")
    ap.add_argument("--tile", type=int, default=0, help="tileSize override (configs[4] sweeps 8 / 16 / 32)")
    ap.add_argument("--multi", action="store_true", help="ONE process, --gpus N devices behind one ps_create_multi handle (host arrays only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--kernel-reps", type=int, default=30)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the velocity / valid fields of the last one to DIR/<name>.npy "
                                                          "(float32; fields of more than 2^21 entries as a fixed sample)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs applies to the CUDA arm (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if a.scene == "S3":
        config = {"workload": f"S3 honey-coil style scene {a.n}^3: floor + pool + jet, reduced tiles 16 pad 2, boundary layers 2/2, CG tol 1e-3 "
                              "(BASELINE.json configs[2])", "grid": [a.n] * 3, "tileSize": a.tile or 16, "tilePadding": 2,
                  "l2": "inputs (9 fp32 grids, 0.6 GB at 256^3) and matrices (>2 GB) exceed the 126 MB L2; no flush needed"}
    elif a.scene == "S4":
        config = {"workload": "S4 armadillos-style pool 384^3 with 6 solid spheres in a solid box, reduced tiles 32 pad 3, boundary layers 3/3, mu 2000, CG tol 1e-4 "
                              "(BASELINE.json configs[3])", "grid": [384] * 3, "tileSize": a.tile or 32, "tilePadding": 3,
                  "l2": "inputs (9 fp32 grids, 2 GB) and matrices exceed the 126 MB L2; no flush needed"}
    else:
        config = {"workload": "S5 jelly-jam style ellipsoidal blob 512x256x256 on a floor, variable viscosity 400 exp(0.7 s(x)), boundary layers 3/3, pad 3, CG tol 1e-3 "
                              "(BASELINE.json configs[4])", "grid": [512, 256, 256], "tileSize": a.tile or 16, "tilePadding": 3,
                  "l2": "inputs (9 fp32 grids, 1.2 GB) and matrices exceed the 126 MB L2; no flush needed"}
    metric = METRIC if (a.scene == "S3" and a.n == SCENE_N) else f"stokes_steps_per_sec_{a.scene}_{'x'.join(str(v) for v in config['grid'])}"

    # ------------------------------------------------------------------ reference arm (CPU)
    # ONE measured, unscaled step of the reference's own solver with every host core, at the largest S3 grid that fits the time / memory budget
    # (256^3 = the metric's configuration if it fits); `config.grid` is what actually ran.  --steps / --warmup do not apply to a run of this
    # length: the line reports steps 1, warmup 0.  Under torchrun only rank 0 works; at N > 1 the N = 1 measurement of this box is reused (the CPU
    # path does not depend on N) and marked "cached".
    if a.impl == "reference":
        if rank != 0:
            return
        cores = host_cores()
        budget = float(os.environ.get("PS_REF_BUDGET_S", "1500"))
        res = None
        cached = False
        if a.gpus > 1:
            res = ref_cache_load()
            cached = res is not None
        if res is None:
            if reference_available():
                if a.n != SCENE_N:
                    n, note = a.n, "grid forced by --n"
                else:
                    cal = run_ref_full(64, cores)
                    n, pred_s, pred_gb = choose_ref_grid(budget, cal)
                    note = (f"grid chosen from a 64^3 calibration run ({cal['seconds']:.1f} s, {cal['maxrss_gb']:.1f} GB): predicted {pred_s:.0f} s / {pred_gb:.0f} GB at {n}^3 "
                            f"against a budget of {budget:.0f} s and {mem_available_gb():.0f} GB available")
                res = run_ref_full(n, cores) if n != 64 or a.n == 64 else cal
                res.update(kind="reference", scene="S3", note=note)
            else:
                n = a.n if a.n != SCENE_N else 128
                res = run_cpu_sample(n)
                res.update(kind="port", scene="S3", note="oracle/_ref absent: the oracle (CPU restatement, OpenMP, all cores) ran instead", cg_s=res["solve_s"], maxrss_gb=0.0, jobs=res["cores"])
            ref_cache_store(res)
        n = res["n"]
        value = 1.0 / res["seconds"]
        config = dict(config, grid=[n] * 3, workload=config["workload"].replace(f"{a.n}^3", f"{n}^3"),
                      same_grid_as_metric=(n == SCENE_N))
        sample = (f"{'the reference solver (exec/HDK_PolyStokesSolver*.cpp + lib/, compiled unmodified into oracle/_ref/libps_ref_full.so)' if res['kind'] == 'reference' else 'the oracle port'}"
                  f" ran ONE complete step on S3 at {n}^3 in {res['seconds']:.1f} s: setup {res['setup_s']:.1f} s ({res['jobs']} jobs), solve + write-back {res['solve_s']:.1f} s "
                  f"({res['iterations']} CG iterations in {res['cg_s']:.1f} s: 3 omp sections, lib/include/ApplyPressureStressMatrix.h:122), n = {res['nSystemSize']} rows, "
                  f"peak RSS {res['maxrss_gb']:.1f} GB; measured, not scaled; {res['note']}" + ("; reused from this box's N = 1 run" if cached else ""))
        emit({"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": 1, "warmup": 0, "ms_per_step": res["seconds"] * 1e3, "higher_is_better": True,
              "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config, "impl": "reference", "cached": cached,
              "reference_digest_check": res.get("digest_check"),
              "cpu_baseline": {"value": value, "unit": UNIT, "cores": res["cores"], "kind": res["kind"], "sample": sample},
              "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        return

    # ------------------------------------------------------------------ our arm (CUDA)
    import numpy as np
    import torch
    from polystokes_b200 import PolyStokesSolver, scenes, PS_SUCCESS

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; polystokes_b200 has no CPU path")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    ov = {"tileSize": a.tile} if a.tile else {}
    sc = scenes.scene_s3(a.n, **ov) if a.scene == "S3" else scenes.scene_s4(384, **ov) if a.scene == "S4" else scenes.scene_s5(1.0, **ov)
    if a.multi:
        return bench_multi(a, sc, config, metric)
    solver = PolyStokesSolver.from_scene(sc, device=local)
    part = None
    if world > 1:
        # ONE scene, z-slab decomposed over the ranks (SURVEY.md 8e): NCCL halo exchange of p / w + two scalar
        # all-reduces per CG iteration inside the library; torch.distributed only carries the NCCL unique id
        part = solver.init_distributed()
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    d_in = [dev(sc.surface), dev(sc.collision), dev(sc.viscosity)]
    d_vel = [dev(v) for v in sc.vel]
    d_cvel = [dev(v) for v in sc.colvel]
    d_out = [v.clone() for v in d_vel]
    d_valid = [torch.zeros_like(v) for v in d_vel]

    def step_device():
        rc = solver.step(d_in[0], d_in[1], d_in[2], d_vel, d_cvel, d_out, d_valid)
        if rc != PS_SUCCESS:
            raise SystemExit(f"bench.py: solver returned {rc}")

    for _ in range(max(a.warmup, 1)):
        step_device()
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    t0 = time.perf_counter()
    solver.timer_start()                   # CUDA event on the solver's own stream (torch events only see torch's stream)
    launches = 0
    dev_ms = 0.0
    for _ in range(a.steps):
        step_device()
        launches += int(solver.stats.gpu_launches)
        dev_ms += sum(solver.stats.stage_ms)
    elapsed = solver.timer_stop() * 1e-3   # records the stop event on that stream and waits for it
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    if dist is not None:
        t = torch.tensor([elapsed, wall], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed, wall = float(t[0].item()), float(t[1].item())
    value = a.steps / elapsed              # N > 1: the SAME 256^3 step, slab-decomposed over the ranks (strong scaling)
    stage_ms = solver.stage_ms()
    counts = {k: solver.count(k) for k in ["nCenter", "nActiveVs", "nSystemSize", "regionCount", "nRowsExt", "nTotalDOFs", "iterations"]}

    # ---- parity of what was just timed (every N): counts, iteration count and a strided sample of the solved velocity against the committed
    #      oracle digest of this configuration (tests/golden/fullsize_*.json; 10 x tol relative, valid masks by SHA-256).  With several ranks every
    #      rank delivers its slab: the slabs are summed into full fields first.  --dump-outputs writes the same full fields.
    parity_checked, parity_note = False, "no committed digest for this configuration"
    gold_path = os.path.join(ROOT, "tests", "golden", f"fullsize_{a.scene}.json")
    check_parity = a.scene == "S3" and a.n == SCENE_N and not a.tile and os.path.exists(gold_path)
    if check_parity or a.dump_outputs:
        outs, vals = [t.clone() for t in d_out], [t.clone() for t in d_valid]
        if dist is not None:
            lo, hi = part[2], part[3]
            for t in outs + vals:
                top = hi if hi < sc.nz else t.shape[0]
                t[:lo] = 0
                t[top:] = 0
                dist.all_reduce(t)
        if a.dump_outputs and rank == 0:
            dump_outputs(a.dump_outputs, outs, vals)
    if check_parity:
        sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
        import make_fullsize
        if rank == 0:
            with open(gold_path) as f:
                gold = json.load(f)
            got = make_fullsize.velocity_sample([t.cpu().numpy() for t in outs], [t.cpu().numpy() for t in vals])
            bad = [k for k, v in gold["counts"].items() if solver.count(k) != v]
            tol = 10 * sc.params["tolerance"]
            worst = max(float(np.abs(np.array(gold[f"vel{ax}_sample"]) - np.array(got[f"vel{ax}_sample"])).max()) / gold[f"vel{ax}_absmax"] for ax in range(3))
            ok = (not bad and abs(counts["iterations"] - gold["iterations"]) <= max(2, gold["iterations"] // 100) and worst <= tol
                  and all(got[f"valid{ax}"] == gold[f"valid{ax}"] for ax in range(3)))
            parity_note = (f"counts {'equal' if not bad else 'DIFFER ' + str(bad)}, iterations {counts['iterations']} vs {gold['iterations']}, velocity sample max rel diff {worst:.2e} "
                           f"(gate {tol:.0e}), valid masks {'equal' if all(got[f'valid{ax}'] == gold[f'valid{ax}'] for ax in range(3)) else 'DIFFER'}")
            if not ok:
                raise SystemExit("bench.py: parity check failed: " + parity_note)
            parity_checked = True
    if check_parity or a.dump_outputs:
        del outs, vals

    # ---- end to end through the public API with HOST (pinned) buffers: H2D + D2H inside the timed region
    pin = lambda x: torch.from_numpy(np.ascontiguousarray(x)).pin_memory()
    h_in = [pin(sc.surface), pin(sc.collision), pin(sc.viscosity)]
    h_vel = [pin(v) for v in sc.vel]
    h_cvel = [pin(v) for v in sc.colvel]
    h_out = [torch.empty_like(v).pin_memory() for v in h_vel]
    h_valid = [torch.empty_like(v).pin_memory() for v in h_vel]
    npv = lambda ts: [t.numpy() for t in ts]

    def step_host():
        rc = solver.step(h_in[0].numpy(), h_in[1].numpy(), h_in[2].numpy(), npv(h_vel), npv(h_cvel), npv(h_out), npv(h_valid))
        if rc != PS_SUCCESS:
            raise SystemExit(f"bench.py: solver returned {rc}")

    step_host()
    barrier()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        step_host()
    barrier()
    e2e_elapsed = time.perf_counter() - t0
    if dist is not None:
        t = torch.tensor([e2e_elapsed], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_elapsed = float(t.item())
    # bytes that cross PCIe per step, all ranks together: every rank moves its slab (+ halo layers of the inputs) with slab-local setup
    h2d = sum(t.numel() * 4 for t in h_in + h_vel + h_cvel)
    d2h = sum(t.numel() * 4 for t in h_out + h_valid)
    if world > 1 and solver.count("slabLocal"):
        halo = 2 * (sc.params["liquidLayers"] + sc.params["solidLayers"] + 3 + 2)
        h2d = int(h2d * min(1.0, (sc.nz + world * halo) / sc.nz))
    elif world > 1:
        h2d *= world
    e2e = {"value": a.steps / e2e_elapsed, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "ms_per_step": e2e_elapsed / a.steps * 1e3,
           "stage_ms": {k: round(v, 3) for k, v in solver.stage_ms().items()},
           "overlap": "SDFs first; viscosity / velocity / collision velocity H2D under weights + classification; valid D2H under the CG loop; velocity D2H pipelined per axis"}

    # ---- roofline of the dominant kernel (pass 2 = SpMV over K_ext^T, the longest kernel of a CG iteration),
    #      timed live with CUDA events on the solver's stream
    peak, peak_src = measured_peak()
    solver.setup(d_in[0], d_in[1], d_in[2], d_vel, d_cvel)
    kern = {}
    for k in ("pass1", "pass1_sweep", "pass2", "pass2_dots", "apply", "cg_update", "cg_iteration"):
        ms = solver.time_kernel(k, a.kernel_reps)
        by = solver.kernel_bytes(k) / world          # per-GPU share of the algorithmic bytes (rows are split ~evenly over the slabs)
        kern[k] = {"ms": ms, "algorithmic_bytes": by, "gbs": by / ms / 1e6, "frac": by / ms / 1e6 / peak}
    # the dominant kernel = the longest of the three kernels of a CG iteration, as timed above
    names = {"pass1": "pass1_kernel + reduced_region_kernel (w = K_ext p with dt Mc^-1, then the region term: moments -> B^-1 -> expand, one CTA per region)",
             "pass2_dots": "pass2_kernel (Ap = -K_ext^T w - 1/2 mu^-1 p, fused p.Ap, r.Ap, Ap.Ap)",
             "cg_update": "cg_update_kernel (x += a p, r -= a Ap, p = r + b p, fused r.r, x.p, p.p)"}
    dom = max(names, key=lambda k: kern[k]["ms"])
    # DRAM traffic of that kernel from the committed `ncu --set full` capture of this build (profiles/ncu_traffic.json, single GPU, full grid): only
    # meaningful next to the N = 1 launch; at N > 1 the per-rank kernel was not captured -> null
    traffic = None
    if world == 1 and a.n == SCENE_N:
        try:
            with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
                tj = json.load(f)
            key = names[dom].split(" ")[0]
            traffic = next((v for k, v in tj.items() if key in k), None)
        except Exception:
            traffic = None
    working_set = kern[dom]["algorithmic_bytes"]
    roofline = {"kernel": names[dom], "bound": "hbm", "achieved": kern[dom]["gbs"], "peak": peak, "unit": "GB/s", "frac": kern[dom]["frac"], "traffic": traffic,
                "peak_source": peak_src, "l2_resident": bool(working_set < 126e6),
                "note": ("per-rank working set below the 126 MB L2: frac is not HBM evidence" if working_set < 126e6 else
                         "achieved = algorithmic bytes of one launch (DESIGN.md section 5, ps_kernel_bytes) / CUDA-event time on the solver's stream"),
                "spmv": {"pass1_frac": kern["pass1"]["frac"], "pass2_frac": kern["pass2_dots"]["frac"]}, "kernels": kern}

    # ---- the same step at the grids the CPU arms ran (N = 1): same-configuration ratios without any scaling
    def gpu_step_rates(n, steps=3):
        sc2 = scenes.scene_s3(n)
        s2 = PolyStokesSolver.from_scene(sc2, device=local)
        hin = [pin(sc2.surface), pin(sc2.collision), pin(sc2.viscosity)]; hv = [pin(v) for v in sc2.vel]; hc = [pin(v) for v in sc2.colvel]
        ho = [torch.empty_like(v).pin_memory() for v in hv]; hval = [torch.empty_like(v).pin_memory() for v in hv]
        def one():
            rc = s2.step(hin[0].numpy(), hin[1].numpy(), hin[2].numpy(), npv(hv), npv(hc), npv(ho), npv(hval))
            if rc != PS_SUCCESS:
                raise SystemExit(f"bench.py: solver returned {rc} at {n}^3")
        one(); one()
        torch.cuda.synchronize(); t0 = time.perf_counter()
        for _ in range(steps):
            one()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / steps
        its = s2.count("iterations"); nsys = s2.count("nSystemSize")
        s2.close()
        return {"grid": n, "e2e_steps_per_s": 1.0 / dt, "e2e_ms_per_step": dt * 1e3, "cg_iterations": its, "nSystemSize": nsys}

    # ---- CPU baseline: the reference's own solver on the box's host cores, BOUNDED sample (rank 0, N = 1 only): one measured step at 96^3
    cpu = None
    same_grid = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        ncal = 96 if a.n >= 96 else a.n
        if reference_available():
            q = run_ref_full(ncal)
            g96 = gpu_step_rates(ncal)
            cpu = {"value": 1.0 / q["seconds"], "unit": UNIT, "cores": q["cores"], "kind": "reference", "grid": [ncal] * 3,
                   "sample": (f"the reference's own solver (oracle/_ref/libps_ref_full.so: exec/HDK_PolyStokesSolver*.cpp + lib/ compiled unmodified on the HDK stand-in / Eigen "
                              f"facade, {q['jobs']} setup jobs + OpenMP) ran ONE full step of the same scene S3 at {ncal}^3 (bounded sample; value = measured steps/s AT THAT GRID, "
                              f"not scaled): {q['seconds']:.2f} s (setup {q['setup_s']:.2f} s, {q['iterations']} CG its in {q['cg_s']:.2f} s, n={q['nSystemSize']})"),
                   "gpu_same_grid": g96, "same_grid_ratio_e2e": g96["e2e_steps_per_s"] * q["seconds"]}
        else:
            q = run_cpu_sample(ncal)
            cpu = {"value": 1.0 / q["seconds"], "unit": UNIT, "cores": q["cores"], "kind": "port", "grid": [ncal] * 3,
                   "sample": f"oracle (OpenMP restatement, all host cores) ran ONE full step of S3 at {ncal}^3 (bounded sample, not scaled): {q['seconds']:.2f} s ({q['iterations']} CG its)"}
        # the full-size run of the reference arm on this box, if it ran before us (bench.py --impl reference writes it)
        try:
            full = ref_cache_load()
            if full is None:
                raise KeyError("no reference run on this machine")
            gfull = {"grid": a.n, "e2e_steps_per_s": e2e["value"], "e2e_ms_per_step": e2e["ms_per_step"]} if full["n"] == a.n else gpu_step_rates(full["n"])
            same_grid = {"grid": [full["n"]] * 3, "reference_seconds_per_step": full["seconds"], "reference_cores": full["cores"], "reference_kind": full["kind"],
                         "ours_e2e_steps_per_s": gfull["e2e_steps_per_s"], "same_config_ratio": gfull["e2e_steps_per_s"] * full["seconds"],
                         "source": "this box's `bench.py --impl reference` run (measured, unscaled)"}
        except Exception:
            same_grid = None

    if rank == 0:
        out = {"metric": metric, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
               "ms_per_step": elapsed / a.steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
               "data": "synthetic", "config": dict(config, parallelism="single GPU" if world == 1 else
                                                   f"z-slab decomposition over {world} GPUs, cuts {part[4]} (one process per GPU; per CG iteration: halo exchange of p and w + "
                                                   "2 scalar all-reduces, " + ("over NVLink peer memory: boundary entries stored straight into the neighbours' vectors, reductions fused into the kernels"
                                                                             if solver.count("peerTransport") else "NCCL") +
                                                   ("; slab-local setup and I/O: every rank classifies / assembles / uploads its slab + halo layers" if solver.count("slabLocal")
                                                    else "; classification replicated") + ")",
                                                   counts=counts, timing="CUDA events on the solver's stream around the K timed steps (max over ranks), bracketed by "
                                                   "barrier + synchronize; wall_ms_per_step = host clock over the same region; "
                                                   "device_ms_per_step = sum of per-stage CUDA-event times"),
               "wall_ms_per_step": wall / a.steps * 1e3, "device_ms_per_step": dev_ms / a.steps, "stage_ms": {k: round(v, 3) for k, v in stage_ms.items()},
               "cg_iterations": counts["iterations"], "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
               "roofline": roofline, "cpu_baseline": cpu, "vs_reference_same_grid": same_grid, "parity_checked": parity_checked, "parity": parity_note}
        emit(out)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

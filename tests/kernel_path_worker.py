"""Child process of tests/test_gpu_kernel_paths.py: runs the library on a few scenes under ONE setting of the region-kernel
knobs (PS_REGION_FUSE_MAX, PS_GRAM_DMMA).  The library reads each knob once per process, so every setting needs a process of its
own; the knob comes in through the environment.

usage: python kernel_path_worker.py [--lib PATH] [--tight] [--no-step] <out_dir> <scene>...

For each scene it writes <out_dir>/<scene>.npz with
  - the counts, among them the ones that say which kernels ran (regionPath, maxRegionRows, maxRegionAxisRows, ...);
  - after setup only: MrDense, ViscDense, BinvDense, bestFit, com, b;
  - apply(x1), apply(x2), apply(x1) again (x1, x2 from `vectors`);
  - after a step: result, iterations, solution, xmag, the velocities and valid fields, and apply(x1) once more -- the CG loop
    has run through the same per-region tickets and device scalars in between;
  - MrDense, ViscDense, BinvDense and bestFit of a second handle set up on the same scene;
  - with --tight, for the scenes in TIGHT: the velocities of the same step solved to tolerance / 1000 on a fresh handle.
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from polystokes_b200 import PolyStokesSolver, scenes  # noqa: E402

SCENES = {
    "blob40": lambda: scenes.blob_scene(40),                                        # 22 regions of tile 8
    "blob32_seed5": lambda: scenes.blob_scene(32, seed=5),                          # a region of 21 cells: less than a warp of Gram work
    "blob64_tile32": lambda: scenes.blob_scene(64, seed=3, tile=32, pad=2),         # > 1024 rows on one (region, axis)
    "blob64_notile": lambda: scenes.blob_scene(64, seed=3, doTile=0),               # one region of 16514 rows: the chunked kernels
    "box96_tile8": lambda: scenes.box_scene(96, liquid_hi_frac=0.95, shell=2, tileSize=8, tilePadding=1),   # 1000 regions
}
# scenes too large for a CPU reference solve: their velocity is compared with a run solved to tolerance / 1000
TIGHT = {"box96_tile8"}

COUNTS = ["regionCount", "nSystemSize", "nActiveVs", "nRowsExt", "maxRegionRows", "maxRegionAxisRows", "maxRegionCells",
          "minRegionCells", "regionPath"]


def vectors(n):
    """The two operands of the applies, drawn from a fixed seed (the parent draws the same)."""
    rng = np.random.default_rng(20261020)
    return rng.standard_normal(n), rng.standard_normal(n)


def run_scene(name, lib, out_dir, tight, step):
    sc = SCENES[name]()
    s = PolyStokesSolver.from_scene(sc, lib_path=lib)
    s.setup_scene(sc)
    out = {"count_" + k: s.count(k) for k in COUNTS}
    for v in ("MrDense", "ViscDense", "BinvDense", "bestFit", "com", "b"):
        out[v] = s.vector(v)
    x1, x2 = vectors(s.count("nSystemSize"))
    out["y1_first"] = s.apply(x1)
    out["y2"] = s.apply(x2)
    out["y1_second"] = s.apply(x1)
    if step:
        rc, vel, valid = s.step_scene(sc)
        out.update(rc=rc, iterations=s.count("iterations"), usedBiCGStab=s.count("usedBiCGStab"), solution=s.vector("solution"),
                   xmag=s.real("xmag"), solveError=s.real("solveError"))
        for a in range(3):
            out[f"vel{a}"], out[f"valid{a}"] = vel[a], valid[a]
        out["y1_after_step"] = s.apply(x1)
    s.close()
    second = PolyStokesSolver.from_scene(sc, lib_path=lib)      # the region blocks of a second handle: bit-identical
    second.setup_scene(sc)
    for v in ("MrDense", "ViscDense", "BinvDense", "bestFit"):
        out[v + "_second_handle"] = second.vector(v)
    second.close()
    if step and tight and name in TIGHT:
        t = PolyStokesSolver.from_scene(sc, lib_path=lib, tolerance=sc.params["tolerance"] * 1e-3)
        rc2, vel2, valid2 = t.step_scene(sc)
        out["tight_rc"] = rc2
        for a in range(3):
            out[f"tight_vel{a}"], out[f"tight_valid{a}"] = vel2[a], valid2[a]
        t.close()
    np.savez(os.path.join(out_dir, name + ".npz"), **out)
    print(f"{name}: regionPath {out['count_regionPath']}, {out['count_regionCount']} regions, n {out['count_nSystemSize']}"
          + (f", {out['iterations']} iterations" if step else ""), flush=True)


def main(argv):
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", default=None, help="library to load (default: the CUDA library; the host-emulation twin for CPU runs)")
    ap.add_argument("--tight", action="store_true", help="also solve the TIGHT scenes to tolerance / 1000")
    ap.add_argument("--no-step", dest="step", action="store_false", help="setup and applies only")
    ap.add_argument("out_dir")
    ap.add_argument("scenes", nargs="+", choices=list(SCENES))
    a = ap.parse_args(argv)
    os.makedirs(a.out_dir, exist_ok=True)
    for name in a.scenes:
        run_scene(name, a.lib, a.out_dir, a.tight, a.step)


if __name__ == "__main__":
    main(sys.argv[1:])

"""Scenes whose reduced regions cross the z cuts of a slab decomposition (doTile off, or tiles without padding), for the
distributed tests of tests/test_distributed_spanning_emul.py (host-emulation twin) and tests/test_gpu_spanning_regions.py.

register() adds them to parity.DIST_CASES so that parity.check_distributed compares them with the oracle like every other
distributed case.  All grids have nz = 64 (or 128): up to four 16-layer slabs (eight for s3_128).
"""
import parity
from polystokes_b200 import scenes

SHAPE = (40, 36, 64)

CASES = {
    # one connected region for the whole untiled blob: it crosses every cut (the octopus configuration)
    "span_blob64_notile": lambda: (scenes.blob_scene(SHAPE, seed=21, doTile=0), {}),
    # tiles without padding: regions touching a tile face; the ones at a cut are shared, the others stay local
    "span_blob64_tile8_pad0": lambda: (scenes.blob_scene(SHAPE, seed=8, tile=8, pad=0, tolerance=1e-6), {}),
    # 16^3 tiles are cut-aligned: a region never has cells on both sides of a cut, it reaches the upper slab only through its
    # z-faces on the cut plane
    "span_blob64_tile16_pad0": lambda: (scenes.blob_scene(SHAPE, seed=13, tile=16, pad=0), {}),
    # CG runs out of iterations -> BiCGSTAB fallback, stopped after 6 iterations (results kept)
    "span_blob64_notile_bicgstab6": lambda: (scenes.blob_scene(SHAPE, seed=21, doTile=0, maxIterations=6, tolerance=1e-12, keepNonConvergedResults=1), {}),
    # the same handle first steps the scene with 24^3 padded tiles (cuts at multiples of lcm(16, 24) = 48), then is switched to
    # doTile 0 (cuts at multiples of 16) with ps_set_params (SWITCH): on 2 ranks the cut moves from z = 48 to z = 32
    "span_blob64_switch_tile_notile": lambda: (scenes.blob_scene(SHAPE, seed=21, doTile=0), {}),
    # padded tiles: no region can reach a cut, nothing is shared
    "span_blob64_tile8_pad1": lambda: (scenes.blob_scene(SHAPE, seed=8, tile=8, pad=1), {}),
    "span_s3_128_notile": lambda: (scenes.scene_s3(128, doTile=0), {}),
}

# cases stepped first with other tiling parameters on the same handle (tests/spanning_worker.py)
SWITCH = {"span_blob64_switch_tile_notile": dict(doTile=1, tileSize=24, tilePadding=1)}

NO_SHARED = {"span_blob64_tile8_pad1"}

# Velocity gates where 10 x tol is not meaningful (as parity.DIST_VEL_GATE): many small unpadded 8^3 tiles make the system ill
# conditioned -- on ONE rank the emulation twin and the oracle, two correct CG runs that sum in different orders, already stop at
# iterates whose velocities differ by 1.3e-4 at tol 1e-6 (1.6e-2 at tol 1e-4).  A wrong shared-region sum shows up as O(1).
VEL_GATE = {"span_blob64_tile8_pad0": 1e-3}


def register():
    parity.DIST_CASES.update(CASES)
    parity.DIST_VEL_GATE.update(VEL_GATE)

"""Scenes whose reduced regions cross the z cuts of a slab decomposition (doTile off, or tiles without padding), for the
distributed tests of tests/test_distributed_spanning_emul.py (host-emulation twin) and tests/test_gpu_spanning_regions.py.

register() adds them to parity.DIST_CASES so that parity.check_distributed compares them with the oracle like every other
distributed case.  All grids have nz = 64 (or 128, or 32 for the pillar lattices): up to four 16-layer slabs (eight for s3_128).
"""
import numpy as np

import parity
from polystokes_b200 import scenes
from polystokes_b200.scenes import DEFAULT_PARAMS, _centres, _finish, sd_box

SHAPE = (40, 36, 64)


def bodies_scene(boxes, shape=SHAPE, seed=99, **overrides):
    """Separate liquid boxes in air (one untiled region each), inside a solid container.  `boxes`: (lo, hi) corners in cells; the
    reduced cells of a box are its liquid cells less one layer on every side ([lo + 1, hi - 1) along z)."""
    nx, ny, nz = shape
    dx = 1.0 / 64
    x, y, z = _centres(nx, ny, nz, dx)
    col = -sd_box(x, y, z, [2.3 * dx] * 3, [(nx - 2.3) * dx, (ny - 2.3) * dx, (nz - 2.3) * dx])
    surf = np.minimum.reduce([sd_box(x, y, z, [c * dx for c in lo], [c * dx for c in hi]) for lo, hi in boxes])
    p = dict(DEFAULT_PARAMS, doTile=0, tolerance=1e-6)
    p.update(overrides)
    return _finish("bodies", shape, dx, 1 / 60, 800.0, surf, col, np.float32(60.0), seed, p)


# Six bodies; at 4 ranks (cuts at z = 16, 32, 48), in region order (first reduced cell, z-slowest):
#   0  z 4..59   crosses every cut: owned by rank 0, rows on every rank
#   1  z 4..11   unshared, rank 0
#   2  z 19..28  unshared, rank 1 -- numbered between shared region 0 (rank 0) and rank 2's own region 4: rank 2 builds it without
#                owning it or holding any of its rows
#   3  z 21..53  crosses z = 32 and 48 but not 16: owned by rank 1
#   4  z 35..47  all cells below z = 48, its top reduced z-faces ON the plane z = 48: shared only through them (rank 2 owns it, rank 3
#                holds those rows)
#   5  z 53..59  unshared, rank 3
# Rank 1 thus owns an unshared region (2), owns a shared one (3) and holds rows of a shared region of rank 0 (0).  At 2 ranks (cut at
# 32) regions 0 and 3 are shared, at 3 ranks more.  The unshared regions stay far below the 16384 coupled rows where the GPU leaves the
# one-CTA region kernel, so the unshared and the shared regions of one rank take different kernels.
BODIES = [((3, 3, 3), (12, 33, 61)),
          ((16, 3, 3), (37, 33, 13)),
          ((16, 3, 18), (26, 16, 30)),
          ((30, 3, 20), (37, 33, 55)),
          ((16, 20, 34), (26, 33, 49)),
          ((16, 3, 52), (26, 16, 61))]


def pillar_lattice(px, py, short_every=24, pitch=8, width=6, nz=32):
    """px x py separate square pillars (width x width cells, 2 cells of air between them) on a 32-layer grid: one untiled region each.
    Pillar k = iy * px + ix has reduced cells z 13..18, across the cut z = 16 of 2 ranks; every `short_every`-th one sits at z 18..23,
    inside the upper slab (unshared)."""
    nx, ny = pitch * px + 6, pitch * py + 6
    dx = 1.0 / 64
    x, y, z = _centres(nx, ny, nz, dx)
    col = -sd_box(x, y, z, [2.3 * dx] * 3, [(nx - 2.3) * dx, (ny - 2.3) * dx, (nz - 2.3) * dx])

    def local(c, n):      # cell coordinate relative to the nearest pillar's low side, in [-1, pitch - 1); and that pillar's index
        i = np.clip(np.floor((c / dx - 2.0) / pitch), 0, n - 1)
        return c / dx - 3.0 - pitch * i, i
    u, ix = local(x, px)
    v, iy = local(y, py)
    short = ((iy * px + ix) % short_every) == 0
    zlo, zhi = np.where(short, 17.0, 12.0), np.where(short, 25.0, 20.0)
    q = [np.abs(u - width / 2) - width / 2, np.abs(v - width / 2) - width / 2, np.abs(z / dx - (zlo + zhi) / 2) - (zhi - zlo) / 2]
    outside = np.sqrt(sum(np.maximum(a, 0) ** 2 for a in q))
    surf = (outside + np.minimum(np.maximum(q[0], np.maximum(q[1], q[2])), 0)) * dx
    p = dict(DEFAULT_PARAMS, doTile=0, tolerance=1e-6)
    return _finish(f"pillars{px}x{py}", (nx, ny, nz), dx, 1 / 60, 800.0, surf, col, np.float32(60.0), 7, p)


CASES = {
    # one connected region for the whole untiled blob: it crosses every cut (the octopus configuration)
    "span_blob64_notile": lambda: (scenes.blob_scene(SHAPE, seed=21, doTile=0), {}),
    # tiles without padding touch each other, so the blob is ONE region here too (one shared region); 8^3 tiles
    "span_blob64_tile8_pad0": lambda: (scenes.blob_scene(SHAPE, seed=8, tile=8, pad=0, tolerance=1e-6), {}),
    # the same with 16^3 tiles, which are cut-aligned: one region, shared
    "span_blob64_tile16_pad0": lambda: (scenes.blob_scene(SHAPE, seed=13, tile=16, pad=0), {}),
    # CG runs out of iterations -> BiCGSTAB fallback, stopped after 6 iterations (results kept)
    "span_blob64_notile_bicgstab6": lambda: (scenes.blob_scene(SHAPE, seed=21, doTile=0, maxIterations=6, tolerance=1e-12, keepNonConvergedResults=1), {}),
    # the same handle first steps the scene with 24^3 padded tiles (cuts at multiples of lcm(16, 24) = 48), then is switched to
    # doTile 0 (cuts at multiples of 16) with ps_set_params (SWITCH): on 2 ranks the cut moves from z = 48 to z = 32
    "span_blob64_switch_tile_notile": lambda: (scenes.blob_scene(SHAPE, seed=21, doTile=0), {}),
    # padded tiles: no region can reach a cut, nothing is shared
    "span_blob64_tile8_pad1": lambda: (scenes.blob_scene(SHAPE, seed=8, tile=8, pad=1), {}),
    "span_s3_128_notile": lambda: (scenes.scene_s3(128, doTile=0), {}),
    # many regions, shared and unshared, on the same ranks (BODIES)
    "span_bodies_notile": lambda: (bodies_scene(BODIES), {}),
    # more shared regions at 2 ranks than the peer moment area holds (4174 of 4356 pillars; the communicator sums them), and just
    # fewer (4048 of 4224; peer memory).  GPU only: 9 M cells
    "span_pillars_over_cap": lambda: (pillar_lattice(66, 66), {}),
    "span_pillars_under_cap": lambda: (pillar_lattice(64, 66), {}),
}

# cases stepped first with other tiling parameters on the same handle (tests/spanning_worker.py)
SWITCH = {"span_blob64_switch_tile_notile": dict(doTile=1, tileSize=24, tilePadding=1)}

NO_SHARED = {"span_blob64_tile8_pad1"}

# Least regionCount / sharedRegions per world size, so that a case cannot collapse to fewer regions unnoticed (check() also compares
# the shared count with the one derived from the oracle's classification).  pad1 gives many regions and no shared one.
MIN_COUNTS = {
    "span_blob64_notile": {w: (1, 1) for w in (2, 3, 4)},
    "span_blob64_tile8_pad0": {w: (1, 1) for w in (2, 3, 4)},
    "span_blob64_tile16_pad0": {w: (1, 1) for w in (2, 3, 4)},
    "span_blob64_notile_bicgstab6": {w: (1, 1) for w in (2, 3, 4)},
    "span_blob64_switch_tile_notile": {2: (1, 1)},
    "span_blob64_tile8_pad1": {w: (10, 0) for w in (2, 3, 4)},
    "span_s3_128_notile": {8: (1, 1)},
    "span_bodies_notile": {2: (6, 2), 3: (6, 3), 4: (6, 3)},
    "span_pillars_over_cap": {2: (4356, 4097)},
    "span_pillars_under_cap": {2: (4224, 4000)},
}

# Velocity gates where 10 x tol is not meaningful (as parity.DIST_VEL_GATE): many small unpadded 8^3 tiles make the system ill
# conditioned -- on ONE rank the emulation twin and the oracle, two correct CG runs that sum in different orders, already stop at
# iterates whose velocities differ by 1.3e-4 at tol 1e-6 (1.6e-2 at tol 1e-4).  A wrong shared-region sum can be far smaller than
# O(1) (a few rows of one region); the componentwise operator gate of parity.check_distributed is what catches it.
VEL_GATE = {"span_blob64_tile8_pad0": 1e-3}


def register():
    parity.DIST_CASES.update(CASES)
    parity.DIST_VEL_GATE.update(VEL_GATE)


def shared_regions(o, cuts):
    """The shared regions by the library's rule for regions that may cross a cut (doTile 0 or tilePadding 0), derived from the oracle's
    classification: the owner of a region is the slab of its
    first reduced cell in voxel order; a region is shared when its reduced faces lie in more than one slab, or in one slab that is not
    its owner's (a z-face on a cut plane belongs to the upper slab).  Returns {region: (owner, sorted slabs of its faces)}."""
    cuts = np.asarray(cuts)
    slab = lambda zs: np.searchsorted(cuts, zs, side="right") - 1
    cells = o.index_field(2, 0)
    R = o.count("regionCount")
    flat = cells.reshape(-1)
    first = np.full(R, flat.size, dtype=np.int64)
    idx = np.nonzero(flat >= 0)[0]
    np.minimum.at(first, flat[idx], idx)
    owner = slab(first // (cells.shape[1] * cells.shape[2]))
    faces = [set() for _ in range(R)]
    for a in range(3):
        f = o.index_field(2, 1 + a)
        z, _, _ = np.nonzero(f >= 0)
        pairs = np.unique(np.stack([f[f >= 0], slab(z)]), axis=1)
        for r, k in pairs.T:
            faces[int(r)].add(int(k))
    return {r: (int(owner[r]), sorted(faces[r])) for r in range(R) if len(faces[r]) > 1 or (faces[r] and int(owner[r]) not in faces[r])}

"""Scenes at the edges of the input domain, for tests/test_input_edges.py and the slab-decomposed border cases of parity.DIST_CASES.

Every builder of polystokes_b200.scenes ends in scenes._finish, which keeps a non-liquid cell on every domain face.  The builders here do
not: liquid reaches the planes x = 0 / x = nx (and likewise for y and z), where the SDF reads clamp to the edge, labels and indices
outside the grid read as UNASSIGNED, and the last z-slab of a decomposed step owns the top layer of the z-face and edge slots.  The
second family keeps ordinary geometry and puts unusual VALUES into the SDFs (NaN, infinities, -0.0, exact zeros, +-FLT_MAX, float
denormals) or into the viscosity (0, six decades).  All of them are seeded.
"""
import numpy as np

from polystokes_b200 import scenes
from polystokes_b200.scenes import DEFAULT_PARAMS, Scene, _centres, _velocities, sd_cylinder_y, sd_sphere


def _scene(name, n, surf, col, visc, seed, params, colvel=None):
    """A Scene straight from the fields: no padding at the border."""
    nx, ny, nz = n
    dx = 1.0 / max(n)
    dt = 1.0 / 60.0
    vel, cv = _velocities(nx, ny, nz, dt, seed)
    if colvel is not None:
        for a in range(3):
            cv[a][...] = np.float32(colvel[a])
    full = lambda a: np.ascontiguousarray(np.broadcast_to(a, (nz, ny, nx)), dtype=np.float32)
    return Scene(name, nx, ny, nz, dx, dt, 800.0, full(surf), full(col), full(visc), vel, cv, params)


def _params(**overrides):
    p = dict(DEFAULT_PARAMS, tolerance=1e-4)
    p.update(overrides)
    return p


def _shape(n):
    return (n, n, n) if isinstance(n, int) else tuple(n)


def tank(n, level=0.55, seed=1, **overrides):
    """Liquid below the plane y = level * ny (off the cell centres), no collision object (collision +1 everywhere): the liquid fills
    the box to the walls x = 0 / nx, z = 0 / nz and the floor y = 0."""
    nx, ny, nz = n = _shape(n)
    dx = 1.0 / max(n)
    x, y, z = _centres(nx, ny, nz, dx)
    surf = y - (level * ny + 0.137) * dx
    return _scene(f"tank{nx}x{ny}x{nz}", n, surf, np.float32(1.0), np.float32(60.0), seed, _params(**overrides))


def border_blob(n, seed=5, **overrides):
    """Spheres cut by the planes x = 0 (that one also by z = 0), y = 0 and z = nz, joined by a sphere in the middle, and a solid
    pillar standing on the floor plane y = 0 (it also cuts the liquid).  No container: the domain walls bound the liquid where it
    reaches them."""
    nx, ny, nz = n = _shape(n)
    dx = 1.0 / max(n)
    x, y, z = _centres(nx, ny, nz, dx)
    L = [nx * dx, ny * dx, nz * dx]
    rng = np.random.Generator(np.random.PCG64(seed))
    u = lambda lo, hi: rng.uniform(lo, hi)
    m = min(L)
    spheres = [([u(-0.05, 0.05) * L[0], u(0.3, 0.5) * L[1], u(0.1, 0.2) * L[2]], u(0.28, 0.34) * m),      # cut by x = 0 and z = 0
               ([u(0.4, 0.6) * L[0], u(-0.05, 0.05) * L[1], u(0.35, 0.6) * L[2]], u(0.28, 0.34) * m),     # cut by y = 0
               ([u(0.4, 0.6) * L[0], u(0.3, 0.5) * L[1], u(0.95, 1.05) * L[2]], u(0.28, 0.34) * m),       # cut by z = nz
               ([0.4 * L[0], 0.35 * L[1], 0.55 * L[2]], 0.27 * m)]
    surf = np.minimum.reduce([sd_sphere(x, y, z, c, r) for c, r in spheres])
    col = sd_cylinder_y(x, y, z, 0.62 * L[0], 0.3 * L[2], 0.09 * L[0], -2.0 * dx, 0.55 * L[1])
    visc = 50.0 * np.exp(0.5 * np.sin(7.0 * x + 3.0 * y) * np.cos(5.0 * z))
    return _scene(f"border_blob{nx}x{ny}x{nz}_s{seed}", n, surf, col, visc, seed + 100, _params(**overrides), colvel=(0.02, -0.01, 0.015))


def full(n, **overrides):
    """Liquid in every cell, no solid."""
    nx, ny, nz = n = _shape(n)
    return _scene(f"full{nx}x{ny}x{nz}", n, np.float32(-1.0), np.float32(1.0), np.float32(60.0), 3, _params(**overrides))


# Border and shape cases: name -> () -> (scene, parameter overrides)
BORDER = {
    "tank24_uniform": lambda: (tank(24, doReduced=0, tolerance=1e-6), {}),
    "tank24_tile8_pad1": lambda: (tank(24, tileSize=8, tilePadding=1), {}),
    "tank_20x28x36_tile16_pad2": lambda: (tank((20, 28, 36), tileSize=16, tilePadding=2), {}),
    "border_blob24_tile8_pad1": lambda: (border_blob(24, tileSize=8, tilePadding=1), {}),
    "border_blob24_notile": lambda: (border_blob(24, seed=6, doTile=0), {}),
    "full20_tile8_pad1": lambda: (full(20, tileSize=8, tilePadding=1), {}),
    "tank_1x20x20": lambda: (tank((1, 20, 20), tileSize=8, tilePadding=1), {}),
    "tank_2x20x17": lambda: (tank((2, 20, 17), tileSize=8, tilePadding=1), {}),
    "tank_20x3x18": lambda: (tank((20, 3, 18), tileSize=8, tilePadding=1), {}),
    "border_blob_15x16x17": lambda: (border_blob((15, 16, 17), seed=7, tileSize=8, tilePadding=1), {}),
}
# tile sizes that do not divide the grid or the 16-layer cut unit, each with several paddings (0: tiles touch)
for _t, _pads in ((4, (0, 1, 2)), (5, (0, 2, 4)), (12, (1, 3, 4))):
    for _p in _pads:
        BORDER[f"border_blob24_tile{_t}_pad{_p}"] = (lambda t, p: lambda: (border_blob(24, seed=9, tileSize=t, tilePadding=p), {}))(_t, _p)


# ---- SDF values ------------------------------------------------------------------------------------------------------------------
# Each value goes into one field of a scene with ordinary geometry, in three places (index order [z, y, x]):
#   "neg"   a block inside the region where the field is negative (liquid for `surface`, the solid wall for `collision`),
#   "pos"   a 4^3 block inside the region where it is non-negative (air / fluid), so that cells deep in the block see only the value,
#   "iface" a patch across the interface, so that the interpolation mixes it with both signs.
# The weight kernel decides a sample from the signs of its 3x3x3 cell block where they agree and interpolates only where they differ:
# the deep cells reach the first way, the block rims and the interface patch the second (test_input_edges checks that they do).
# `surface` cases run on box_scene(24, doReduced=0): liquid y < 14 inside a 4-cell solid shell, air 14 <= y < 20.  `collision` cases
# run on blob_scene(24, seed=3): a 2-cell solid wall (collision < 0 for cells 0 and 1 of every axis) and a pillar.
SDF_BASE = {
    "surface": (lambda: scenes.box_scene(24, doReduced=0),
                dict(neg=np.s_[7:11, 6:10, 7:11], pos=np.s_[10:14, 15:19, 10:14], iface=np.s_[14:17, 13:15, 14:17], plane=np.s_[:, 14, :])),
    "collision": (lambda: scenes.blob_scene(24, seed=3),
                  dict(neg=np.s_[0:2, 8:12, 8:12], pos=np.s_[6:10, 14:18, 14:18], iface=np.s_[1:4, 8:12, 14:18], plane=np.s_[12, :, :])),
}

FLT_MAX = float(np.finfo(np.float32).max)
DENORM_MIN = float(np.float32(1e-45))        # the smallest positive float denormal
DENORM = 3e-39


def _checker(a, v):
    """+v / -v alternating cell by cell: every interpolation across it sums +inf and -inf (NaN) when v is inf."""
    k, j, i = np.indices(a.shape)
    return np.where((i + j + k) % 2 == 0, v, -v).astype(np.float32)


def _signed(a, mag):
    """the value of magnitude `mag` with the sign of a (a >= 0: +mag)"""
    return np.where(a < 0, -mag, mag).astype(np.float32)


# value case -> what it writes: {region: value or function of the region's current values}
SDF_VALUES = {
    "nan_only": dict(pos=np.nan, neg=np.nan),                       # blocks of NaN only
    # a 2^3 NaN hole in an otherwise negative block, and one NaN cell on the negative side of the interface
    "nan_in_negative": dict(neg=lambda a: _hole(a), iface=lambda a: _nan_cell(a, a < 0)),
    "nan_in_positive": dict(pos=lambda a: _hole(a), iface=lambda a: _nan_cell(a, a >= 0)),     # ... positive
    "nan_interface": dict(iface=np.nan),
    "neg_inf": dict(pos=-np.inf, iface=-np.inf),
    "pos_inf": dict(neg=np.inf, iface=np.inf),
    "inf_mix": dict(pos=lambda a: _checker(a, np.inf), iface=lambda a: _checker(a, np.inf), neg=-np.inf),
    "neg_zero": dict(pos=-0.0, iface=lambda a: np.where(a >= 0, np.float32(-0.0), a)),
    "zero_plane": dict(plane=0.0),
    "flt_max": dict(pos=FLT_MAX, neg=-FLT_MAX, iface=lambda a: _signed(a, FLT_MAX)),
    "denormal": dict(pos=DENORM, neg=-DENORM, iface=lambda a: _signed(a, DENORM_MIN)),
}


def _hole(a):
    a = a.copy()
    c = [s // 2 for s in a.shape]
    a[max(c[0] - 1, 0):c[0] + 1, c[1] - 1:c[1] + 1, c[2] - 1:c[2] + 1] = np.nan
    return a


def _nan_cell(a, where):
    a = a.copy()
    cells = np.argwhere(where)
    a[tuple(cells[len(cells) // 2])] = np.nan
    return a


def sdf_case(field, value):
    """(scene, cells written): the base scene of `field` with SDF_VALUES[value] written into that field."""
    build, regions = SDF_BASE[field]
    sc = build()
    a = np.array(sc.surface if field == "surface" else sc.collision)
    written = np.zeros(a.shape, dtype=bool)
    for where, v in SDF_VALUES[value].items():
        s = regions[where]
        a[s] = v(a[s]) if callable(v) else np.float32(v)
        written[s] = True
    if field == "surface":
        sc.surface = np.ascontiguousarray(a)
    else:
        sc.collision = np.ascontiguousarray(a)
    sc.name = f"{sc.name}_{field}_{value}"
    return sc, written


SDF_CASES = {f"{field}_{value}": (lambda f, v: lambda: (sdf_case(f, v)[0], {}))(field, value) for field in SDF_BASE for value in SDF_VALUES}


# ---- viscosity -------------------------------------------------------------------------------------------------------------------
def visc_zero_half():
    """Viscosity 0 in the half x < nx / 2 of a blob (the reference clamps 1 / mu to 1e10 there)."""
    sc = scenes.blob_scene(24, seed=4)
    v = np.array(sc.viscosity)
    v[:, :, :12] = 0.0
    sc.viscosity = np.ascontiguousarray(v)
    return sc


def visc_six_decades():
    """mu = 10^u, u uniform in [-2, 4] per cell: six decades in one blob."""
    sc = scenes.blob_scene(24, seed=4)
    rng = np.random.Generator(np.random.PCG64(77))
    sc.viscosity = np.ascontiguousarray(10.0 ** rng.uniform(-2.0, 4.0, size=sc.viscosity.shape), dtype=np.float32)
    return sc


VISC_CASES = {"visc_zero_half": lambda: (visc_zero_half(), {}), "visc_six_decades": lambda: (visc_six_decades(), {})}

CASES = {**BORDER, **SDF_CASES, **VISC_CASES}


# ---- slab-decomposed border runs (parity.DIST_CASES) -----------------------------------------------------------------------------
# Cut units: 16 layers uniform or untiled, lcm(16, tileSize) tiled.  The 48^3 scenes cover 2 and 3 ranks, the 128-layer tank 4 and 8;
# 12^3 tiles cut at multiples of 48, which is not a multiple of 32.
DIST = {
    "border_tank48_uniform": lambda: (tank(48, doReduced=0, tolerance=1e-6), {}),
    "border_tank48_tile16_pad2": lambda: (tank(48, tileSize=16, tilePadding=2), {}),
    "border_blob48_tile8_pad1": lambda: (border_blob(48, seed=12, tileSize=8, tilePadding=1), {}),
    "border_blob48_notile": lambda: (border_blob(48, seed=12, doTile=0), {}),
    "border_tank_40x40x128_tile16_pad2": lambda: (tank((40, 40, 128), tileSize=16, tilePadding=2), {}),
    "border_tank_32x32x96_tile12_pad1": lambda: (tank((32, 32, 96), tileSize=12, tilePadding=1), {}),
}
SLAB_LOCAL = {"border_tank48_uniform", "border_tank48_tile16_pad2", "border_tank_40x40x128_tile16_pad2"}     # tanks without boundary fix-up work
SHARED = {"border_blob48_notile"}       # doTile 0: the blob is one region across every cut

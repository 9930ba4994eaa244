"""Host-side mirror of the reference's solver entry point, on top of the C ABI.

``PolyStokesSolver`` plays the role of ``HDK_PolyStokes`` + ``HDK_PolyStokes::Solver``
(exec/HDK_PolyStokes.h:15-119, exec/HDK_PolyStokesSolver.h:27-887): same parameter names as the DOP
node (exec/HDK_PolyStokes.h:23-43, defaults exec/HDK_PolyStokes.C:123-206), one ``solve`` call per
substep (``solveGasSubclass``, exec/HDK_PolyStokes.C:222-609) and the same ``SolverResult`` values.
All computation happens in ``libpolystokes_b200.so`` (CUDA); numpy / torch are used for buffers only.
"""
from __future__ import annotations

import ctypes as C
import numpy as np

from . import _capi
from ._capi import (PS_SUCCESS, PS_NOCONVERGE, PS_FAILED, PS_INVALID, PS_UNSUPPORTED_SOLVER, PS_INCOMPLETE,
                    PS_MEM_HOST, PS_MEM_DEVICE, STAGE_NAMES)

SLOTS = ["center", "faceX", "faceY", "faceZ", "edgeYZ", "edgeXZ", "edgeXY"]

# node defaults, exec/HDK_PolyStokes.C:123-206
DEFAULTS = dict(tolerance=1e-3, maxSolverIterations=5000, activeLiquidBoundaryLayerSize=2, activeSolidBoundaryLayerSize=2,
                doReducedRegions=1, doTile=1, tileSize=16, tilePadding=2, exportMatrices=0, exportComponentMatrices=0,
                exportStats=0, exportDataPrefix="", doSolve=1, keepNonConvergedResults=1, useWarmStart=1, matrixSetup=0,
                solverType=0, useInputSurfaceWeights=0, useInputCollisionWeights=0, minDensity=0.0, maxDensity=100000.0,
                device=0, checkEvery=0)

# scene.params uses the oracle's short names; map them onto the node's PRM names
_ALIASES = dict(maxIterations="maxSolverIterations", liquidLayers="activeLiquidBoundaryLayerSize",
                solidLayers="activeSolidBoundaryLayerSize", doReduced="doReducedRegions")


class PolyStokesError(RuntimeError):
    pass


def slot_shape(slot, nx, ny, nz):
    r = [nx, ny, nz]
    if 1 <= slot <= 3:
        r[slot - 1] += 1
    elif slot >= 4:
        for a in range(3):
            if a != slot - 4:
                r[a] += 1
    return (r[2], r[1], r[0])


def _ptr(a):
    """Address of a numpy array or a torch tensor (host or device)."""
    if a is None:
        return None
    if hasattr(a, "data_ptr"):
        return C.c_void_p(a.data_ptr())
    return C.c_void_p(a.ctypes.data)


def _is_device(a):
    return hasattr(a, "is_cuda") and a.is_cuda


class PolyStokesSolver:
    def __init__(self, nx, ny, nz, dx, dt, density, lib_path=None, devices=None, **params):
        """``devices``: a list of CUDA device ordinals -> ONE handle that slab-decomposes the step over those GPUs inside this
        process (ps_create_multi: one host thread per GPU); the step then takes HOST arrays."""
        self.lib = _capi.load(lib_path)
        self.nx, self.ny, self.nz = int(nx), int(ny), int(nz)
        p = dict(DEFAULTS)
        for k, v in params.items():
            k = _ALIASES.get(k, k)
            if k not in p:
                raise TypeError(f"unknown parameter {k!r}")
            p[k] = v
        P = _capi.ps_params()
        P.nx, P.ny, P.nz = self.nx, self.ny, self.nz
        P.dx, P.dt, P.constantDensity = float(dx), float(dt), float(density)
        for k, v in p.items():
            if k == "exportDataPrefix":
                P.exportDataPrefix = str(v).encode()
            else:
                setattr(P, k, v)
        self.params = p
        self._P = P
        self.h = C.c_void_p()
        self.devices = list(devices) if devices is not None else None
        if self.devices is not None:
            arr = (C.c_int * len(self.devices))(*self.devices)
            rc = self.lib.ps_create_multi(C.byref(P), len(self.devices), arr, C.byref(self.h))
        else:
            rc = self.lib.ps_create(C.byref(P), C.byref(self.h))
        if rc != PS_SUCCESS:
            raise PolyStokesError(f"ps_create failed ({rc}): {self.last_error()}")
        self.stats = None

    @classmethod
    def from_scene(cls, scene, lib_path=None, devices=None, **overrides):
        p = dict(scene.params)
        p.update(overrides)
        return cls(scene.nx, scene.ny, scene.nz, scene.dx, scene.dt, scene.density, lib_path=lib_path, devices=devices, **p)

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            self.lib.ps_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- several GPUs: one process per GPU (include/polystokes_b200.h, "several GPUs") ----
    def init_distributed(self, group=None):
        """Collective over a torch.distributed process group: rank 0 creates the NCCL unique id, torch.distributed
        (any backend) carries its 128 bytes to the other ranks, then every rank joins the solver's own NCCL
        communicator.  After this, step / setup / solve / apply are collective calls on the z-slab decomposition."""
        import torch
        import torch.distributed as dist
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        buf = (C.c_uint8 * 128)()
        if rank == 0:
            rc = self.lib.ps_comm_unique_id(buf)
            if rc != PS_SUCCESS:
                raise PolyStokesError(f"ps_comm_unique_id failed ({rc}): {self.last_error()}")
        t = torch.tensor(list(buf), dtype=torch.uint8)
        if dist.get_backend(group) == "nccl":
            t = t.cuda()
        dist.broadcast(t, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
        ident = (C.c_uint8 * 128)(*t.cpu().tolist())
        rc = self.lib.ps_comm_init(self.h, rank, world, ident)
        if rc != PS_SUCCESS:
            raise PolyStokesError(f"ps_comm_init failed ({rc}): {self.last_error()}")
        return self.partition()

    def partition(self):
        """(rank, nranks, zLo, zHi, zCut[nranks+1]) of the slab decomposition (single GPU: one slab)."""
        r, lo, hi = C.c_int32(), C.c_int32(), C.c_int32()
        n = self.lib.ps_get_partition(self.h, C.byref(r), C.byref(lo), C.byref(hi), None)
        cuts = (C.c_int32 * (n + 1))()
        self.lib.ps_get_partition(self.h, C.byref(r), C.byref(lo), C.byref(hi), cuts)
        return r.value, n, lo.value, hi.value, list(cuts)

    def set_partition(self, cuts=None):
        """Collective: z cuts [nranks+1] for the next setup / step (None = the even cuts).  Returns PS_SUCCESS, or PS_INVALID on every
        rank when the cuts break a rule or differ between ranks (the handle keeps its cuts)."""
        arr = None if cuts is None else (C.c_int32 * len(cuts))(*[int(c) for c in cuts])
        rc = self.lib.ps_set_partition(self.h, arr)
        if rc == PS_FAILED:
            raise PolyStokesError(f"ps_set_partition failed: {self.last_error()}")
        return rc

    def rebalance(self):
        """Collective: cuts that balance the CG-iteration bytes of the last setup over the slabs (vector "unitLoad").  Returns
        (rc, cuts): PS_SUCCESS when the cuts moved (effective at the next setup / step), PS_NOCHANGE, or PS_INVALID before a setup."""
        n = self.partition()[1]
        cuts = (C.c_int32 * (n + 1))()
        rc = self.lib.ps_rebalance(self.h, cuts)
        if rc == PS_FAILED:
            raise PolyStokesError(f"ps_rebalance failed: {self.last_error()}")
        return rc, list(cuts)

    def last_error(self):
        e = self.lib.ps_last_error()
        return e.decode() if e else ""

    # ---- the entry point: one substep ----
    def _fields_in(self, surface, collision, viscosity, vel, colvel):
        arrs = [surface, collision, viscosity] + list(vel) + list(colvel)
        dev = [_is_device(a) for a in arrs]
        if any(dev) and not all(dev):
            raise PolyStokesError("inputs must be all host or all device")
        fin = _capi.ps_fields_in()
        fin.memory = PS_MEM_DEVICE if all(dev) else PS_MEM_HOST
        fin.surface, fin.collision, fin.viscosity = _ptr(surface), _ptr(collision), _ptr(viscosity)
        for a in range(3):
            fin.velocity[a] = _ptr(vel[a]).value
            fin.collisionvel[a] = _ptr(colvel[a]).value
        self._keep_in = arrs
        return fin

    def _fields_out(self, vel_out, valid_out):
        fout = _capi.ps_fields_out()
        arrs = [a for a in list(vel_out) + list(valid_out) if a is not None]
        fout.memory = PS_MEM_DEVICE if arrs and all(_is_device(a) for a in arrs) else PS_MEM_HOST
        for a in range(3):
            fout.velocity[a] = _ptr(vel_out[a]).value if vel_out[a] is not None else None
            fout.valid[a] = _ptr(valid_out[a]).value if valid_out[a] is not None else None
        return fout

    def step(self, surface, collision, viscosity, vel, colvel, vel_out=None, valid_out=None):
        """solveGasSubclass body: returns the SolverResult; writes vel_out / valid_out (3 arrays each) if given."""
        fin = self._fields_in(surface, collision, viscosity, vel, colvel)
        st = _capi.ps_stats()
        fout = None
        if vel_out is not None or valid_out is not None:
            fout = self._fields_out(vel_out or [None] * 3, valid_out or [None] * 3)
        rc = self.lib.ps_step(self.h, C.byref(fin), C.byref(fout) if fout is not None else None, C.byref(st))
        self.stats = st
        if rc in (PS_FAILED, PS_INVALID):
            raise PolyStokesError(f"ps_step failed ({rc}): {self.last_error()}")
        return rc

    def step_scene(self, scene, write_back=True):
        """Convenience for numpy scenes: returns (result, velocity[3], valid[3])."""
        vel_out = [np.array(v, dtype=np.float32, copy=True) for v in scene.vel] if write_back else None
        valid_out = [np.zeros_like(v) for v in scene.vel] if write_back else None
        rc = self.step(scene.surface, scene.collision, scene.viscosity, scene.vel, scene.colvel, vel_out, valid_out)
        return rc, vel_out, valid_out

    def setup(self, surface, collision, viscosity, vel, colvel):
        fin = self._fields_in(surface, collision, viscosity, vel, colvel)
        rc = self.lib.ps_setup(self.h, C.byref(fin))
        if rc != PS_SUCCESS:
            raise PolyStokesError(f"ps_setup failed ({rc}): {self.last_error()}")
        return rc

    def setup_scene(self, scene):
        return self.setup(scene.surface, scene.collision, scene.viscosity, scene.vel, scene.colvel)

    def solve(self, vel_out=None, valid_out=None):
        st = _capi.ps_stats()
        fout = None
        if vel_out is not None or valid_out is not None:
            fout = self._fields_out(vel_out or [None] * 3, valid_out or [None] * 3)
        rc = self.lib.ps_solve(self.h, C.byref(fout) if fout is not None else None, C.byref(st))
        self.stats = st
        if rc in (PS_FAILED, PS_INVALID):
            raise PolyStokesError(f"ps_solve failed ({rc}): {self.last_error()}")
        return rc

    def export(self, prefix, what=7):
        rc = self.lib.ps_export(self.h, str(prefix).encode(), int(what))
        if rc != PS_SUCCESS:
            raise PolyStokesError(f"ps_export failed ({rc}): {self.last_error()}")

    # ---- introspection (parity tests) ----
    def count(self, name):
        v = self.lib.ps_get_count(self.h, name.encode())
        if v == -2 ** 63:
            raise KeyError(name)
        return int(v)

    def real(self, name):
        return float(self.lib.ps_get_real(self.h, name.encode()))

    def index_field(self, kind, slot):
        out = np.empty(slot_shape(slot, self.nx, self.ny, self.nz), dtype=np.int32)
        n = self.lib.ps_get_index_field(self.h, kind, slot, out.ctypes.data)
        if n != out.size:
            raise PolyStokesError(f"ps_get_index_field: {self.last_error()}")
        return out

    def weight_field(self, liquid, slot):
        out = np.empty(slot_shape(slot, self.nx, self.ny, self.nz), dtype=np.float32)
        n = self.lib.ps_get_weight_field(self.h, int(liquid), slot, out.ctypes.data)
        if n != out.size:
            raise PolyStokesError(f"ps_get_weight_field: {self.last_error()}")
        return out

    def csr(self, name):
        r, c, n = C.c_int64(), C.c_int64(), C.c_int64()
        rc = self.lib.ps_get_csr(self.h, name.encode(), C.byref(r), C.byref(c), C.byref(n), None, None, None)
        if rc != PS_SUCCESS:
            raise KeyError(f"{name}: {self.last_error()}")
        ptr = np.empty(r.value + 1, dtype=np.int64)
        idx = np.empty(n.value, dtype=np.int32)
        val = np.empty(n.value, dtype=np.float64)
        self.lib.ps_get_csr(self.h, name.encode(), C.byref(r), C.byref(c), C.byref(n), ptr.ctypes.data, idx.ctypes.data, val.ctypes.data)
        return (r.value, c.value), ptr, idx, val

    def vector(self, name):
        n = self.lib.ps_get_vector(self.h, name.encode(), None)
        if n < 0:
            raise KeyError(name)
        out = np.empty(n, dtype=np.float64)
        self.lib.ps_get_vector(self.h, name.encode(), out.ctypes.data)
        return out

    def apply(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.empty_like(x)
        rc = self.lib.ps_apply(self.h, x.ctypes.data, y.ctypes.data)
        if rc != PS_SUCCESS:
            raise PolyStokesError(f"ps_apply failed: {self.last_error()}")
        return y

    def time_kernel(self, name, reps=20):
        """Average ms of `name` in ("pass1", "pass2", "apply", "cg_iteration") over `reps` runs (CUDA events)."""
        t = float(self.lib.ps_time_kernel(self.h, name.encode(), int(reps)))
        if t < 0:
            raise PolyStokesError(f"ps_time_kernel({name}) failed: {self.last_error()}")
        return t

    def timer_start(self):
        """Record the start event of the device stopwatch on the solver's stream (ps_timer)."""
        if float(self.lib.ps_timer(self.h, 0)) < 0:
            raise PolyStokesError(f"ps_timer failed: {self.last_error()}")

    def timer_stop(self):
        """Record the stop event, wait for it, return the device milliseconds since timer_start()."""
        t = float(self.lib.ps_timer(self.h, 1))
        if t < 0:
            raise PolyStokesError(f"ps_timer failed: {self.last_error()}")
        return t

    def kernel_bytes(self, name):
        return float(self.lib.ps_kernel_bytes(self.h, name.encode()))

    def stage_ms(self):
        return {n: self.stats.stage_ms[i] for i, n in enumerate(STAGE_NAMES)} if self.stats is not None else {}

"""Host-side mirror of the reference's controller API over the C ABI.

``ErgodicControl`` keeps the reference's method names and argument meaning
(ergodic_control.hpp:90-134: control, optTraj, addStateMemory, timeStep,
setTarget, configTarget) for a BATCH of B independent instances living on one
GPU.  numpy arrays go through the ``_host`` entry points (copies + sync, the
end-to-end path); torch CUDA tensors go through the ``_dev`` entry points on
torch's current stream (device-resident path).  Every number is computed by
the CUDA kernels in csrc/ -- this file only marshals pointers.

Array convention: Armadillo column-major 3xN == numpy (N, 3); batched buffers
are (B, N, 3) / (B, 3) / (B, K).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Optional, Sequence

import numpy as np

from . import capi
from .capi import MODEL_CART, MODEL_MECANUM, MODEL_OMNI, MODEL_SIMPLE_CART, EbConfig, ErgodicB200Error, check

try:  # torch is plumbing only (device memory, streams); optional for the host path
    import torch
except Exception:  # pragma: no cover
    torch = None


@dataclass
class Gaussian:
    """target.hpp:56-107 -- 2-D Gaussian with diagonal covariance"""

    mu: Sequence[float]
    sigmas: Sequence[float]


@dataclass
class Target:
    """target.hpp:110-161 -- list of Gaussians (addGaussian / deleteGaussian)"""

    gaussians: list = field(default_factory=list)

    def addGaussian(self, g: Gaussian) -> None:
        self.gaussians.append(g)

    def deleteGaussian(self, idx: int) -> None:
        del self.gaussians[idx]


class _Model:
    """operator() / fdx / fdu / wheels2Twist of the reference's model structs, evaluated by model_eval_kernel
    (csrc/model_kernels.cuh) for one state or a batch (rows)."""

    model_id = -1
    state_space = 3
    params = ()

    def _eval(self, x, u, want):
        lib = capi.load()
        nu = lib.eb_model_controls(self.model_id)
        x = _np_f64(x).reshape(-1, 3)
        u = _np_f64(u).reshape(-1, nu)
        n = x.shape[0]
        if u.shape[0] != n:
            raise ValueError("x and u need the same number of rows")
        f, A, B, vb = np.empty((n, 3)), np.empty((n, 3, 3)), np.empty((n, nu, 3)), np.empty((n, 3))
        par = _np_f64(self.params) if len(self.params) else None
        st = lib.eb_model_eval_host(0, self.model_id, par.ctypes.data if par is not None else None, x.ctypes.data,
                                    u.ctypes.data, n, f.ctypes.data if "f" in want else None,
                                    A.ctypes.data if "A" in want else None, B.ctypes.data if "B" in want else None,
                                    vb.ctypes.data if "vb" in want else None)
        if st == capi.EB_ERR_INVALID_ARGUMENT:
            raise ValueError(lib.eb_last_error().decode())  # std::invalid_argument (cart.hpp:167-170)
        check(st)
        # column-major 3 x 3 / 3 x nu blocks -> numpy (row, col)
        return f, np.transpose(A, (0, 2, 1)), np.transpose(B, (0, 2, 1)), vb

    def __call__(self, x, u):
        f = self._eval(x, u, "f")[0]
        return f[0] if np.ndim(x) == 1 else f

    def fdx(self, x, u):
        A = self._eval(x, u, "A")[1]
        return A[0] if np.ndim(x) == 1 else A

    def fdu(self, x):
        nu = capi.load().eb_model_controls(self.model_id)
        xs = _np_f64(x).reshape(-1, 3)
        B = self._eval(xs, np.zeros((xs.shape[0], nu)), "B")[2]
        return B[0] if np.ndim(x) == 1 else B

    def wheels2Twist(self, u):
        nu = capi.load().eb_model_controls(self.model_id)
        us = _np_f64(u).reshape(-1, nu)
        vb = self._eval(np.zeros((us.shape[0], 3)), us, "vb")[3]
        return vb[0] if np.ndim(u) == 1 else vb


class SimpleCart(_Model):
    """models/cart.hpp:152-206"""

    model_id = MODEL_SIMPLE_CART


class Omni(_Model):
    """models/omni.hpp:164-215"""

    model_id = MODEL_OMNI


class Cart(_Model):
    """models/cart.hpp:60-145 -- 2-wheel differential drive, controls = wheel velocities [uL, uR]"""

    model_id = MODEL_CART

    def __init__(self, wheel_radius: float, wheel_base: float):
        self.wheel_radius, self.wheel_base = float(wheel_radius), float(wheel_base)
        self.params = (self.wheel_radius, self.wheel_base)


class Mecanum(_Model):
    """models/omni.hpp:59-157 -- 4 mecanum wheels, controls = wheel velocities [u0..u3]"""

    model_id = MODEL_MECANUM

    def __init__(self, wheel_radius: float, wheel_base_x: float, wheel_base_y: float):
        self.wheel_radius, self.wheel_base_x, self.wheel_base_y = float(wheel_radius), float(wheel_base_x), float(wheel_base_y)
        self.params = (self.wheel_radius, self.wheel_base_x, self.wheel_base_y)


class RungeKutta:
    """integrator.hpp:60-129 -- the forward problem: solve(model, x0, ut, horizon) -> xt (steps, 3), batched when
    x0 has rows.  Every step is computed by rk4_solve_kernel (one thread per instance)."""

    def __init__(self, dt: float):
        self.dt = float(dt)

    def solve(self, model, x0, ut, horizon: float, device: int = 0):
        lib = capi.load()
        nu = lib.eb_model_controls(model.model_id)
        steps = int(abs(horizon / self.dt))
        single = np.ndim(x0) == 1
        x0 = _np_f64(x0).reshape(-1, 3)
        n = x0.shape[0]
        ut = _np_f64(ut)
        per_instance = ut.ndim == 3
        if ut.shape[-2:] != (steps, nu) and ut.shape[-2:] == (nu, steps):
            ut = np.ascontiguousarray(np.swapaxes(ut, -1, -2))  # Armadillo nu x steps -> (steps, nu) rows
        if ut.shape[-2:] != (steps, nu) or (per_instance and ut.shape[0] != n):
            raise ValueError(f"ut must be (steps={steps}, nu={nu}) or (count, steps, nu)")
        xt = np.empty((n, steps, 3))
        par = _np_f64(model.params) if len(model.params) else None
        st = lib.eb_rk4_solve_host(device, model.model_id, par.ctypes.data if par is not None else None, self.dt,
                                   float(horizon), x0.ctypes.data, ut.ctypes.data, int(per_instance), n, xt.ctypes.data)
        if st == capi.EB_ERR_INVALID_ARGUMENT:
            raise ValueError(lib.eb_last_error().decode())
        check(st)
        return xt[0] if single else xt

    def step(self, model, x, u):
        """one RK4 step (integrator.hpp:176-184), heading NOT wrapped (solve wraps)"""
        raise NotImplementedError("use solve(); the unwrapped single step is not exported")


@dataclass
class GridBounds:
    """The only part of GridMap the controller reads (grid.hpp:214-235)."""

    xmin: float
    xmax: float
    ymin: float
    ymax: float

    def as_tuple(self):
        return (float(self.xmin), float(self.xmax), float(self.ymin), float(self.ymax))


def _is_cuda_tensor(a) -> bool:
    return torch is not None and isinstance(a, torch.Tensor) and a.is_cuda


def _np_f64(a, shape=None) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None and a.shape != tuple(shape):
        raise ValueError(f"expected shape {tuple(shape)}, got {a.shape}")
    return a


def map_batch_args(B: int, cells, resolution, origin, update, name: str):
    """Checks and marshals the per-instance map arguments of eb_set_map_targets_batch_* / eb_grid_batch_set_maps_*.
    Returns (device path?, the C arguments after the handle, the host arrays that must outlive the call)."""
    if len(cells) != B:
        raise ValueError(f"{name} needs {B} maps, got {len(cells)}")
    res = np.broadcast_to(np.asarray(resolution, dtype=np.float64), (B,)).copy() if np.ndim(resolution) == 0 \
        else _np_f64(resolution, (B,))
    org = _np_f64(origin, (B, 2))
    upd = None
    if update is not None:
        upd = np.ascontiguousarray(update)
        if upd.shape != (B,):
            raise ValueError(f"update must be ({B},), got {upd.shape}")
        upd = upd.astype(np.int32)
    present = [c for c in cells if c is not None]
    dev = bool(present) and _is_cuda_tensor(present[0])
    if any(_is_cuda_tensor(c) != dev for c in present):
        raise ValueError(f"{name}: cells must be all numpy arrays or all CUDA tensors")
    xs = np.zeros(B, dtype=np.uint32)
    ys = np.zeros(B, dtype=np.uint32)
    ptrs = (C.c_void_p * B)()
    keep = [ptrs, xs, ys, res, org, upd]
    for i, c in enumerate(cells):
        if c is None:
            continue
        if c.ndim != 2:
            raise ValueError(f"{name}: cells[{i}] must be 2-D (ysize, xsize), got {tuple(c.shape)}")
        if dev:
            if c.dtype != torch.int8 or not c.is_contiguous():
                raise ValueError(f"{name}: cells[{i}] must be a contiguous int8 tensor")
            ptrs[i] = c.data_ptr()
        else:
            c = np.ascontiguousarray(c)
            if c.dtype != np.int8:
                raise ValueError(f"{name}: cells[{i}] must be int8, got {c.dtype}")
            keep.append(c)
            ptrs[i] = c.ctypes.data
        ys[i], xs[i] = c.shape
    args = (C.addressof(ptrs), xs.ctypes.data, ys.ctypes.data, res.ctypes.data, org.ctypes.data,
            upd.ctypes.data if upd is not None else None)
    return dev, args, keep


def row_args(B: int, a, name: str) -> np.ndarray:
    """row_begin / row_count of the row-band calls as a (B,) uint32 host array"""
    a = np.asarray(a.cpu().numpy() if _is_cuda_tensor(a) else a)
    if a.shape != (B,) or (a.size and (not np.issubdtype(a.dtype, np.integer) or a.min() < 0 or a.max() > 0xFFFFFFFF)):
        raise ValueError(f"{name} must be ({B},) non-negative integers, got shape {a.shape}, dtype {a.dtype}")
    return np.ascontiguousarray(a, dtype=np.uint32)


def update_arg(B: int, update):
    """update of the batched map calls as a (B,) int32 host array, or None (all)"""
    if update is None:
        return None
    upd = np.ascontiguousarray(update)
    if upd.shape != (B,):
        raise ValueError(f"update must be ({B},), got {upd.shape}")
    return upd.astype(np.int32)


class ErgodicControl:
    """Batched drop-in for ErgodicControl<ModelT> (ergodic_control.hpp:72-185)."""

    def __init__(self, model, dt: float, horizon: float, resolution: float, exploration_weight: float,
                 num_basis: int, buffer_size: int, batch_size: int, Rinv, umin, umax, *, batch: int = 1,
                 device: int = 0, seed: int = 0xE16C0D1C, barrier_weight: float = 25.0,
                 barrier_eps: float = 0.05):
        self._lib = capi.load()
        cfg = EbConfig()
        model_id = model if isinstance(model, int) else model.model_id
        self._lib.eb_config_defaults(C.byref(cfg), model_id)
        cfg.batch, cfg.device = int(batch), int(device)
        cfg.dt, cfg.horizon, cfg.resolution = float(dt), float(horizon), float(resolution)
        cfg.expl_weight = float(exploration_weight)
        cfg.num_basis, cfg.buffer_size, cfg.batch_size = int(num_basis), int(buffer_size), int(batch_size)
        R = _np_f64(Rinv, (3, 3))
        for r in range(3):
            for c in range(3):
                cfg.Rinv[r + 3 * c] = R[r, c]  # column-major
        for i in range(3):
            cfg.umin[i] = float(umin[i])
            cfg.umax[i] = float(umax[i])
        cfg.barrier_weight, cfg.barrier_eps, cfg.seed = float(barrier_weight), float(barrier_eps), int(seed)
        h = C.c_void_p()
        st = self._lib.eb_create(C.byref(cfg), C.byref(h))
        if st == capi.EB_ERR_INVALID_ARGUMENT:
            raise ValueError(self._lib.eb_last_error().decode())  # std::invalid_argument in the reference
        check(st)
        self._h = h
        self.cfg = cfg
        self.batch = int(batch)
        self.device = int(device)
        self.steps = self._lib.eb_steps(h)
        self.num_coeff = self._lib.eb_num_coeff(h)
        self.batch_size = int(batch_size)

    # -- lifetime ---------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._lib.eb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def clone(self) -> "ErgodicControl":
        other = object.__new__(ErgodicControl)
        other.__dict__.update({k: v for k, v in self.__dict__.items() if k != "_h"})
        h = C.c_void_p()
        check(self._lib.eb_clone(self._h, C.byref(h)))
        other._h = h
        return other

    def _host_ptr(self, a: np.ndarray) -> int:
        """data pointer of a host array; a control loop passes the same buffers every tick, so the
        last few (array, pointer) pairs are remembered (holding the array keeps its id unique)"""
        cache = self.__dict__.setdefault("_ptrs", {})
        hit = cache.get(id(a))
        if hit is not None and hit[0] is a:
            return hit[1]
        if len(cache) >= 8:
            cache.clear()
        ptr = a.ctypes.data
        cache[id(a)] = (a, ptr)
        return ptr

    def _sync_stream(self):
        if torch is not None and torch.cuda.is_available():
            s = torch.cuda.current_stream(self.device).cuda_stream
            check(self._lib.eb_set_stream(self._h, C.c_void_p(s)))

    # -- reference API ------------------------------------------------------
    def timeStep(self) -> float:
        return self._lib.eb_time_step(self._h)

    def setTarget(self, target) -> None:
        gs = target.gaussians if isinstance(target, Target) else list(target)
        mu = _np_f64([g.mu for g in gs]).reshape(-1)
        sg = _np_f64([g.sigmas for g in gs]).reshape(-1)
        check(self._lib.eb_set_target_gaussians(self._h, len(gs), mu.ctypes.data, sg.ctypes.data))

    def configTarget(self, grid) -> bool:
        b = grid.as_tuple() if hasattr(grid, "as_tuple") else tuple(float(v) for v in grid)
        self._sync_stream()
        rebuilt = C.c_int(0)
        check(self._lib.eb_config_target(self._h, *b, C.byref(rebuilt)))
        return bool(rebuilt.value)

    def reserve_memory(self, count: int) -> None:
        """room for `count` stored states up front (no re-allocation inside the control loop)"""
        check(self._lib.eb_reserve_state_memory(self._h, int(count)))

    def addStateMemory(self, x) -> None:
        if _is_cuda_tensor(x):
            self._sync_stream()
            assert x.dtype == torch.float64 and x.is_contiguous() and x.numel() == 3 * self.batch
            check(self._lib.eb_add_state_memory_dev(self._h, C.c_void_p(x.data_ptr())))
        else:
            x = _np_f64(x).reshape(self.batch, 3)
            check(self._lib.eb_add_state_memory_host(self._h, x.ctypes.data))

    def control(self, grid, x, mem_idx=None, u0=None, metric=None):
        """One control() iteration for all instances.  Returns u0 (B, 3); pass
        ``metric`` (B,) to also receive sum_k lamda_k (c_k - phi_k)^2.

        ``grid``: one map for the whole batch (bounds or an object with them), or per-instance
        bounds (B, 4) {xmin, xmax, ymin, ymax} (array or CUDA tensor), or None on a per-instance
        controller: the frames of the last configure, no frame launch."""
        if grid is None or (type(grid) is not tuple and np.ndim(grid) == 2):
            return self._control_batch(grid, x, mem_idx, u0, metric)
        if type(grid) is tuple:  # a control loop passes the same bounds tuple every tick
            b = grid
        else:
            b = grid.as_tuple() if hasattr(grid, "as_tuple") else tuple(float(v) for v in grid)
        if _is_cuda_tensor(x):
            self._sync_stream()  # device path: run on torch's current stream
            assert x.dtype == torch.float64 and x.is_contiguous() and x.numel() == 3 * self.batch
            if u0 is None:
                u0 = torch.empty((self.batch, 3), dtype=torch.float64, device=x.device)
            idx_p = C.c_void_p(mem_idx.data_ptr()) if mem_idx is not None else None
            met_p = C.c_void_p(metric.data_ptr()) if metric is not None else None
            st = self._lib.eb_control_dev(self._h, *b, C.c_void_p(x.data_ptr()), idx_p,
                                          C.c_void_p(u0.data_ptr()), met_p)
        else:
            # host path: the call copies / maps the buffers and synchronises by itself
            if not (type(x) is np.ndarray and x.dtype == np.float64 and x.flags.c_contiguous
                    and x.size == 3 * self.batch):
                x = _np_f64(x).reshape(self.batch, 3)
            if u0 is None:
                u0 = np.empty((self.batch, 3))
            idx_p = None
            if mem_idx is not None:
                mem_idx = np.ascontiguousarray(mem_idx, dtype=np.int32)
                idx_p = mem_idx.ctypes.data
            met_p = self._host_ptr(metric) if metric is not None else None
            st = self._lib.eb_control_host(self._h, *b, self._host_ptr(x), idx_p, self._host_ptr(u0), met_p)
        if st != capi.EB_OK:
            if st == capi.EB_ERR_INVALID_ARGUMENT:
                raise ValueError(self._lib.eb_last_error().decode())
            check(st)
        return u0

    # -- per-instance targets (one target and map frame per instance) -------------------
    def _bounds_dev(self, bounds):
        b = torch.as_tensor(bounds, dtype=torch.float64, device=f"cuda:{self.device}").contiguous()
        if tuple(b.shape) != (self.batch, 4):
            raise ValueError(f"per-instance bounds must be ({self.batch}, 4), got {tuple(b.shape)}")
        return b

    def setTargets(self, targets) -> None:
        """Target::setTarget per instance: ``targets`` holds B Targets (or lists of Gaussians).
        Does not rebuild phi_k by itself (configTargets / control with bounds does)."""
        if len(targets) != self.batch:
            raise ValueError(f"setTargets needs {self.batch} targets, got {len(targets)}")
        gss = [t.gaussians if isinstance(t, Target) else list(t) for t in targets]
        counts = np.array([len(g) for g in gss], dtype=np.int32)
        max_n = max(1, int(counts.max()))
        mu = np.zeros((self.batch, max_n, 2))
        sg = np.ones((self.batch, max_n, 2))
        for i, g in enumerate(gss):
            for j, gi in enumerate(g):
                mu[i, j] = gi.mu
                sg[i, j] = gi.sigmas
        st = self._lib.eb_set_target_gaussians_batch(self._h, max_n, counts.ctypes.data, mu.ctypes.data, sg.ctypes.data)
        if st == capi.EB_ERR_INVALID_ARGUMENT:
            raise ValueError(self._lib.eb_last_error().decode())
        check(st)

    def configTargets(self, bounds) -> np.ndarray:
        """configTarget of every instance, bounds (B, 4) {xmin, xmax, ymin, ymax}.  Returns rebuilt (B,) bool.
        A moved extent without Gaussians surfaces from the next check()."""
        self._sync_stream()
        b = self._bounds_dev(bounds)
        rebuilt = torch.zeros(self.batch, dtype=torch.int32, device=b.device)
        check(self._lib.eb_config_target_batch_dev(self._h, C.c_void_p(b.data_ptr()), C.c_void_p(rebuilt.data_ptr())))
        return rebuilt.cpu().numpy().astype(bool)

    def set_phik_batch(self, phik, extent) -> None:
        """phi_k rows (B, K) and extents (B, 2) {lx, ly}, CUDA tensors (e.g. MapTarget.execute outputs);
        the origins of the frames are kept."""
        self._sync_stream()
        assert _is_cuda_tensor(phik) and _is_cuda_tensor(extent), "set_phik_batch takes CUDA tensors"
        assert phik.dtype == torch.float64 and phik.is_contiguous() and phik.numel() == self.batch * self.num_coeff
        assert extent.dtype == torch.float64 and extent.is_contiguous() and extent.numel() == 2 * self.batch
        check(self._lib.eb_set_phik_batch_dev(self._h, C.c_void_p(phik.data_ptr()), C.c_void_p(extent.data_ptr())))

    def setMapTargets(self, cells, resolution=None, origin=None, update=None, *, row_begin=None,
                      row_count=None) -> None:
        """Map-derived (entropy) target and map frame per instance, one kernel launch for the batch.

        ``cells`` may be a GridMapBatch of the same B on the same device: setMapTargets(grids, row_begin=None,
        row_count=None, update=None) (positionally, the second and third arguments are then row_begin and row_count)
        derives every flagged instance from map i of the batch, without uploading the cells again, bit for bit what
        the call with map i's cells, resolution and origin gives.  row_begin / row_count (B,) declare the rows of map i
        that changed (GridMapBatch.set_rows) since this controller last derived instance i from this batch; only the
        64-row units that meet them are recomputed.  None: whole maps.  Runs on torch's current stream when CUDA is
        available, after the work enqueued on the grid batch, without a host synchronisation.

        ``cells``: B int8 occupancy grids (ysize_i, xsize_i) in GridMap layout, all numpy (host path) or all CUDA
        tensors (device path, torch's current stream); the entry of an instance that is not updated may be None.
        ``resolution``: scalar or (B,); ``origin``: (B, 2) GridMap xmin / ymin; ``update``: (B,) bool or None (all).
        Instance i gets the row MapTarget(xsize_i, ysize_i, resolution_i, nb).execute(cells_i) and the frame
        origin_i, (xsize_i * res_i, ysize_i * res_i); control(None) or control(bounds of the maps) then uses them."""
        from .collision import GridMapBatch

        if isinstance(cells, GridMapBatch):
            if resolution is not None or origin is not None:
                if row_begin is not None or row_count is not None:
                    raise TypeError("setMapTargets(grids, ...): row_begin / row_count given twice")
                row_begin, row_count = resolution, origin
            return self._map_targets_from_grids(cells, row_begin, row_count, update)
        if resolution is None or origin is None:
            raise TypeError("setMapTargets(cells, resolution, origin, update=None) needs resolution and origin")
        dev, args, keep = map_batch_args(self.batch, cells, resolution, origin, update, "setMapTargets")
        if dev:
            self._sync_stream()
            st = self._lib.eb_set_map_targets_batch_dev(self._h, *args)
        else:
            st = self._lib.eb_set_map_targets_batch_host(self._h, *args)
        if st == capi.EB_ERR_INVALID_ARGUMENT:
            raise ValueError(self._lib.eb_last_error().decode())
        check(st)

    def _map_targets_from_grids(self, grids, row_begin, row_count, update):
        B = self.batch
        if grids.batch != B:
            raise ValueError(f"setMapTargets: the grid batch holds {grids.batch} maps for {B} instances")
        if (row_begin is None) != (row_count is None):
            raise ValueError("setMapTargets: row_begin and row_count must both be given or both be None")
        rb = row_args(B, row_begin, "row_begin") if row_begin is not None else None
        rc = row_args(B, row_count, "row_count") if row_count is not None else None
        upd = update_arg(B, update)
        self._sync_stream()
        grids._stream()
        st = self._lib.eb_set_map_targets_from_grid_batch(
            self._h, grids._h, rb.ctypes.data if rb is not None else None, rc.ctypes.data if rc is not None else None,
            upd.ctypes.data if upd is not None else None)
        if st == capi.EB_ERR_INVALID_ARGUMENT:
            raise ValueError(self._lib.eb_last_error().decode())
        check(st)

    def get_phik_batch(self):
        """(phik (B, K), extent (B, 2)) of a per-instance controller"""
        ph = np.empty((self.batch, self.num_coeff))
        ext = np.empty((self.batch, 2))
        st = self._lib.eb_get_phik_batch(self._h, ph.ctypes.data, ext.ctypes.data)
        if st == capi.EB_ERR_INVALID_ARGUMENT:
            raise ValueError(self._lib.eb_last_error().decode())
        check(st)
        return ph, ext

    def _control_batch(self, bounds, x, mem_idx, u0, metric):
        if _is_cuda_tensor(x):
            self._sync_stream()
            assert x.dtype == torch.float64 and x.is_contiguous() and x.numel() == 3 * self.batch
            b = self._bounds_dev(bounds) if bounds is not None else None
            if u0 is None:
                u0 = torch.empty((self.batch, 3), dtype=torch.float64, device=x.device)
            st = self._lib.eb_control_batch_dev(
                self._h, C.c_void_p(b.data_ptr()) if b is not None else None, C.c_void_p(x.data_ptr()),
                C.c_void_p(mem_idx.data_ptr()) if mem_idx is not None else None, C.c_void_p(u0.data_ptr()),
                C.c_void_p(metric.data_ptr()) if metric is not None else None)
        else:
            x = _np_f64(x).reshape(self.batch, 3)
            b = None
            if bounds is not None:
                b = bounds.cpu().numpy() if _is_cuda_tensor(bounds) else bounds
                b = _np_f64(b, (self.batch, 4))
            if u0 is None:
                u0 = np.empty((self.batch, 3))
            idx_p = None
            if mem_idx is not None:
                mem_idx = np.ascontiguousarray(mem_idx, dtype=np.int32)
                idx_p = mem_idx.ctypes.data
            st = self._lib.eb_control_batch_host(self._h, b.ctypes.data if b is not None else None, x.ctypes.data,
                                                 idx_p, u0.ctypes.data, metric.ctypes.data if metric is not None else None)
        if st != capi.EB_OK:
            if st == capi.EB_ERR_INVALID_ARGUMENT:
                raise ValueError(self._lib.eb_last_error().decode())
            check(st)
        return u0

    def control_safe(self, grids, dwa, x, vb, val_dt: float, val_horizon: float, bounds=None, mem_idx=None,
                     metric=None, collision=None):
        """One safe control tick of B robots on B maps, the reference loop's arbitration between the ergodic twist
        and the safety planner (exploration.hpp:238-247): control(bounds, x) of every instance, validate_control of
        its twist on its own map (``grids``, a GridMapBatch) with val_dt and val_horizon, and only where that twist
        collides DynamicWindow.control on that map with ``dwa``'s window, ``vb`` and the instance's optTraj() as the
        reference trajectory.  ``collision`` (default ``dwa.collision``) is the Collision of the tick: both the
        validation and the window's rollouts are checked with it, as in the reference node, which builds the window
        from the controller's Collision.

        Returns (u (B, 3), branch (B,) int32): branch 0 = the ergodic twist, 1 = the window's twist, 2 = the window
        found nothing and u = 0.  Bit for bit what those calls return one after the other, with the window run only
        for the robots that need it.  numpy inputs take the host path (copies, one synchronisation); CUDA tensors run
        on torch's current stream without a host synchronisation (``metric`` (B,) float64 and ``mem_idx`` int32 then
        tensors too).  ``bounds`` (B, 4) as in control(); None: the frames of the last configure."""
        B = self.batch
        dev = _is_cuda_tensor(x)
        x, vb = self._safe_rows(grids, x, vb, dev)
        col = dwa.collision if collision is None else collision
        if dev:
            b = self._dev_tick_args(bounds, mem_idx, metric)
            u = torch.empty((B, 3), dtype=torch.float64, device=x.device)
            branch = torch.empty(B, dtype=torch.int32, device=x.device)
            fn = self._lib.eb_control_safe_batch_dev
        else:
            b = None
            if bounds is not None:
                b = _np_f64(bounds.cpu().numpy() if _is_cuda_tensor(bounds) else bounds, (B, 4))
            if metric is not None and not (isinstance(metric, np.ndarray) and metric.dtype == np.float64 and
                                           metric.flags.c_contiguous and metric.shape == (B,)):
                raise ValueError(f"metric must be a contiguous ({B},) float64 numpy array on the host path")
            if mem_idx is not None:
                mem_idx = np.ascontiguousarray(mem_idx, dtype=np.int32)
            u, branch = np.empty((B, 3)), np.empty(B, dtype=np.int32)
            fn = self._lib.eb_control_safe_batch_host
        P = grids._ptr
        self._sync_stream()
        grids._stream()
        st = fn(self._h, grids._h, C.byref(col.cfg), C.byref(dwa.cfg), float(val_dt), float(val_horizon),
                P(b) if b is not None else None, P(x), P(mem_idx) if mem_idx is not None else None, P(vb), P(u),
                P(branch), P(metric) if metric is not None else None)
        if st != capi.EB_OK:
            if st == capi.EB_ERR_INVALID_ARGUMENT:
                raise ValueError(self._lib.eb_last_error().decode())
            check(st)
        return u, branch

    def _safe_rows(self, grids, x, vb, dev):
        """x and vb of a safe tick as (B, 3) rows of the grid batch's robots, on the path of the call"""
        if grids.batch != self.batch:
            raise ValueError(f"control_safe: the grid batch holds {grids.batch} maps for {self.batch} instances")
        x, _, _ = grids._rows("x", x, dev, per_ok=False)
        vb, _, _ = grids._rows("vb", vb, dev, per_ok=False)
        return x, vb

    def _dev_tick_args(self, bounds, mem_idx, metric):
        """the device path's bounds (B, 4) as a CUDA tensor or None, after checking metric and mem_idx"""
        B = self.batch
        b = self._bounds_dev(bounds) if bounds is not None else None
        if metric is not None and not (_is_cuda_tensor(metric) and metric.dtype == torch.float64 and
                                       metric.is_contiguous() and tuple(metric.shape) == (B,)):
            raise ValueError(f"metric must be a contiguous ({B},) float64 CUDA tensor on the device path")
        if mem_idx is not None and not (_is_cuda_tensor(mem_idx) and mem_idx.dtype == torch.int32 and
                                        mem_idx.is_contiguous()):
            raise ValueError("mem_idx must be a contiguous int32 CUDA tensor on the device path")
        return b

    def check(self) -> None:
        """Synchronise and surface device-side faults of earlier device-path calls."""
        st = self._lib.eb_check_status(self._h)
        if st == capi.EB_ERR_INVALID_ARGUMENT:
            raise ValueError(self._lib.eb_last_error().decode())
        check(st)

    def optTraj(self, out=None):
        self._sync_stream()
        if _is_cuda_tensor(out):
            check(self._lib.eb_opt_traj_dev(self._h, C.c_void_p(out.data_ptr())))
            return out
        xt = np.empty((self.batch, self.steps, 3))
        st = self._lib.eb_opt_traj_host(self._h, xt.ctypes.data)
        if st == capi.EB_ERR_INVALID_ARGUMENT:
            raise ValueError(self._lib.eb_last_error().decode())
        check(st)
        return xt

    # -- state access (checkpoint / teacher forcing) -------------------------
    def get_ut(self) -> np.ndarray:
        ut = np.empty((self.batch, self.steps, 3))
        check(self._lib.eb_get_ut(self._h, ut.ctypes.data))
        return ut

    def set_ut(self, ut) -> None:
        ut = _np_f64(ut).reshape(self.batch, self.steps, 3)
        check(self._lib.eb_set_ut(self._h, ut.ctypes.data))

    def keep_ck(self, keep: bool) -> None:
        """store (default) or skip the per-instance c_k by-product of control()"""
        check(self._lib.eb_set_keep_ck(self._h, int(bool(keep))))

    def get_ck(self) -> np.ndarray:
        ck = np.empty((self.batch, self.num_coeff))
        check(self._lib.eb_get_ck(self._h, ck.ctypes.data))
        return ck

    def get_phik(self):
        ph = np.empty(self.num_coeff)
        lx, ly = C.c_double(0), C.c_double(0)
        check(self._lib.eb_get_phik(self._h, ph.ctypes.data, C.byref(lx), C.byref(ly)))
        return ph, lx.value, ly.value

    def set_phik(self, phik, lx: float, ly: float) -> None:
        if _is_cuda_tensor(phik):  # e.g. the output of MapTarget.execute / PhikPlan.execute: no host round trip
            self._sync_stream()
            assert phik.dtype == torch.float64 and phik.is_contiguous() and phik.numel() == self.num_coeff
            check(self._lib.eb_set_phik_dev(self._h, C.c_void_p(phik.data_ptr()), float(lx), float(ly)))
            return
        ph = _np_f64(phik).reshape(self.num_coeff)
        check(self._lib.eb_set_phik(self._h, ph.ctypes.data, float(lx), float(ly)))

    def memory_size(self) -> int:
        return int(self._lib.eb_memory_size(self._h))

    def last_mem_idx(self) -> Optional[np.ndarray]:
        n = C.c_int(0)
        idx = np.zeros((self.batch, self.batch_size), dtype=np.int32)
        check(self._lib.eb_get_last_mem_idx(self._h, idx.ctypes.data, C.byref(n)))
        return idx[:, : n.value] if n.value > 0 else None

    def launch_count(self) -> int:
        return int(self._lib.eb_launch_count(self._h))


class PhikPlan:
    """phi_k = (C_y^T Phi C_x) / sum(Phi) for a dense density on the
    configTarget grid (Target::fill normalisation + Basis::spatialCoeff)."""

    def __init__(self, nx: int, ny: int, resolution: float, lx: float, ly: float, nb: int, device: int = 0,
                 algo: int = 0, row_begin: int = 0, ny_total: Optional[int] = None, x_first: float = 0.0,
                 y_first: float = 0.0):
        """ny rows starting at row_begin of an ny_total-row grid (default: the whole grid); x_first / y_first: the
        coordinate of the first sample point (0: the configTarget grid; resolution / 2: cell centres)"""
        self._lib = capi.load()
        h = C.c_void_p()
        ny_total = ny if ny_total is None else ny_total
        st = self._lib.eb_phik_plan_create_ex(device, nx, ny_total, row_begin, ny, float(resolution), float(lx),
                                              float(ly), nb, float(x_first), float(y_first), C.byref(h))
        if st == capi.EB_ERR_INVALID_ARGUMENT:
            raise ValueError(self._lib.eb_last_error().decode())
        check(st)
        self._h, self.nx, self.ny, self.nb, self.device = h, nx, ny, nb, device
        if algo:
            check(self._lib.eb_phik_plan_set_algo(h, algo))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.eb_phik_plan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def execute(self, phi, phik=None, phi_sum=None):
        if _is_cuda_tensor(phi):
            s = torch.cuda.current_stream(self.device).cuda_stream
            check(self._lib.eb_phik_plan_set_stream(self._h, C.c_void_p(s)))
            assert phi.dtype == torch.float64 and phi.is_contiguous() and phi.numel() == self.nx * self.ny
            if phik is None:
                phik = torch.empty(self.nb * self.nb, dtype=torch.float64, device=phi.device)
            sp = C.c_void_p(phi_sum.data_ptr()) if phi_sum is not None else None
            check(self._lib.eb_phik_execute_dev(self._h, C.c_void_p(phi.data_ptr()), C.c_void_p(phik.data_ptr()), sp))
            return phik
        phi = _np_f64(phi).reshape(self.ny, self.nx)
        out = np.empty(self.nb * self.nb)
        s = C.c_double(0.0)
        check(self._lib.eb_phik_execute_host(self._h, phi.ctypes.data, out.ctypes.data, C.byref(s)))
        self.last_sum = s.value
        return out

    def execute_raw(self, phi, raw=None):
        """un-normalised contraction of this plan's rows: (ld, ld) torch tensor with ld = 32 for nb <= 32, else nb
        rounded up to a multiple of 32; raw[0, 0] = sum(phi)"""
        s = torch.cuda.current_stream(self.device).cuda_stream
        check(self._lib.eb_phik_plan_set_stream(self._h, C.c_void_p(s)))
        assert _is_cuda_tensor(phi) and phi.dtype == torch.float64 and phi.is_contiguous()
        assert phi.numel() == self.nx * self.ny
        if raw is None:
            ld = 32 if self.nb <= 32 else (self.nb + 31) // 32 * 32
            raw = torch.empty((ld, ld), dtype=torch.float64, device=phi.device)
        check(self._lib.eb_phik_execute_raw_dev(self._h, C.c_void_p(phi.data_ptr()), C.c_void_p(raw.data_ptr())))
        return raw

    def launch_count(self) -> int:
        return int(self._lib.eb_phik_launch_count(self._h))

    def fold(self):
        """(mirror fold usable on this grid, measured asymmetry of the cosine table)"""
        f, d = C.c_int(0), C.c_double(0.0)
        check(self._lib.eb_phik_plan_fold(self._h, C.byref(f), C.byref(d)))
        return bool(f.value), d.value


class MapTarget:
    """Map-derived target (SURVEY.md section 8f-4): int8 occupancy grid -> entropy per cell (numerics.hpp:164-179
    over GridMap::getCell) -> normalised density -> phi_k, all on the device.  One execute per map update."""

    def __init__(self, xsize: int, ysize: int, resolution: float, nb: int, device: int = 0):
        self._lib = capi.load()
        h = C.c_void_p()
        st = self._lib.eb_map_target_create(device, int(xsize), int(ysize), float(resolution), int(nb), C.byref(h))
        if st == capi.EB_ERR_INVALID_ARGUMENT:
            raise ValueError(self._lib.eb_last_error().decode())
        check(st)
        self._h, self.xsize, self.ysize, self.nb, self.device = h, int(xsize), int(ysize), int(nb), int(device)
        self.lx, self.ly = xsize * float(resolution), ysize * float(resolution)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.eb_map_target_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def execute(self, cells, phik=None):
        """cells: (ysize, xsize) int8, torch CUDA tensor (device path, current stream) or numpy (host path)"""
        if _is_cuda_tensor(cells):
            s = torch.cuda.current_stream(self.device).cuda_stream
            check(self._lib.eb_map_target_set_stream(self._h, C.c_void_p(s)))
            assert cells.dtype == torch.int8 and cells.is_contiguous() and cells.numel() == self.xsize * self.ysize
            if phik is None:
                phik = torch.empty(self.nb * self.nb, dtype=torch.float64, device=cells.device)
            check(self._lib.eb_map_target_execute_dev(self._h, C.c_void_p(cells.data_ptr()), C.c_void_p(phik.data_ptr()), None))
            return phik
        cells = np.ascontiguousarray(cells, dtype=np.int8).reshape(self.ysize, self.xsize)
        out = np.empty(self.nb * self.nb)
        s = C.c_double(0.0)
        check(self._lib.eb_map_target_execute_host(self._h, cells.ctypes.data, out.ctypes.data, C.byref(s)))
        self.last_sum = s.value
        return out

    def density(self):
        """the un-normalised entropy density of the last execute, (ysize, xsize) torch view of device memory"""
        from .sharding import _DevView
        ptr = self._lib.eb_map_target_density_dev(self._h)
        return torch.as_tensor(_DevView(ptr, (self.ysize, self.xsize)), device=torch.device("cuda", self.device))

    def launch_count(self) -> int:
        return int(self._lib.eb_map_target_launch_count(self._h))


def l2_gather_peak(device: int = 0) -> float:
    """measured G sectors/s of random 1-byte loads over a 16 MB L2-resident buffer"""
    lib = capi.load()
    v = C.c_double(0)
    check(lib.eb_l2_gather_peak(device, C.byref(v)))
    return v.value


def fp64_peak(device: int = 0):
    """Measured FP64 TFLOP/s of the device: (DFMA loop, DMMA loop)."""
    lib = capi.load()
    a, b = C.c_double(0), C.c_double(0)
    check(lib.eb_fp64_peak(device, C.byref(a), C.byref(b)))
    return a.value, b.value

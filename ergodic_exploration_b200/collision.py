"""Host-side mirror of the reference's occupancy-grid collision API over the C ABI.

``Collision`` (collision.hpp:85-165), ``GridMap`` (grid.hpp:80-260, the parts the
checks read), ``validate_control`` (numerics.hpp:312-330) and ``DynamicWindow``
(dynamic_window.hpp:60-172) keep the
reference's names and argument meaning for a BATCH of poses / candidate twists
sharing one map (``GridMap``) or for B instances on B maps (``GridMapBatch``).  numpy arrays go through the ``_host`` entry points, torch
CUDA tensors through the ``_dev`` ones.  Everything is computed by
csrc/collision_kernels.cuh; this file only marshals pointers.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi
from .capi import EbCollision, EbDwa, check
from .controller import map_batch_args, row_args, update_arg

try:
    import torch
except Exception:  # pragma: no cover
    torch = None


def _is_cuda(a) -> bool:
    return torch is not None and isinstance(a, torch.Tensor) and a.is_cuda


class Collision:
    """2-D collision detector parameters (collision.hpp:95-96).  Raises ValueError
    where the reference constructor throws std::invalid_argument (collision.cpp:52-63)."""

    def __init__(self, boundary_radius: float, search_radius: float, obstacle_threshold: float,
                 occupied_threshold: float):
        if search_radius < boundary_radius:
            raise ValueError("Search radius must be at least the same size as the boundary radius")
        if occupied_threshold > 100.0 or occupied_threshold < 0.0:
            raise ValueError("Occupied threshold must be between 0 and 100")
        self.cfg = EbCollision(float(boundary_radius), float(search_radius), float(obstacle_threshold),
                               float(occupied_threshold))

    def totalPadding(self) -> float:
        return self.cfg.boundary_radius + self.cfg.obstacle_threshold

    def collisionCheck(self, grid, pose):
        """collision.cpp:126-143 for a batch of poses, 1 = collision.  GridMap: (n, 3) -> int32 (n,).
        GridMapBatch: (B, 3) -> (B,) or (B, per, 3) -> (B, per), instance i's poses checked against map i."""
        return grid._check(self, pose)


class GridMap:
    """Occupancy grid resident on the GPU (grid.hpp:94-95: bounds, resolution, int8 cells
    in row-major order, i = y row / j = x column)."""

    def __init__(self, xmin: float, xmax: float, ymin: float, ymax: float, resolution: float, grid_data,
                 device: int = 0):
        self._lib = capi.load()
        data = np.ascontiguousarray(grid_data, dtype=np.int8)
        xsize = int(round((xmax - xmin) / resolution))  # axis_length grid.hpp:61-64
        ysize = int(round((ymax - ymin) / resolution))
        if xsize * ysize != data.size:
            raise ValueError("Grid data size does not match the grid size")  # grid.cpp:57-60
        self.xsize, self.ysize, self.resolution = xsize, ysize, float(resolution)
        self.xmin, self.xmax, self.ymin, self.ymax = float(xmin), float(xmax), float(ymin), float(ymax)
        self.device = device
        h = C.c_void_p()
        check(self._lib.eb_grid_create(device, data.ctypes.data, xsize, ysize, float(resolution), float(xmin),
                                       float(ymin), C.byref(h)))
        self._h = h

    def as_tuple(self):
        return (self.xmin, self.xmax, self.ymin, self.ymax)

    def update(self, grid_data) -> None:
        data = np.ascontiguousarray(grid_data, dtype=np.int8)
        if data.size != self.xsize * self.ysize:
            raise ValueError("Grid data size does not match the grid size")
        check(self._lib.eb_grid_update(self._h, data.ctypes.data))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.eb_grid_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def launch_count(self) -> int:
        return int(self._lib.eb_grid_launch_count(self._h))

    def dilation(self, mode: int) -> None:
        """0 = automatic, 1 = always walk the circles, 2 = always use the pre-dilated map"""
        check(self._lib.eb_grid_set_dilation(self._h, int(mode)))

    def _stream(self):
        if torch is not None and torch.cuda.is_available():
            s = torch.cuda.current_stream(self.device).cuda_stream
            check(self._lib.eb_grid_set_stream(self._h, C.c_void_p(s)))

    def _check(self, collision: Collision, pose):
        self._stream()
        if _is_cuda(pose):
            assert pose.dtype == torch.float64 and pose.is_contiguous() and pose.numel() % 3 == 0
            n = pose.numel() // 3
            out = torch.empty(n, dtype=torch.int32, device=pose.device)
            check(self._lib.eb_collision_check_dev(self._h, C.byref(collision.cfg), C.c_void_p(pose.data_ptr()), n,
                                                   C.c_void_p(out.data_ptr())))
            return out
        pose = np.ascontiguousarray(pose, dtype=np.float64).reshape(-1, 3)
        out = np.empty(len(pose), dtype=np.int32)
        check(self._lib.eb_collision_check_host(self._h, C.byref(collision.cfg), pose.ctypes.data, len(pose),
                                                out.ctypes.data))
        return out

    def _validate(self, collision: Collision, x0, u, dt: float, horizon: float):
        self._stream()
        if _is_cuda(x0):
            assert _is_cuda(u) and x0.dtype == torch.float64 and u.dtype == torch.float64
            assert x0.is_contiguous() and u.is_contiguous() and x0.numel() == u.numel()
            n = x0.numel() // 3
            out = torch.empty(n, dtype=torch.int32, device=x0.device)
            check(self._lib.eb_validate_control_dev(self._h, C.byref(collision.cfg), C.c_void_p(x0.data_ptr()),
                                                    C.c_void_p(u.data_ptr()), n, float(dt), float(horizon),
                                                    C.c_void_p(out.data_ptr())))
            return out
        x0 = np.ascontiguousarray(x0, dtype=np.float64).reshape(-1, 3)
        u = np.ascontiguousarray(u, dtype=np.float64).reshape(-1, 3)
        if x0.shape != u.shape:
            raise ValueError("x0 and u must have the same shape")
        out = np.empty(len(x0), dtype=np.int32)
        check(self._lib.eb_validate_control_host(self._h, C.byref(collision.cfg), x0.ctypes.data, u.ctypes.data,
                                                 len(x0), float(dt), float(horizon), out.ctypes.data))
        return out


def validate_control(collision: Collision, grid, x0, u, dt: float, horizon: float):
    """numerics.hpp:312-330 for a batch: (B, 3) start poses and twists -> int32 (B,),
    1 = the twist held for |horizon / dt| steps stays collision free.  With a GridMapBatch, x0 and u may also be
    (B, per, 3) -> (B, per), instance i's rows checked against map i."""
    return grid._validate(collision, x0, u, dt, horizon)


class DynamicWindow:
    """Dynamic window approach for a batch of robots sharing one map (dynamic_window.hpp:60-65;
    same constructor argument order).  ``control`` mirrors both reference overloads
    (dynamic_window.cpp:93-139 with a reference twist, :141-187 with a reference trajectory)
    and returns (found (B,), u_opt (B, 3)) -- numpy in, numpy out; torch CUDA in, torch out."""

    def __init__(self, collision: Collision, dt: float, horizon: float, acc_dt: float, acc_lim_x: float,
                 acc_lim_y: float, acc_lim_th: float, max_vel_x: float, min_vel_x: float, max_vel_y: float,
                 min_vel_y: float, max_rot_vel: float, min_rot_vel: float, vx_samples: int, vy_samples: int,
                 vth_samples: int):
        self._lib = capi.load()
        self.collision = collision
        self.cfg = EbDwa(float(dt), float(horizon), float(acc_dt), float(acc_lim_x), float(acc_lim_y),
                         float(acc_lim_th), float(max_vel_x), float(min_vel_x), float(max_vel_y), float(min_vel_y),
                         float(max_rot_vel), float(min_rot_vel), int(vx_samples), int(vy_samples), int(vth_samples))

    def timeStep(self) -> float:
        return self.cfg.dt

    def horizon(self) -> float:
        return self.cfg.horizon

    def steps(self) -> int:
        return int(abs(self.cfg.horizon / self.cfg.dt))

    def control(self, grid, x0, vb, vref=None, xt_ref=None, dt_ref: float = 0.0, min_cost=None, out=None):
        """vref: (B, 3) reference twists, or xt_ref: a reference trajectory (ncols, 3) shared by the batch
        or (B, ncols, 3) per instance (e.g. ErgodicControl.optTraj()) with its time step dt_ref.
        Host path: ``out=(found int32 (B,), u (B, 3))`` lets a control loop reuse (page-locked) result buffers;
        with every buffer page-locked, large batches are copied and computed in overlapping slices.
        grid may be a GridMapBatch: robot i (row i of x0, vb, vref / xt_ref) is then driven on map i."""
        if (vref is None) == (xt_ref is None):
            raise ValueError("give either vref or xt_ref")
        if isinstance(grid, GridMapBatch):
            return grid._dwa(self, x0, vb, vref, xt_ref, dt_ref, min_cost)
        grid._stream()
        col, cfg = C.byref(self.collision.cfg), C.byref(self.cfg)
        if _is_cuda(x0):
            n = x0.numel() // 3
            found = torch.empty(n, dtype=torch.int32, device=x0.device)
            u = torch.empty((n, 3), dtype=torch.float64, device=x0.device)
            ref = vref if vref is not None else xt_ref
            for t in (x0, vb, ref):
                assert _is_cuda(t) and t.dtype == torch.float64 and t.is_contiguous()
            mc = C.c_void_p(min_cost.data_ptr()) if min_cost is not None else None
            P = lambda t: C.c_void_p(t.data_ptr())
            if vref is not None:
                check(self._lib.eb_dwa_control_twist_dev(grid._h, col, cfg, P(x0), P(vb), P(vref), n, P(found), P(u), mc))
            else:
                per = 1 if xt_ref.dim() == 3 else 0
                ncols = xt_ref.shape[-2]
                check(self._lib.eb_dwa_control_traj_dev(grid._h, col, cfg, P(x0), P(vb), P(xt_ref), ncols, per,
                                                        float(dt_ref), n, P(found), P(u), mc))
            return found, u
        x0 = np.ascontiguousarray(x0, dtype=np.float64).reshape(-1, 3)
        vb = np.ascontiguousarray(vb, dtype=np.float64).reshape(-1, 3)
        n = len(x0)
        if out is not None:
            found, u = out
            assert found.dtype == np.int32 and found.size == n and u.dtype == np.float64 and u.size == 3 * n
            assert found.flags.c_contiguous and u.flags.c_contiguous
        else:
            found, u = np.empty(n, dtype=np.int32), np.empty((n, 3))
        mc = min_cost.ctypes.data if min_cost is not None else None
        if vref is not None:
            vref = np.ascontiguousarray(vref, dtype=np.float64).reshape(-1, 3)
            st = self._lib.eb_dwa_control_twist_host(grid._h, col, cfg, x0.ctypes.data, vb.ctypes.data, vref.ctypes.data,
                                                     n, found.ctypes.data, u.ctypes.data, mc)
        else:
            xt = np.ascontiguousarray(xt_ref, dtype=np.float64)
            per = 1 if xt.ndim == 3 else 0
            st = self._lib.eb_dwa_control_traj_host(grid._h, col, cfg, x0.ctypes.data, vb.ctypes.data, xt.ctypes.data,
                                                    xt.shape[-2], per, float(dt_ref), n, found.ctypes.data,
                                                    u.ctypes.data, mc)
        if st == capi.EB_ERR_INVALID_ARGUMENT:
            raise ValueError(self._lib.eb_last_error().decode())
        check(st)
        return found, u


class GridMapBatch:
    """B occupancy grids resident on the GPU, one per instance, each with its own shape, resolution and origin.
    Collision.collisionCheck, validate_control and DynamicWindow.control take it in place of a GridMap and check
    instance i against map i, one kernel launch per call; every result equals the GridMap call on map i with
    dilation(1), bit for bit."""

    def __init__(self, batch: int, device: int = 0):
        self._lib = capi.load()
        self.batch, self.device = int(batch), device
        h = C.c_void_p()
        check(self._lib.eb_grid_batch_create(device, self.batch, C.byref(h)))
        self._h = h
        self._shape = [None] * self.batch  # (ysize, xsize) of each map that has been set

    def set(self, cells, resolution, origin, update=None) -> None:
        """The maps of the flagged instances, with the arguments of ErgodicControl.setMapTargets: ``cells`` B int8
        (ysize_i, xsize_i) grids, all numpy (host path) or all CUDA tensors (device path, torch's current stream; the
        tensors must stay alive until the copy has run on that stream); ``resolution`` scalar or (B,); ``origin``
        (B, 2) GridMap xmin / ymin; ``update`` (B,) bool or None (all).  Unflagged instances keep their maps."""
        dev, args, keep = map_batch_args(self.batch, cells, resolution, origin, update, "GridMapBatch.set")
        self._stream()
        st = (self._lib.eb_grid_batch_set_maps_dev if dev else self._lib.eb_grid_batch_set_maps_host)(self._h, *args)
        if st == capi.EB_ERR_INVALID_ARGUMENT:
            raise ValueError(self._lib.eb_last_error().decode())
        check(st)
        del keep
        for i, c in enumerate(cells):
            if update is None or update[i]:
                self._shape[i] = tuple(int(v) for v in c.shape)

    def set_rows(self, rows, row_begin, update=None) -> None:
        """Rows [row_begin[i], row_begin[i] + n_i) of map i of every flagged instance <- ``rows[i]``, an (n_i, xsize_i)
        int8 array (all numpy: host path; all CUDA tensors: device path on torch's current stream, the tensors must
        stay alive until the copy has run) or None (nothing written).  Shapes, resolutions and origins do not change;
        the map must have been set.  One kernel launch.  Pass the same row_begin and each band's n_i as row_count to
        ErgodicControl.setMapTargets(grids, row_begin, row_count) to recompute only the changed rows' targets."""
        B = self.batch
        if len(rows) != B:
            raise ValueError(f"GridMapBatch.set_rows needs {B} bands, got {len(rows)}")
        rb = row_args(B, row_begin, "row_begin")
        upd = update_arg(B, update)
        present = [r for r in rows if r is not None]
        dev = bool(present) and _is_cuda(present[0])
        if any(_is_cuda(r) != dev for r in present):
            raise ValueError("GridMapBatch.set_rows: rows must be all numpy arrays or all CUDA tensors")
        rc = np.zeros(B, dtype=np.uint32)
        ptrs = (C.c_void_p * B)()
        keep = []
        for i, r in enumerate(rows):
            if r is None or (upd is not None and not upd[i]):
                continue
            if self._shape[i] is None:
                raise ValueError(f"GridMapBatch.set_rows: instance {i} has no map")
            if r.ndim != 2 or r.shape[1] != self._shape[i][1]:
                raise ValueError(f"GridMapBatch.set_rows: rows[{i}] must be (n, {self._shape[i][1]}), got {tuple(r.shape)}")
            if dev:
                if r.dtype != torch.int8 or not r.is_contiguous():
                    raise ValueError(f"GridMapBatch.set_rows: rows[{i}] must be a contiguous int8 tensor")
                ptrs[i] = r.data_ptr()
            else:
                r = np.ascontiguousarray(r)
                if r.dtype != np.int8:
                    raise ValueError(f"GridMapBatch.set_rows: rows[{i}] must be int8, got {r.dtype}")
                keep.append(r)
                ptrs[i] = r.ctypes.data
            rc[i] = r.shape[0]
        self._stream()
        fn = self._lib.eb_grid_batch_set_rows_dev if dev else self._lib.eb_grid_batch_set_rows_host
        self._raise(fn(self._h, C.addressof(ptrs), rb.ctypes.data, rc.ctypes.data,
                       upd.ctypes.data if upd is not None else None))
        del keep

    def get_map(self, i: int) -> np.ndarray:
        """map i as held on the device, a (ysize_i, xsize_i) int8 numpy array (synchronises)"""
        if not 0 <= i < self.batch or self._shape[i] is None:
            raise ValueError(f"GridMapBatch.get_map: instance {i} has no map")
        out = np.empty(self._shape[i], dtype=np.int8)
        self._raise(self._lib.eb_grid_batch_get_map_host(self._h, int(i), out.ctypes.data))
        return out

    def launch_count(self) -> int:
        return int(self._lib.eb_grid_batch_launch_count(self._h))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.eb_grid_batch_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        if torch is not None and torch.cuda.is_available():
            s = torch.cuda.current_stream(self.device).cuda_stream
            check(self._lib.eb_grid_batch_set_stream(self._h, C.c_void_p(s)))

    def _raise(self, st):
        if st == capi.EB_ERR_INVALID_ARGUMENT:
            raise ValueError(self._lib.eb_last_error().decode())
        check(st)

    def _rows(self, name, a, dev, per_ok=True):
        """a as (B, 3) or (B, per, 3) float64, C-contiguous, on the path of the call; returns (a, per, shape)"""
        if _is_cuda(a) != dev:
            raise ValueError(f"{name}: inputs must be all numpy arrays or all CUDA tensors")
        if dev:
            if a.dtype != torch.float64 or not a.is_contiguous():
                raise ValueError(f"{name} must be a contiguous float64 tensor")
        else:
            a = np.ascontiguousarray(a, dtype=np.float64)
        shape = tuple(a.shape)
        if not ((len(shape) == 2 or (per_ok and len(shape) == 3)) and shape[0] == self.batch and shape[-1] == 3):
            raise ValueError(f"{name} must be ({self.batch}, 3)" + (f" or ({self.batch}, per, 3)" if per_ok else "") +
                             f", got {shape}")
        return a, (shape[1] if len(shape) == 3 else 1), shape[:-1]

    @staticmethod
    def _ptr(a):
        return C.c_void_p(a.data_ptr()) if _is_cuda(a) else a.ctypes.data

    @staticmethod
    def _out(dev, shape, like, dtype):
        if dev:
            return torch.empty(shape, dtype=torch.int32 if dtype == np.int32 else torch.float64, device=like.device)
        return np.empty(shape, dtype=dtype)

    def _check(self, collision: Collision, pose):
        dev = _is_cuda(pose)
        pose, per, shape = self._rows("poses", pose, dev)
        self._stream()
        out = self._out(dev, shape, pose, np.int32)
        fn = self._lib.eb_collision_check_batch_dev if dev else self._lib.eb_collision_check_batch_host
        self._raise(fn(self._h, C.byref(collision.cfg), self._ptr(pose), per, self._ptr(out)))
        return out

    def _validate(self, collision: Collision, x0, u, dt: float, horizon: float):
        dev = _is_cuda(x0)
        x0, per, shape = self._rows("x0", x0, dev)
        u, _, ushape = self._rows("u", u, dev)
        if ushape != shape:
            raise ValueError(f"x0 and u must have the same shape, got {shape} and {ushape}")
        self._stream()
        out = self._out(dev, shape, x0, np.int32)
        fn = self._lib.eb_validate_control_batch_dev if dev else self._lib.eb_validate_control_batch_host
        self._raise(fn(self._h, C.byref(collision.cfg), self._ptr(x0), self._ptr(u), per, float(dt), float(horizon),
                       self._ptr(out)))
        return out

    def _dwa(self, dwa: "DynamicWindow", x0, vb, vref, xt_ref, dt_ref, min_cost):
        B, dev = self.batch, _is_cuda(x0)
        x0, _, _ = self._rows("x0", x0, dev, per_ok=False)
        vb, _, _ = self._rows("vb", vb, dev, per_ok=False)
        if vref is not None:
            ref, _, _ = self._rows("vref", vref, dev, per_ok=False)
        else:
            if _is_cuda(xt_ref) != dev:
                raise ValueError("xt_ref: inputs must be all numpy arrays or all CUDA tensors")
            ref = xt_ref if dev else np.ascontiguousarray(xt_ref, dtype=np.float64)
            if dev and (ref.dtype != torch.float64 or not ref.is_contiguous()):
                raise ValueError("xt_ref must be a contiguous float64 tensor")
            shape = tuple(ref.shape)
            if not (shape[-1:] == (3,) and (len(shape) == 2 or (len(shape) == 3 and shape[0] == B)) and shape[-2] >= 1):
                raise ValueError(f"xt_ref must be (ncols, 3) or ({B}, ncols, 3), got {shape}")
        if min_cost is not None and (tuple(min_cost.shape) != (B,) or _is_cuda(min_cost) != dev or
                                     (not dev and (min_cost.dtype != np.float64 or not min_cost.flags.c_contiguous))):
            raise ValueError(f"min_cost must be a contiguous ({B},) float64 array on the path of x0")
        self._stream()
        found = self._out(dev, (B,), x0, np.int32)
        u = self._out(dev, (B, 3), x0, np.float64)
        col, cfg = C.byref(dwa.collision.cfg), C.byref(dwa.cfg)
        mc = self._ptr(min_cost) if min_cost is not None else None
        P = self._ptr
        if vref is not None:
            fn = self._lib.eb_dwa_control_twist_batch_dev if dev else self._lib.eb_dwa_control_twist_batch_host
            st = fn(self._h, col, cfg, P(x0), P(vb), P(ref), P(found), P(u), mc)
        else:
            fn = self._lib.eb_dwa_control_traj_batch_dev if dev else self._lib.eb_dwa_control_traj_batch_host
            st = fn(self._h, col, cfg, P(x0), P(vb), P(ref), ref.shape[-2], 1 if ref.ndim == 3 else 0, float(dt_ref),
                    P(found), P(u), mc)
        self._raise(st)
        return found, u


def integrate_twist(x, u, dt: float, out=None):
    """numerics.hpp:273-298 + the angle wrap :77-89 for (B, 3) torch CUDA poses and twists, on the
    current stream; ``out`` may be ``x`` itself"""
    assert _is_cuda(x) and _is_cuda(u) and x.dtype == torch.float64 and u.dtype == torch.float64
    assert x.is_contiguous() and u.is_contiguous() and x.numel() == u.numel()
    if out is None:
        out = torch.empty_like(x)
    dev = x.device.index or 0
    s = torch.cuda.current_stream(dev).cuda_stream
    check(capi.load().eb_integrate_twist_dev(dev, C.c_void_p(x.data_ptr()), C.c_void_p(u.data_ptr()), float(dt),
                                             x.numel() // 3, C.c_void_p(out.data_ptr()), C.c_void_p(s)))
    return out

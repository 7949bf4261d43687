"""Multi-GPU plumbing: one process per GPU, torch.distributed (NCCL over
NVLink/NVSwitch on the GPU box, gloo in the CPU tests).

The hot path shards by construction (SURVEY.md §8e):
  * control(): instances are independent, so they are block-partitioned over
    the ranks, every rank keeps its instances' ut_/memory resident for the
    whole run, there is NO data-path collective inside a step, and the first
    twists are collected with one all_gather per step.
  * phi_k: the density grid is partitioned by row blocks, every rank contracts
    its rows (eb_phik_execute_raw_dev) and ONE all_reduce(sum) of the 32x32 raw
    block (which includes sum(Phi) at [0,0]) finishes the job.
  * PeerGather replaces that per-step all_gather by the fused gather of
    csrc/peer_gather.cuh: every rank maps the others' gathered buffers once
    (CUDA IPC, NVLink peer memory) and the solve kernel itself stores its rows
    into all of them -- no collective call inside the step.  Its control_batch /
    control_safe do the same for per-instance controllers and the safe tick of
    B robots on B maps (the validation and fallback kernels store the rows).
Nothing here computes; it only decides who owns what and moves results.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Tuple

import torch
import torch.distributed as dist

from . import capi
from .capi import check


def shard_bounds(total: int, world: int, rank: int) -> Tuple[int, int]:
    """Contiguous block partition of `total` units: the first total % world
    ranks get one extra unit.  Returns [lo, hi)."""
    if world < 1 or not (0 <= rank < world) or total < 0:
        raise ValueError("bad shard request")
    base, extra = divmod(total, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def shard_sizes(total: int, world: int) -> List[int]:
    return [shard_bounds(total, world, r)[1] - shard_bounds(total, world, r)[0] for r in range(world)]


def all_gather_rows(local: torch.Tensor, total: int, group=None) -> torch.Tensor:
    """Gathers the ranks' row blocks (shard_bounds order) into the full
    (total, ...) tensor on every rank.  Uneven shards are padded to the largest
    shard so a single all_gather_into_tensor moves everything."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    sizes = shard_sizes(total, world)
    if local.shape[0] != sizes[rank]:
        raise ValueError(f"rank {rank}: local block has {local.shape[0]} rows, expected {sizes[rank]}")
    if world == 1:
        return local.clone()
    biggest = max(sizes)
    padded = local
    if local.shape[0] != biggest:
        padded = torch.zeros((biggest,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
        padded[: local.shape[0]] = local
    out = torch.empty((world * biggest,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(out, padded.contiguous(), group=group)
    if all(s == biggest for s in sizes):
        return out
    return torch.cat([out[r * biggest: r * biggest + sizes[r]] for r in range(world)], dim=0)


def finish_phik(raw_local: torch.Tensor, nb: int, group=None):
    """raw_local: this rank's (32, 32) un-normalised partial contraction.
    all_reduce(sum), then phi_k[ky*nb + kx] = raw[ky, kx] / raw[0, 0]
    (target.cpp:87: the density is normalised to sum to one).  Returns
    (phi_k (nb*nb,), sum(Phi))."""
    raw = raw_local.clone()
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(raw, op=dist.ReduceOp.SUM, group=group)
    total = raw[0, 0]
    return (raw[:nb, :nb] / total).reshape(-1), total


class ShardedErgodicControl:
    """B instances block-partitioned over the ranks of a process group; each
    rank drives an ErgodicControl for its own block on its own GPU."""

    def __init__(self, make_local, total_batch: int, group=None):
        """make_local(batch) -> ErgodicControl for `batch` instances on this rank's device"""
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.total = total_batch
        self.lo, self.hi = shard_bounds(total_batch, self.world, self.rank)
        self.local = make_local(self.hi - self.lo)

    def local_rows(self, full):
        return full[self.lo: self.hi]

    def control(self, grid, x_local: torch.Tensor, gather: bool = True):
        u0 = self.local.control(grid, x_local)
        if not gather or self.world == 1:
            return u0
        return all_gather_rows(u0, self.total, self.group)


def gather_mode_for_batch(batch: int) -> str:
    """which branch of eb_control_dev_gather publishes a batch of this size"""
    lib = capi.load()
    if lib.eb_gather_fuse_min_batch() <= batch:
        return ("fused into the solve kernel: every warp stores its row into all ranks' gathered buffers "
                "(P2P stores over NVLink peer memory), arrival flags raised by the launch's last warp")
    return ("solve kernel writes u0 locally, peer_publish_kernel on the group's side stream copies the block to all "
            "ranks over NVLink peer memory and raises the arrival flags")


class _DevView:
    """zero-copy torch view of device memory owned by the C library"""

    def __init__(self, ptr: int, shape):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<f8", "data": (int(ptr), False),
                                         "version": 2, "strides": None}


class PeerGather:
    """Fused gather of the first twists over NVLink peer memory for one rank's
    ErgodicControl (include/ergodic_b200.h, eb_peer_group_*).  Collective at
    construction (the ranks exchange CUDA IPC handles with one all_gather of a
    few hundred bytes); afterwards ``control()`` launches the solve kernel, which
    writes this rank's rows into every rank's gathered buffer by itself."""

    def __init__(self, ctl, group=None):
        self._lib = capi.load()
        self.ctl, self.group = ctl, group
        multi = dist.is_initialized() and dist.get_world_size(group) > 1
        self.world = dist.get_world_size(group) if multi else 1
        self.rank = dist.get_rank(group) if multi else 0
        if multi:
            # every rank's row block starts at rank * 3 * batch in every gathered buffer: the batches must be
            # equal, or ranks would store over each other's rows (and past the end of the smaller buffers)
            dev0 = torch.device("cuda", ctl.device)
            mm = torch.tensor([ctl.batch, -ctl.batch], dtype=torch.int64, device=dev0)
            dist.all_reduce(mm, op=dist.ReduceOp.MIN, group=group)
            if int(mm[0].item()) != -int(mm[1].item()):
                raise ValueError(f"PeerGather needs the same batch on every rank (min {int(mm[0].item())}, "
                                 f"max {-int(mm[1].item())}); pad the smaller shards or use all_gather_rows")
        h = C.c_void_p()
        check(self._lib.eb_peer_group_create(ctl.device, self.rank, self.world, 3 * ctl.batch, C.byref(h)))
        self._h = h
        nbytes = self._lib.eb_peer_blob_bytes()
        blob = (C.c_ubyte * nbytes)()
        check(self._lib.eb_peer_group_export(h, blob))
        if multi:
            dev = torch.device("cuda", ctl.device)
            mine = torch.tensor(list(bytes(blob)), dtype=torch.uint8, device=dev)
            allb = torch.empty(self.world * nbytes, dtype=torch.uint8, device=dev)
            dist.all_gather_into_tensor(allb, mine, group=group)
            raw = bytes(allb.cpu().numpy().tobytes())
            buf = (C.c_ubyte * len(raw)).from_buffer_copy(raw)
            st = self._lib.eb_peer_group_connect(h, buf)
            # every rank has mapped every buffer before the first store -- or all give up together
            ok = torch.tensor([1 if st == capi.EB_OK else 0], dtype=torch.int32, device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
            if int(ok.item()) == 0:
                msg = self._lib.eb_last_error().decode(errors="replace") if st != capi.EB_OK else "failed on another rank"
                self._lib.eb_peer_group_destroy(h)
                self._h = None
                raise RuntimeError(f"peer mapping: {msg}")
        else:
            check(self._lib.eb_peer_group_connect(h, None))

    def close(self):
        if getattr(self, "_h", None):
            if dist.is_initialized() and self.world > 1:
                torch.cuda.synchronize(self.ctl.device)
                dist.barrier(group=self.group)  # nobody is still storing into a buffer about to be freed
            self._lib.eb_peer_group_destroy(self._h)
            self._h = None

    def __del__(self):
        # Without the barrier of close() a peer may still be storing into buffers freed here: with more than
        # one rank the group is deliberately leaked (and reported) instead of destroyed behind the peers' backs.
        try:
            if getattr(self, "_h", None):
                if self.world > 1:
                    import warnings
                    warnings.warn("PeerGather dropped without close(): peer-mapped buffers are left allocated",
                                  ResourceWarning)
                else:
                    self._lib.eb_peer_group_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def mode(self) -> str:
        """the publication branch eb_control_dev_gather takes for this controller's batch"""
        return gather_mode_for_batch(self.ctl.batch)

    def fused(self) -> bool:
        """True when a batch of this controller's size publishes from inside the solve kernel"""
        return bool(self._lib.eb_peer_group_fused(self._h, int(self.ctl.batch)))

    @property
    def steps(self) -> int:
        return int(self._lib.eb_peer_group_steps(self._h))

    def control(self, grid, x: torch.Tensor, mem_idx: Optional[torch.Tensor] = None,
                metric: Optional[torch.Tensor] = None, ctl=None) -> int:
        """one control() step of this rank's instances; returns the step number (1-based)
        whose gathered rows ``gathered(step)`` will hold once ``wait(step)`` has passed.
        ``ctl``: another controller of the SAME batch size on this device (the group only fixes the row count)"""
        b = grid.as_tuple() if hasattr(grid, "as_tuple") else tuple(float(v) for v in grid)
        ctl = self.ctl if ctl is None else ctl
        assert ctl.batch == self.ctl.batch and ctl.device == self.ctl.device
        ctl._sync_stream()
        assert x.is_cuda and x.dtype == torch.float64 and x.is_contiguous() and x.numel() == 3 * self.ctl.batch
        idx_p = C.c_void_p(mem_idx.data_ptr()) if mem_idx is not None else None
        met_p = C.c_void_p(metric.data_ptr()) if metric is not None else None
        st = self._lib.eb_control_dev_gather(ctl._h, self._h, *b, C.c_void_p(x.data_ptr()), idx_p, met_p)
        if st == capi.EB_ERR_INVALID_ARGUMENT:
            raise ValueError(self._lib.eb_last_error().decode())
        check(st)
        return self.steps

    def control_wait(self, grid, x: torch.Tensor, mem_idx: Optional[torch.Tensor] = None,
                     metric: Optional[torch.Tensor] = None, ctl=None) -> int:
        """control() + gather + wait as one stream-ordered operation (eb_control_dev_gather_wait): when the work
        enqueued by this call has run, ``gathered(step)`` holds every rank's rows.  Returns the step number."""
        b = grid.as_tuple() if hasattr(grid, "as_tuple") else tuple(float(v) for v in grid)
        ctl = self.ctl if ctl is None else ctl
        assert ctl.batch == self.ctl.batch and ctl.device == self.ctl.device
        ctl._sync_stream()
        assert x.is_cuda and x.dtype == torch.float64 and x.is_contiguous() and x.numel() == 3 * self.ctl.batch
        idx_p = C.c_void_p(mem_idx.data_ptr()) if mem_idx is not None else None
        met_p = C.c_void_p(metric.data_ptr()) if metric is not None else None
        st = self._lib.eb_control_dev_gather_wait(ctl._h, self._h, *b, C.c_void_p(x.data_ptr()), idx_p, met_p)
        if st == capi.EB_ERR_INVALID_ARGUMENT:
            raise ValueError(self._lib.eb_last_error().decode())
        check(st)
        return self.steps

    def _ctl(self, ctl):
        ctl = self.ctl if ctl is None else ctl
        assert ctl.batch == self.ctl.batch and ctl.device == self.ctl.device
        return ctl

    def _raise(self, st):
        if st == capi.EB_ERR_INVALID_ARGUMENT:
            raise ValueError(self._lib.eb_last_error().decode())
        check(st)

    def _batch(self, fn, bounds, x, mem_idx, metric, ctl) -> int:
        ctl = self._ctl(ctl)
        if not (torch.is_tensor(x) and x.is_cuda and x.dtype == torch.float64 and x.is_contiguous()
                and x.numel() == 3 * ctl.batch):
            raise ValueError(f"x must be a contiguous ({ctl.batch}, 3) float64 CUDA tensor")
        b = ctl._dev_tick_args(bounds, mem_idx, metric)
        ctl._sync_stream()
        P = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        self._raise(fn(ctl._h, self._h, P(b), P(x), P(mem_idx), P(metric)))
        return self.steps

    def control_batch(self, bounds, x: torch.Tensor, mem_idx: Optional[torch.Tensor] = None,
                      metric: Optional[torch.Tensor] = None, ctl=None) -> int:
        """ErgodicControl.control(bounds, x) of a per-instance controller (``bounds`` (B, 4) or None: the frames of
        the last configure) whose twists land in every rank's gathered buffer (eb_control_batch_dev_gather); returns
        the step number, whose rows ``gathered(step)`` holds once ``wait(step)`` has passed.  CUDA tensors only."""
        return self._batch(self._lib.eb_control_batch_dev_gather, bounds, x, mem_idx, metric, ctl)

    def control_batch_wait(self, bounds, x: torch.Tensor, mem_idx: Optional[torch.Tensor] = None,
                           metric: Optional[torch.Tensor] = None, ctl=None) -> int:
        """control_batch + wait as one stream-ordered operation (eb_control_batch_dev_gather_wait)"""
        return self._batch(self._lib.eb_control_batch_dev_gather_wait, bounds, x, mem_idx, metric, ctl)

    def _safe(self, fn, grids, dwa, x, vb, val_dt, val_horizon, bounds, mem_idx, metric, collision, ctl):
        ctl = self._ctl(ctl)
        if not torch.is_tensor(x) or not x.is_cuda:
            raise ValueError("PeerGather.control_safe takes CUDA tensors")
        x, vb = ctl._safe_rows(grids, x, vb, True)
        b = ctl._dev_tick_args(bounds, mem_idx, metric)
        col = dwa.collision if collision is None else collision
        branch = torch.empty(ctl.batch, dtype=torch.int32, device=x.device)
        ctl._sync_stream()
        grids._stream()
        P = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        self._raise(fn(ctl._h, self._h, grids._h, C.byref(col.cfg), C.byref(dwa.cfg), float(val_dt), float(val_horizon),
                       P(b), P(x), P(mem_idx), P(vb), P(branch), P(metric)))
        return self.steps, branch

    def control_safe(self, grids, dwa, x: torch.Tensor, vb: torch.Tensor, val_dt: float, val_horizon: float,
                     bounds=None, mem_idx: Optional[torch.Tensor] = None, metric: Optional[torch.Tensor] = None,
                     collision=None, ctl=None):
        """ErgodicControl.control_safe on the device path whose final twists u land in every rank's gathered buffer
        (eb_control_safe_batch_dev_gather).  Returns (step, branch): ``gathered(step)`` holds every rank's u once
        ``wait(step)`` has passed; branch (B,) int32 stays local."""
        return self._safe(self._lib.eb_control_safe_batch_dev_gather, grids, dwa, x, vb, val_dt, val_horizon, bounds,
                          mem_idx, metric, collision, ctl)

    def control_safe_wait(self, grids, dwa, x: torch.Tensor, vb: torch.Tensor, val_dt: float, val_horizon: float,
                          bounds=None, mem_idx: Optional[torch.Tensor] = None, metric: Optional[torch.Tensor] = None,
                          collision=None, ctl=None):
        """control_safe + wait as one stream-ordered operation (eb_control_safe_batch_dev_gather_wait)"""
        return self._safe(self._lib.eb_control_safe_batch_dev_gather_wait, grids, dwa, x, vb, val_dt, val_horizon,
                          bounds, mem_idx, metric, collision, ctl)

    def wait(self, step: Optional[int] = None) -> None:
        """enqueue (on the current stream) a wait until every rank's rows of ``step`` are here"""
        self.ctl._sync_stream()
        check(self._lib.eb_peer_group_wait(self._h, self.ctl._h, int(self.steps if step is None else step)))

    def gathered(self, step: Optional[int] = None) -> torch.Tensor:
        """this rank's copy of all ranks' first twists of ``step``: (world * batch, 3), zero-copy"""
        step = self.steps if step is None else step
        ptr = self._lib.eb_peer_gathered_dev(self._h, int(step))
        return torch.as_tensor(_DevView(ptr, (self.world * self.ctl.batch, 3)), device=torch.device("cuda", self.ctl.device))


class PhikAllReduce:
    """Row-sharded phi_k with the cross-GPU reduction fused into the tile kernel (include/ergodic_b200.h,
    eb_phik_peer_*): every rank contracts its row block and the last CTA of its kernel exchanges the raw 32 x 32
    blocks over NVLink peer memory -- one kernel launch per rank and step, no NCCL call on the data path.
    Collective at construction (IPC handles through one all_gather) and in ``execute`` (every rank calls it)."""

    def __init__(self, plan, group=None):
        self._lib = capi.load()
        self.plan, self.group = plan, group
        multi = dist.is_initialized() and dist.get_world_size(group) > 1
        self.world = dist.get_world_size(group) if multi else 1
        self.rank = dist.get_rank(group) if multi else 0
        h = C.c_void_p()
        check(self._lib.eb_phik_peer_create(plan.device, self.rank, self.world, C.byref(h)))
        self._h = h
        nbytes = self._lib.eb_phik_peer_blob_bytes()
        blob = (C.c_ubyte * nbytes)()
        check(self._lib.eb_phik_peer_export(h, blob))
        if multi:
            dev = torch.device("cuda", plan.device)
            mine = torch.tensor(list(bytes(blob)), dtype=torch.uint8, device=dev)
            allb = torch.empty(self.world * nbytes, dtype=torch.uint8, device=dev)
            dist.all_gather_into_tensor(allb, mine, group=group)
            raw = bytes(allb.cpu().numpy().tobytes())
            buf = (C.c_ubyte * len(raw)).from_buffer_copy(raw)
            st = self._lib.eb_phik_peer_connect(h, buf)
            ok = torch.tensor([1 if st == capi.EB_OK else 0], dtype=torch.int32, device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
            if int(ok.item()) == 0:
                msg = self._lib.eb_last_error().decode(errors="replace") if st != capi.EB_OK else "failed on another rank"
                self._lib.eb_phik_peer_destroy(h)
                self._h = None
                raise RuntimeError(f"peer mapping: {msg}")
        else:
            check(self._lib.eb_phik_peer_connect(h, None))

    def execute(self, phi: torch.Tensor, phik: Optional[torch.Tensor] = None, phi_sum: Optional[torch.Tensor] = None):
        """phi: this rank's (rows, nx) block; returns the (nb * nb,) coefficients of the WHOLE grid (every rank alike)"""
        s = torch.cuda.current_stream(self.plan.device).cuda_stream
        check(self._lib.eb_phik_plan_set_stream(self.plan._h, C.c_void_p(s)))
        assert phi.is_cuda and phi.dtype == torch.float64 and phi.is_contiguous() and phi.numel() == self.plan.nx * self.plan.ny
        if phik is None:
            phik = torch.empty(self.plan.nb * self.plan.nb, dtype=torch.float64, device=phi.device)
        sp = C.c_void_p(phi_sum.data_ptr()) if phi_sum is not None else None
        check(self._lib.eb_phik_execute_allreduce_dev(self.plan._h, self._h, C.c_void_p(phi.data_ptr()),
                                                      C.c_void_p(phik.data_ptr()), sp))
        return phik

    def close(self):
        if getattr(self, "_h", None):
            if dist.is_initialized() and self.world > 1:
                torch.cuda.synchronize(self.plan.device)
                dist.barrier(group=self.group)  # nobody is still storing into a buffer about to be freed
            self._lib.eb_phik_peer_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            if getattr(self, "_h", None) and self.world == 1:
                self._lib.eb_phik_peer_destroy(self._h)
                self._h = None
        except Exception:
            pass

// safe_control.cuh -- the safe control tick of B robots on B maps (eb_control_safe_batch_*), sm_100a.
//
// The reference's loop arbitrates, per robot, between the ergodic twist and the safety planner: control(), then
// validate_control on the returned twist (exploration.hpp:238); only when that twist collides, optTraj() and
// DynamicWindow::control(grid, pose, vb, optTraj, ec_dt) (exploration.hpp:247), and a zero twist when the window
// finds nothing.  After the solve launch, two kernels do the rest without the host knowing which robots failed:
//  * validate_compact_kernel: one thread per robot runs validate_control_ok on its own map (the code of
//    validate_control_kernel<true>), keeps the solve's twist for a valid robot (branch 0) and appends a failing
//    robot's index to a device list through a warp-aggregated atomic counter.  The list's order does not matter:
//    every robot's result depends on that robot alone.
//  * dwa_fallback_kernel: one CTA per listed robot, on a grid of at most the resident CTAs that strides over the
//    list, whose length it reads from device memory.  Warp 0 rolls the robot's control signal out into shared memory
//    with rollout_kernel's code (the trajectory eb_opt_traj_dev would return, bit for bit; the B x N x 3 optTraj is
//    never written), then every thread evaluates candidate twists of the window, one each (striding past the block),
//    with dwa_objective on the robot's map against that trajectory.  A block arg-min with ties to the lower candidate
//    is the warp kernel's first strict minimum in loop order; the window, the candidates and found come from the
//    helpers dwa_control_kernel uses.
// CTA per robot rather than dwa_control_kernel's warp per robot: when few robots fail, the call's latency is one
// robot's window, and one candidate per thread evaluates a 3 x 8 x 5 window in one round of rollouts instead of four.
//
// Multi-GPU (eb_control_safe_batch_dev_gather[_wait], PUBLISH = true): a robot's final twist is known only in one of the
// two kernels, so each of them stores the rows it decides straight into every rank's gathered buffer over peer memory
// (peer_gather.cuh's layout and reuse guard): the validation kernel the rows of the valid robots -- they travel while
// the window runs -- and the fallback the rows of the listed ones.  The fallback's last CTA raises this rank's arrival
// flag on every peer and, in the _wait form, waits for every rank's.  The PUBLISH = false instantiations are the
// single-GPU tick.
#pragma once

#include <type_traits>

#include "collision_kernels.cuh"
#include "peer_gather.cuh"
#include "solve_kernel.cuh"

namespace eb
{
constexpr int kSafeThreads = 128;

struct SafeParams
{
  int* list;         // [B] failing robots, *count of them
  int* count;
  const double* ut;  // [B][N][3] ut_ after the solve
  double dt;         // the controller's time step (optTraj)
  int N;
  double* u;         // [B][3]
  int* branch;       // [B]
  int* fault;        // SimpleCart twist with a y-velocity (rollout_kernel)
};

// the safe tick whose twists also go to every rank of a peer group
struct SafePublishParams : SafeParams
{
  PublishParams peer;     // dst / flag / flag_value / my_flags / need / done_counter of the step (src, elems unused)
  unsigned int arrivals;  // what counts out on peer.done_counter: every validation warp, then every fallback CTA
  int wait;               // 1: the fallback's last CTA also waits for every rank's flag (the _wait form)
};

template <bool PUBLISH>
using SafeArgs = std::conditional_t<PUBLISH, SafePublishParams, SafeParams>;

// peer_gather.cuh's reuse guard, by one warp before it stores into this step's buffer: every rank has finished the step
// that last read it
__device__ __forceinline__ void peer_reuse_guard(const PublishParams& pp, const int lane)
{
  if (lane < pp.n_peer)
    while (*(const volatile unsigned long long*)(pp.my_flags + lane) < pp.need) __nanosleep(100);
  __syncwarp();
}

// one robot's final twist into its row of every rank's gathered buffer
__device__ __forceinline__ void peer_store_row(const PublishParams& pp, const size_t inst, const double u0, const double u1,
                                               const double u2)
{
#pragma unroll
  for (int q = 0; q < kPublishPeers; q++)
    if (q < pp.n_peer)
    {
      pp.dst[q][inst * 3 + 0] = u0;
      pp.dst[q][inst * 3 + 1] = u1;
      pp.dst[q][inst * 3 + 2] = u2;
    }
}

// p.x0 = the poses, p.u = the solve's twists: branch 0 for a valid twist, else the robot goes on the list
template <bool PUBLISH>
__global__ void __launch_bounds__(128) validate_compact_kernel(const CollisionParams p, const MapSet m, const SafeArgs<PUBLISH> s)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const bool fails = i < p.B && !validate_control_ok(on_map(p, m, i), i);
  if (i < p.B && !fails) s.branch[i] = 0;
  if constexpr (PUBLISH)
  {
    // A valid robot's twist is final: its row goes to every rank now, while the window of the failing ones runs.
    // Then every warp releases its rows at GPU scope into the arrival counter; the fallback's last CTA takes them up
    // (see there), so no warp here pays for a system-scope fence.
    const int lane = threadIdx.x & 31;
    peer_reuse_guard(s.peer, lane);
    if (i < p.B && !fails) peer_store_row(s.peer, i, p.u[(size_t)i * 3 + 0], p.u[(size_t)i * 3 + 1], p.u[(size_t)i * 3 + 2]);
    __threadfence();
    __syncwarp();
    if (lane == 0) atomicAdd(s.peer.done_counter, 1u);
  }
  const unsigned int mask = __ballot_sync(kFull, fails);
  if (mask == 0) return;
  const int lane = threadIdx.x & 31, leader = __ffs(mask) - 1;
  int base = 0;
  if (lane == leader) base = atomicAdd(s.count, __popc(mask));
  base = __shfl_sync(kFull, base, leader);
  if (fails) s.list[base + __popc(mask & ((1u << lane) - 1u))] = i;
}

// robot i of the list: p.x0 the poses, p.vb the body twists, p.ncols = N and p.tf = N * dt (the optTraj reference)
template <int MODEL, bool PUBLISH>
__global__ void __launch_bounds__(kSafeThreads) dwa_fallback_kernel(const DwaParams p, const MapSet m, const SafeArgs<PUBLISH> s)
{
  extern __shared__ double s_xt[];  // [N][3]: the robot's optTraj()
  __shared__ double w_best[kSafeThreads / 32];
  __shared__ unsigned int w_c[kSafeThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n = *s.count;
  const unsigned int total = p.n[0] * p.n[1] * p.n[2];
  for (int li = blockIdx.x; li < n; li += gridDim.x)
  {
    const int inst = s.list[li];
    const double x = p.x0[(size_t)inst * 3 + 0], y = p.x0[(size_t)inst * 3 + 1], th = p.x0[(size_t)inst * 3 + 2];
    if (warp == 0)
    {  // rollout_kernel for this robot, from pose_ = x
      const double* u = s.ut + (size_t)inst * s.N * 3;
      RolloutCarry cy;
      cy.x = x;
      cy.y = y;
      cy.th = th;
      fast_sincos(cy.th, &cy.sth, &cy.cth);
      for (int base = 0; base < s.N; base += 32)
      {
        const int i = base + lane;
        const bool valid = i < s.N;
        double u0 = 0.0, u1 = 0.0, u2 = 0.0;
        if (valid)
        {
          u0 = u[i * 3 + 0];
          u1 = u[i * 3 + 1];
          u2 = u[i * 3 + 2];
        }
        if (MODEL == kModelSimpleCart && !(fabs(u1 - 0.0) < 1.0e-12)) atomicOr(s.fault, 1);
        double xo, yo, tho, ce, se;
        rollout_round<MODEL>(s.dt, valid, lane, u0, u1, u2, cy, xo, yo, tho, ce, se);
        if (valid)
        {
          s_xt[i * 3 + 0] = xo;
          s_xt[i * 3 + 1] = yo;
          s_xt[i * 3 + 2] = normalize_angle_pi(tho);
        }
      }
    }
    __syncthreads();
    const CollisionParams col = on_map(p.col, m, inst);
    double lower[3], delta[3];
    dwa_window(p, inst, lower, delta);
    double best = kDblMax;
    unsigned int best_c = 0xffffffffu;
    for (unsigned int c = threadIdx.x; c < total; c += kSafeThreads)
    {
      double u0, u1, u2;
      dwa_twist(p, lower, delta, c, u0, u1, u2);
      const double cost = dwa_objective(p, col, s_xt, x, y, th, u0, u1, u2, nullptr);
      if (cost < best)
      {
        best = cost;
        best_c = c;
      }
    }
    dwa_argmin_warp(best, best_c);
    if (lane == 0)
    {
      w_best[warp] = best;
      w_c[warp] = best_c;
    }
    __syncthreads();
    if (warp == 0)
    {
      best = lane < kSafeThreads / 32 ? w_best[lane] : kDblMax;
      best_c = lane < kSafeThreads / 32 ? w_c[lane] : 0xffffffffu;
      dwa_argmin_warp(best, best_c);
      if constexpr (PUBLISH) peer_reuse_guard(s.peer, lane);
      if (lane == 0)
      {
        double u0 = 0.0, u1 = 0.0, u2 = 0.0;  // nothing found: the zero twist
        const int found = dwa_found(best);
        if (found) dwa_twist(p, lower, delta, best_c, u0, u1, u2);
        s.u[(size_t)inst * 3 + 0] = u0;
        s.u[(size_t)inst * 3 + 1] = u1;
        s.u[(size_t)inst * 3 + 2] = u2;
        s.branch[inst] = found ? 1 : 2;
        if constexpr (PUBLISH) peer_store_row(s.peer, inst, u0, u1, u2);
      }
    }
    __syncthreads();  // s_xt and the warp minima are the next robot's
  }
  if constexpr (PUBLISH)
  {
    // Every CTA counts out, also one whose stride found no robot: the list's length is known only on the device.
    // Memory ordering, as in publish_first_twist (solve_kernel.cuh): thread 0 stored this CTA's rows; its GPU-scope
    // fence and counter increment release them, and every validation warp did the same for its rows before.  The
    // increments are atomic RMWs on one counter of this device, so the last CTA's increment reads a value that
    // follows all of them, synchronises with each of those releases at GPU scope, and its system-scope fence is
    // cumulative over every row they released -- of both kernels.  The argument needs no ordering from the kernel
    // boundary: the PTX memory model says nothing about stream order, and a peer reading the flag is not on this stream.
    __shared__ unsigned int s_last;
    if (threadIdx.x == 0)
    {
      __threadfence();
      const unsigned int prev = atomicAdd(s.peer.done_counter, 1u);
      s_last = prev == s.arrivals - 1u ? 1u : 0u;
      if (s_last)
      {
        *s.peer.done_counter = 0u;  // ready for the next step on this stream
        __threadfence_system();
#pragma unroll
        for (int q = 0; q < kPublishPeers; q++)
          if (q < s.peer.n_peer) *(volatile unsigned long long*)s.peer.flag[q] = s.peer.flag_value;
      }
    }
    __syncthreads();
    if (s.wait && s_last)
    {  // peer_publish_wait_kernel's wait: every rank's rows of this step are here for what follows on the stream
      if (threadIdx.x < s.peer.n_peer)
        while (*(const volatile unsigned long long*)(s.peer.my_flags + threadIdx.x) < s.peer.flag_value) __nanosleep(64);
      __syncthreads();
      __threadfence_system();  // acquire
    }
  }
}
}  // namespace eb

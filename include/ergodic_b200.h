/*
 * ergodic_b200.h -- C ABI of the B200-native ergodic-control hot path.
 *
 * This is the drop-in boundary for the reference's (bostoncleek/
 * ergodic_exploration) receding-horizon controller step
 * ErgodicControl<ModelT>::control() and the phi_k target-coefficient
 * contraction it depends on.  The reference has no FFI of its own: its
 * boundary is the C++ class API (ergodic_control.hpp:72-185).  The
 * header-only adapter include/ergodic_exploration_b200/ergodic_control.hpp
 * re-exposes that class API (Armadillo in, Armadillo out) on top of the
 * entry points below; INTEGRATION.md shows the binding.
 *
 * Conventions
 *  - one handle = B independent controllers ("instances") on ONE CUDA device
 *    and one CUDA stream.  B = 1 is the reference's single-robot case.
 *  - all matrices are column-major doubles, byte-identical to
 *    arma::mat::memptr(): a 3xN matrix is N consecutive (x, y, theta)
 *    triples; batched buffers are B such matrices back to back
 *    (instance-major).
 *  - `_host` entry points take host pointers, copy in/out and synchronise;
 *    `_dev` entry points take device pointers, enqueue on the handle's
 *    stream and return immediately.
 *  - every call returns an eb_status; no exception crosses the ABI.
 *    eb_last_error() returns the message of the last failure.  The adapter
 *    rethrows the reference's exception types (std::invalid_argument, ...).
 *  - there is NO CPU fallback: without a CUDA device every call fails with
 *    EB_ERR_NO_DEVICE / EB_ERR_CUDA.
 *
 * Citations are file:line in the reference tree.
 */
#ifndef ERGODIC_B200_H
#define ERGODIC_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EB_ABI_VERSION 1

typedef enum eb_status {
  EB_OK = 0,
  EB_ERR_INVALID_ARGUMENT = 1, /* reference: std::invalid_argument */
  EB_ERR_OUT_OF_RANGE = 2,     /* reference: std::out_of_range (buffer.cpp:84,103) */
  EB_ERR_CUDA = 3,             /* CUDA runtime failure (message has the cudaError) */
  EB_ERR_NO_DEVICE = 4,        /* no usable CUDA device: there is no CPU path */
  EB_ERR_UNSUPPORTED = 5
} eb_status;

/* models the controller can run (SURVEY App. B-1: 3-twist models only) */
typedef enum eb_model {
  EB_MODEL_SIMPLE_CART = 0, /* models/cart.hpp:152-206 */
  EB_MODEL_OMNI = 1,        /* models/omni.hpp:164-215 */
  EB_MODEL_CART = 2,        /* models/cart.hpp:60-145  -- forward rollout / model evaluation only (eb_rk4_solve_*) */
  EB_MODEL_MECANUM = 3      /* models/omni.hpp:59-157  -- forward rollout / model evaluation only */
} eb_model;

/* Constructor arguments of ErgodicControl (ergodic_control.hpp:90-94) plus
 * the two constants the reference hard-codes in gradBarrier (:457-458). */
/* num_basis: 1..EB_MAX_NUM_BASIS (the reference accepts any count, basis.cpp:48-77).  Up to 32 the coefficient block of
 * an instance lives in the registers of one warp (the tuned kernels); 33..128 run a CTA per instance with the block
 * spread over its threads (csrc/solve_kernel_big.cuh) and the phi_k contraction over blocks of 32 orders.  Beyond 128
 * the cosine tables of 32 states no longer fit shared memory: eb_create returns EB_ERR_INVALID_ARGUMENT. */
#define EB_MAX_NUM_BASIS 128
typedef struct eb_config {
  int model;            /* eb_model */
  int batch;            /* B >= 1 independent instances */
  int device;           /* CUDA device ordinal */
  double dt;            /* time step in integration */
  double horizon;       /* control horizon; steps = (unsigned)|horizon/dt| (:199) */
  double resolution;    /* target grid resolution (m) */
  double expl_weight;   /* exploration_weight */
  unsigned num_basis;   /* cosine bases per dimension, 1..EB_MAX_NUM_BASIS */
  unsigned buffer_size; /* max past states kept per instance (ReplayBuffer) */
  unsigned batch_size;  /* past states sampled per control() */
  double Rinv[9];       /* 3x3 column-major */
  double umin[3];
  double umax[3];
  double barrier_weight; /* 25.0 in the reference (:457) */
  double barrier_eps;    /* 0.05 in the reference (:458) */
  unsigned long long seed; /* seed of the on-device replay sampler */
} eb_config;

typedef struct eb_controller eb_controller;

/* fills cfg with the reference defaults (explore_omni.yaml / node mains) */
void eb_config_defaults(eb_config *cfg, int model);

int eb_abi_version(void);
const char *eb_last_error(void);

/* number of CUDA devices visible (0 when none; never fails) */
int eb_device_count(void);

/* ---- lifetime (ctor ergodic_control.hpp:188-222) ------------------------ */
/* EB_ERR_INVALID_ARGUMENT when steps == 1 (:212-216). */
eb_status eb_create(const eb_config *cfg, eb_controller **out);
/* deep copy, including device state (the reference object is copied by
 * value into Exploration, exploration.hpp:137-138) */
eb_status eb_clone(const eb_controller *src, eb_controller **out);
void eb_destroy(eb_controller *c);
/* use the caller's CUDA stream (cudaStream_t) for all subsequent work */
eb_status eb_set_stream(eb_controller *c, void *cuda_stream);

int eb_steps(const eb_controller *c);      /* N */
int eb_num_coeff(const eb_controller *c);  /* K = num_basis^2 */
int eb_batch(const eb_controller *c);      /* B */
double eb_time_step(const eb_controller *c); /* timeStep() :351-354 */
long long eb_memory_size(const eb_controller *c); /* stored past states per instance */

/* ---- target (setTarget :357-360, configTarget :363-416) ----------------- */
/* mu, sigma: 2 x n column-major (host) */
eb_status eb_set_target_gaussians(eb_controller *c, int n, const double *mu, const double *sigma);
/* Rebuilds phi_k on the device when the map extent changed by >= 1e-12
 * (:374); always records the map origin.  *rebuilt (may be NULL) = 1 if so. */
eb_status eb_config_target(eb_controller *c, double xmin, double xmax, double ymin, double ymax,
                           int *rebuilt);
/* direct access to phi_k (K doubles, host) and the Fourier domain lengths */
eb_status eb_set_phik(eb_controller *c, const double *phik, double lx, double ly);
eb_status eb_get_phik(const eb_controller *c, double *phik, double *lx, double *ly);

/* ---- replay memory (addStateMemory :345-348, buffer.cpp:54-62) ---------- */
/* x: 3 x B.  Silently dropped when buffer_size states are stored.
 * Next to the stored rows the library keeps 16 bytes per state and instance with the two Fourier-frame cosines the
 * solve kernels need from a sampled state (re-derived when the map origin / extent changes; results are bit-identical
 * with or without it; environment EB_REPLAY_COS=0 switches it off). */
/* room for `count` stored states up front (capped at buffer_size): keeps allocations out of the control loop */
eb_status eb_reserve_state_memory(eb_controller *c, long long count);
eb_status eb_add_state_memory_host(eb_controller *c, const double *x);
eb_status eb_add_state_memory_dev(eb_controller *c, const double *x_dev);

/* ---- control() (:225-311), batched --------------------------------------
 * x       3 x B current states (map frame)
 * mem_idx batch_size x B int32 indices of the sampled past states, used only
 *         when more than batch_size states are stored (replaces arma::randi,
 *         buffer.cpp:98).  NULL -> indices are drawn on the device with a
 *         counter-based generator (seed, call count, instance) and can be
 *         read back with eb_get_last_mem_idx().
 * u0      3 x B first twist of the updated control signal (ut_.col(0))
 * metric  B ergodic metric sum_k lamda_k (c_k - phi_k)^2, may be NULL
 * EB_ERR_INVALID_ARGUMENT if SimpleCart is given |u(1)| >= 1e-12
 * (cart.hpp:167-170) -- detected on the device, reported by the _host call
 * and by eb_check_status() for _dev calls. */
eb_status eb_control_host(eb_controller *c, double xmin, double xmax, double ymin, double ymax,
                          const double *x, const int *mem_idx, double *u0, double *metric);
eb_status eb_control_dev(eb_controller *c, double xmin, double xmax, double ymin, double ymax,
                         const double *x_dev, const int *mem_idx_dev, double *u0_dev,
                         double *metric_dev);
/* synchronises the stream and reports device-side faults of earlier _dev calls */
eb_status eb_check_status(eb_controller *c);

/* ---- optTraj() (:314-317) ------------------------------------------------ */
/* xt: 3 x N x B, forward rollout of the current ut_ from the last pose */
eb_status eb_opt_traj_host(eb_controller *c, double *xt);
eb_status eb_opt_traj_dev(eb_controller *c, double *xt_dev);

/* ---- controller state (checkpoint / teacher forcing) -------------------- */
eb_status eb_get_ut(const eb_controller *c, double *ut); /* 3 x N x B host */
eb_status eb_set_ut(eb_controller *c, const double *ut);
eb_status eb_get_ck(const eb_controller *c, double *ck); /* K x B host, last control() */
eb_status eb_get_last_mem_idx(const eb_controller *c, int *mem_idx, int *count); /* batch_size x B */
/* device pointers to the resident state (valid for the handle's lifetime) */
double *eb_ut_dev(eb_controller *c);
double *eb_ck_dev(eb_controller *c);
/* c_k of every instance is a by-product of control() (not part of the reference's
 * return value); keep = 0 skips its K x B store (default: kept) */
eb_status eb_set_keep_ck(eb_controller *c, int keep);

/* number of kernels this handle has launched so far */
long long eb_launch_count(const eb_controller *c);

/* ---- stateless phi_k (Target::fill normalisation target.cpp:87 +
 *      Basis::spatialCoeff basis.cpp:122-133) --------------------------------
 * phi: ny x nx dense density, x fastest (index i*nx + j), un-normalised, on the
 * configTarget grid (x_j, y_i accumulated by += resolution from 0,
 * ergodic_control.hpp:391-408).  Output phik[ky*nb + kx] = (C_y^T phi C_x) /
 * sum(phi), K doubles; *phi_sum = sum(phi).
 *
 * A plan owns the cosine tables for one (nx, ny, resolution, lx, ly, nb) and
 * the scratch buffers; execute runs the contraction only. */
typedef struct eb_phik_plan eb_phik_plan;
eb_status eb_phik_plan_create(int device, int nx, int ny, double resolution, double lx, double ly,
                              int nb, eb_phik_plan **out);
/* Row-sharded variant for multi-GPU (SURVEY §8e): the plan covers rows
 * [row_begin, row_begin + row_count) of an ny_total-row grid; phi passed to
 * execute holds only those rows.  Combine shards with eb_phik_execute_raw_dev
 * + one all-reduce(sum) of the 1024 raw values, then divide by raw[0]. */
eb_status eb_phik_plan_create_rows(int device, int nx, int ny_total, int row_begin, int row_count,
                                   double resolution, double lx, double ly, int nb, eb_phik_plan **out);
/* as eb_phik_plan_create_rows with the grid's first sample point at (x_first, y_first) instead of (0, 0): the
 * coordinates are x_first + accumulated j * resolution (cell CENTRES of an occupancy grid: x_first = resolution / 2) */
eb_status eb_phik_plan_create_ex(int device, int nx, int ny_total, int row_begin, int row_count, double resolution,
                                 double lx, double ly, int nb, double x_first, double y_first, eb_phik_plan **out);
void eb_phik_plan_destroy(eb_phik_plan *p);
eb_status eb_phik_plan_set_stream(eb_phik_plan *p, void *cuda_stream);
/* algo: 0 = auto, 1 = simple (any shape), 2 = DMMA tiles (TMA-fed; mirror-folded when the
 * grid's cosine table is symmetric, see eb_phik_plan_fold), 3 = DMMA tiles without the fold */
eb_status eb_phik_plan_set_algo(eb_phik_plan *p, int algo);
/* fold = 1 when the plan's grid allows the mirror fold (x_j + x_{nx-1-j} == lx to rounding, so
 * cos(k pi x / lx) is (-1)^k-symmetric and half the contraction suffices); deviation = the
 * measured asymmetry of the table, which bounds the fold's coefficient error (taken iff <= 1e-10) */
eb_status eb_phik_plan_fold(const eb_phik_plan *p, int *fold, double *deviation);
eb_status eb_phik_execute_dev(eb_phik_plan *p, const double *phi_dev, double *phik_dev,
                              double *phi_sum_dev);
eb_status eb_phik_execute_host(eb_phik_plan *p, const double *phi, double *phik, double *phi_sum);
/* un-normalised contraction: raw[ky*ld + kx] = (C_y^T phi C_x)[ky][kx], ld * ld doubles with ld = 32 for nb <= 32
 * (1024 doubles) and nb rounded up to a multiple of 32 beyond (entries with ky or kx >= nb are 0); raw[0] = sum(phi) */
eb_status eb_phik_execute_raw_dev(eb_phik_plan *p, const double *phi_dev, double *raw_dev);
/* one-shot convenience (host buffers): plan + execute + destroy */
eb_status eb_phik_from_grid_host(int device, const double *phi, int nx, int ny, double resolution,
                                 double lx, double ly, int nb, double *phik, double *phi_sum);
long long eb_phik_launch_count(const eb_phik_plan *p);

/* ---- stateless Basis / Target entry points on ARBITRARY points ----------
 * (the public methods of the reference's Basis and Target classes; host
 * buffers, computed on the device, synchronous)
 * eb_basis_traj_coeff_host   Basis::trajCoeff (basis.cpp:109-120); xt is ld x ncols
 *                            (ld = 2 or 3, only rows 0,1 are read).  With
 *                            ncols = 1 this is Basis::fourierBasis (:79-89).
 * eb_basis_grad_host         Basis::gradFourierBasis (:91-107); dfk is 2 x K
 * eb_basis_spatial_coeff_host Basis::spatialCoeff (:122-133); phi_grid is 2 x G
 * eb_target_fill_host        Target::fill (target.cpp:78-89): values at the
 *                            points of phi_grid, normalised to sum to 1 */
eb_status eb_basis_traj_coeff_host(int device, double lx, double ly, int nb, const double *xt, int ld,
                                   int ncols, double *ck);
eb_status eb_basis_grad_host(int device, double lx, double ly, int nb, const double *x, double *dfk);
eb_status eb_basis_spatial_coeff_host(int device, double lx, double ly, int nb, const double *phi_vals,
                                      const double *phi_grid, long long G, double *phik);
eb_status eb_target_fill_host(int device, int ng, const double *mu, const double *sigma,
                              const double *trans, const double *phi_grid, long long G, double *phi_vals);

/* ---- fused multi-GPU gather of the first twists (SURVEY.md section 8e) --------
 * One process per GPU; the instances are block-partitioned and the only exchange of
 * a control() step is the gather of u0.  Instead of a collective call per step, every
 * rank maps every other rank's gathered buffer once (CUDA IPC over NVLink / NVSwitch
 * peer memory) and the solve kernel stores its rows into all of them directly.
 *   create -> export blob -> exchange the blobs of all ranks (e.g. one all_gather of
 *   eb_peer_blob_bytes() bytes at start-up) -> connect -> eb_control_dev_gather per step.
 * eb_peer_group_wait enqueues a wait until all ranks' rows of a step have arrived here;
 * eb_peer_gathered_dev is this rank's copy, [world][batch][3] doubles.  Four buffers rotate by
 * step: read a step's rows (after its wait) before launching the next step on the same stream,
 * and the kernel itself holds back its stores until every rank is past the reads of the step
 * whose buffer it is about to reuse -- no per-step wait is needed between launches. */
typedef struct eb_peer_group eb_peer_group;
int eb_peer_blob_bytes(void);
eb_status eb_peer_group_create(int device, int rank, int world, long long elems_per_rank /* 3 * batch */,
                               eb_peer_group **out);
eb_status eb_peer_group_export(eb_peer_group *g, unsigned char *blob);
eb_status eb_peer_group_connect(eb_peer_group *g, const unsigned char *blobs /* world blobs, rank order */);
void eb_peer_group_destroy(eb_peer_group *g);
eb_status eb_control_dev_gather(eb_controller *c, eb_peer_group *g, double xmin, double xmax, double ymin,
                                double ymax, const double *x_dev, const int *mem_idx_dev, double *metric_dev);
eb_status eb_peer_group_wait(eb_peer_group *g, eb_controller *c, unsigned long long step);
/* control() + gather + wait as ONE stream-ordered operation on the controller's stream: afterwards the rows of every rank
 * for this step are in eb_peer_gathered_dev(g, eb_peer_group_steps(g)).  The form a closed loop wants (every tick needs
 * the complete step); single-wave batches publish and wait in one kernel right behind the solve kernel. */
eb_status eb_control_dev_gather_wait(eb_controller *c, eb_peer_group *g, double xmin, double xmax, double ymin,
                                     double ymax, const double *x_dev, const int *mem_idx_dev, double *metric_dev);
double *eb_peer_gathered_dev(eb_peer_group *g, unsigned long long step);
unsigned long long eb_peer_group_steps(const eb_peer_group *g);
/* 1: a batch of this size publishes from inside the solve kernel, 0: from the group's side stream */
int eb_peer_group_fused(const eb_peer_group *g, int batch);
int eb_gather_fuse_min_batch(void); /* the threshold behind eb_peer_group_fused (EB_GATHER_FUSE_MIN_BATCH overrides) */
/* NOTE (equal shards): every rank's row block starts at rank * elems_per_rank in every gathered buffer, so all
 * ranks of a group MUST be created with the same elems_per_rank (= 3 * batch); uneven shards have to be padded
 * by the caller (the Python PeerGather checks this with one all_reduce at construction). */

/* ---- occupancy-grid collision checks (SURVEY.md section 8f-2) ----------------
 * Batched Collision::collisionCheck (collision.cpp:126-143) and validate_control
 * (numerics.hpp:312-330) -- the call the exploration loop makes on the twist control()
 * returns, every tick (exploration.hpp:238).  One occupancy grid (GridMap: int8 cells,
 * row-major, i = y row / j = x column, grid.hpp:52) is shared by the whole batch. */
typedef struct eb_grid eb_grid;
typedef struct eb_collision {
  double boundary_radius;    /* collision.hpp:95-96 */
  double search_radius;
  double obstacle_threshold;
  double occupied_threshold;
} eb_collision;
/* copies ysize x xsize cells to the device; resolution / xmin / ymin as GridMap (grid.cpp:46-61) */
eb_status eb_grid_create(int device, const signed char *data, unsigned int xsize, unsigned int ysize,
                         double resolution, double xmin, double ymin, eb_grid **out);
eb_status eb_grid_update(eb_grid *g, const signed char *data); /* GridMap::update, same geometry */
void eb_grid_destroy(eb_grid *g);
eb_status eb_grid_set_stream(eb_grid *g, void *cuda_stream);
/* EB_ERR_INVALID_ARGUMENT where the Collision constructor throws (collision.cpp:46-64) */
/* hit[i] = 1 when pose i (x, y, theta; 3 x count) collides */
eb_status eb_collision_check_host(eb_grid *g, const eb_collision *c, const double *poses, int count, int *hit);
eb_status eb_collision_check_dev(eb_grid *g, const eb_collision *c, const double *poses_dev, int count,
                                 int *hit_dev);
/* valid[i] = 1 when twist u_i held for |horizon / dt| steps of dt from x0_i stays collision free */
eb_status eb_validate_control_host(eb_grid *g, const eb_collision *c, const double *x0, const double *u, int count,
                                   double dt, double horizon, int *valid);
eb_status eb_validate_control_dev(eb_grid *g, const eb_collision *c, const double *x0_dev, const double *u_dev,
                                  int count, double dt, double horizon, int *valid_dev);
long long eb_grid_launch_count(const eb_grid *g);
/* The checks can run against a pre-dilated copy of the map (one lookup per pose instead of the circle
 * walk; identical flags, built once per map update and set of radii).  mode 0 = automatic (when a call
 * checks more poses than a quarter of the map's cells, or a matching copy already exists), 1 = never,
 * 2 = always. */
eb_status eb_grid_set_dilation(eb_grid *g, int mode);

/* integrate_twist + normalize_angle_PI (numerics.hpp:273-298, 77-89) for 3 x count poses and twists on the
 * device (out may alias x): the constant-twist step of validate_control / DynamicWindow, exported for closed loops */
eb_status eb_integrate_twist_dev(int device, const double *x_dev, const double *u_dev, double dt, int count,
                                 double *out_dev, void *cuda_stream);

/* ---- DynamicWindow (SURVEY.md section 8f-3) -----------------------------------
 * Batched DynamicWindow::control (dynamic_window.cpp:93-187): for every instance the
 * vx x vy x vth candidate twists of its dynamic window (:189-235) are rolled out as
 * constant twists with a collision check per step (objective :237-286) and the first
 * minimum-cost collision-free twist in the reference's loop order is returned.
 * eb_dwa = the constructor arguments after `collision` (dynamic_window.hpp:60-65). */
typedef struct eb_dwa {
  double dt, horizon, acc_dt, acc_lim_x, acc_lim_y, acc_lim_th;
  double max_vel_x, min_vel_x, max_vel_y, min_vel_y, max_rot_vel, min_rot_vel;
  unsigned int vx_samples, vy_samples, vth_samples; /* 0 is promoted to 1 (:71-91) */
} eb_dwa;
/* control(grid, x0, vb, vref) :93-139 -- x0, vb, vref, u_opt: 3 x count; found[i] = 0 when no twist is
 * collision free (u_opt = 0); min_cost may be NULL */
eb_status eb_dwa_control_twist_host(eb_grid *g, const eb_collision *c, const eb_dwa *d, const double *x0,
                                    const double *vb, const double *vref, int count, int *found, double *u_opt,
                                    double *min_cost);
eb_status eb_dwa_control_twist_dev(eb_grid *g, const eb_collision *c, const eb_dwa *d, const double *x0_dev,
                                   const double *vb_dev, const double *vref_dev, int count, int *found_dev,
                                   double *u_opt_dev, double *min_cost_dev);
/* control(grid, x0, vb, xt_ref, dt_ref) :141-187 -- xt_ref is 3 x ncols, one trajectory for the whole batch
 * (per_instance = 0) or 3 x ncols x count, e.g. the output of eb_opt_traj_dev (per_instance = 1) */
eb_status eb_dwa_control_traj_host(eb_grid *g, const eb_collision *c, const eb_dwa *d, const double *x0,
                                   const double *vb, const double *xt_ref, int ncols, int per_instance,
                                   double dt_ref, int count, int *found, double *u_opt, double *min_cost);
eb_status eb_dwa_control_traj_dev(eb_grid *g, const eb_collision *c, const eb_dwa *d, const double *x0_dev,
                                  const double *vb_dev, const double *xt_ref_dev, int ncols, int per_instance,
                                  double dt_ref, int count, int *found_dev, double *u_opt_dev, double *min_cost_dev);

/* ---- per-instance occupancy maps -------------------------------------------------------------------------------
 * An eb_grid_batch holds B occupancy maps on one device and one stream, each with its own shape, resolution and origin,
 * so B robots on B maps run their collision checks, validate_control and DynamicWindow as one launch per call.  For
 * every instance i each output equals, bit for bit, what the eb_grid calls above return for eb_grid_create(map i) with
 * eb_grid_set_dilation(1), whatever the other maps are: the radii r_bnd, r_col, r_max are derived per instance from the
 * call's eb_collision and map i's resolution (collision.cpp:130-133), and the circles are always walked (there is no
 * pre-dilated map per instance).
 * eb_grid_batch_set_maps_dev / _host: the same arguments and rules as eb_set_map_targets_batch_dev / _host, so one set
 *   of arrays per map update feeds both.  Instance i with update[i] != 0 (update NULL: all) gets a device copy of map i
 *   (cells ysize[i] x xsize[i], GridMap layout), its resolution and its origin (origin[2i], origin[2i+1] = xmin, ymin).
 *   The maps live in one device arena; unflagged instances keep their cells and geometry, also when a flagged map
 *   outgrows its slot and every map moves to a new arena.  One kernel launch per call (none when nothing is flagged).
 *   _dev is stream-ordered: the cells must stay alive until the copy kernel has run.  _host packs the flagged maps
 *   into one pinned buffer, copies it with one cudaMemcpyAsync and synchronises.  EB_ERR_INVALID_ARGUMENT, before
 *   anything is launched, for a flagged map with a zero size, a resolution <= 0 or non-finite, more than 2^31 - 1 cells,
 *   or a NULL cells pointer.
 * eb_collision_check_batch_* / eb_validate_control_batch_*: poses / x0 / u are 3 x (per * B), instance-major: pose p is
 *   checked against map p / per (per >= 1); outputs per * B ints.
 * eb_dwa_control_*_batch_*: robot i on map i (B robots); the other arguments as eb_dwa_control_twist_* / _traj_*
 *   (xt_ref 3 x ncols shared, or 3 x ncols x B with per_instance = 1, e.g. the output of eb_opt_traj_dev).
 * Every check is one kernel launch; _host adds the copies of inputs and outputs and a synchronise.  The checks return
 * EB_ERR_INVALID_ARGUMENT before launching where the Collision constructor throws, for per < 1, per * B beyond INT_MAX,
 * and while some instance has never been given a map. */
typedef struct eb_grid_batch eb_grid_batch;
eb_status eb_grid_batch_create(int device, int batch, eb_grid_batch **out);
void eb_grid_batch_destroy(eb_grid_batch *g);
eb_status eb_grid_batch_set_stream(eb_grid_batch *g, void *cuda_stream);
long long eb_grid_batch_launch_count(const eb_grid_batch *g);
eb_status eb_grid_batch_set_maps_dev(eb_grid_batch *g, const signed char *const *cells_dev, const unsigned *xsize,
                                     const unsigned *ysize, const double *resolution, const double *origin /* 2 x B */,
                                     const int *update /* B or NULL */);
eb_status eb_grid_batch_set_maps_host(eb_grid_batch *g, const signed char *const *cells, const unsigned *xsize,
                                      const unsigned *ysize, const double *resolution, const double *origin,
                                      const int *update);
/* eb_grid_batch_set_rows_dev / _host: rows [row_begin[i], row_begin[i] + row_count[i]) of map i <- rows[i], row_count[i]
 *   x xsize_i int8 cells in GridMap layout (device pointers for _dev, host pointers for _host), for every instance i
 *   with update[i] != 0 (update NULL: all).  The map must be there already; its geometry, resolution and origin do not
 *   change (a map that changes shape or origin goes through eb_grid_batch_set_maps_*).  row_begin, row_count and update
 *   are host arrays of B; a flagged instance with row_count 0, and every unflagged instance, is not read.  One kernel
 *   launch per call (none when no row is written), after the grid batch's last safe tick or
 *   eb_set_map_targets_from_grid_batch; _dev is stream-ordered, _host packs the bands into one pinned buffer, copies
 *   it with one cudaMemcpyAsync and synchronises.  EB_ERR_INVALID_ARGUMENT, before anything is copied or launched, for
 *   a NULL handle or array, a flagged instance without a map, row_begin + row_count > ysize_i, or a NULL band of a
 *   flagged instance with row_count > 0.
 * eb_grid_batch_get_map_host: map i (ysize_i x xsize_i bytes) out of the arena into cells; synchronises. */
eb_status eb_grid_batch_set_rows_dev(eb_grid_batch *g, const signed char *const *rows_dev, const unsigned *row_begin,
                                     const unsigned *row_count, const int *update /* B or NULL */);
eb_status eb_grid_batch_set_rows_host(eb_grid_batch *g, const signed char *const *rows, const unsigned *row_begin,
                                      const unsigned *row_count, const int *update);
eb_status eb_grid_batch_get_map_host(const eb_grid_batch *g, int i, signed char *cells);
eb_status eb_collision_check_batch_host(eb_grid_batch *g, const eb_collision *c, const double *poses, int per, int *hit);
eb_status eb_collision_check_batch_dev(eb_grid_batch *g, const eb_collision *c, const double *poses_dev, int per,
                                       int *hit_dev);
eb_status eb_validate_control_batch_host(eb_grid_batch *g, const eb_collision *c, const double *x0, const double *u,
                                         int per, double dt, double horizon, int *valid);
eb_status eb_validate_control_batch_dev(eb_grid_batch *g, const eb_collision *c, const double *x0_dev,
                                        const double *u_dev, int per, double dt, double horizon, int *valid_dev);
eb_status eb_dwa_control_twist_batch_host(eb_grid_batch *g, const eb_collision *c, const eb_dwa *d, const double *x0,
                                          const double *vb, const double *vref, int *found, double *u_opt,
                                          double *min_cost);
eb_status eb_dwa_control_twist_batch_dev(eb_grid_batch *g, const eb_collision *c, const eb_dwa *d, const double *x0_dev,
                                         const double *vb_dev, const double *vref_dev, int *found_dev,
                                         double *u_opt_dev, double *min_cost_dev);
eb_status eb_dwa_control_traj_batch_host(eb_grid_batch *g, const eb_collision *c, const eb_dwa *d, const double *x0,
                                         const double *vb, const double *xt_ref, int ncols, int per_instance,
                                         double dt_ref, int *found, double *u_opt, double *min_cost);
eb_status eb_dwa_control_traj_batch_dev(eb_grid_batch *g, const eb_collision *c, const eb_dwa *d, const double *x0_dev,
                                        const double *vb_dev, const double *xt_ref_dev, int ncols, int per_instance,
                                        double dt_ref, int *found_dev, double *u_opt_dev, double *min_cost_dev);

/* ---- row-sharded phi_k on several GPUs (SURVEY.md section 8e) -----------------------
 * The all-reduce of the ranks' raw 32 x 32 blocks is fused into the tile kernel: the last CTA of every rank stores its
 * block into all ranks' receive buffers over NVLink peer memory (CUDA IPC mappings, exchanged once like eb_peer_group),
 * raises an arrival flag, waits for the others' and sums the slots in rank order.  eb_phik_execute_allreduce_dev is a
 * COLLECTIVE call: every rank of the group makes it once per step with a plan of its own row block. */
typedef struct eb_phik_peer eb_phik_peer;
int eb_phik_peer_blob_bytes(void);
eb_status eb_phik_peer_create(int device, int rank, int world, eb_phik_peer **out);
eb_status eb_phik_peer_export(eb_phik_peer *g, unsigned char *blob);
eb_status eb_phik_peer_connect(eb_phik_peer *g, const unsigned char *blobs /* world blobs, rank order */);
void eb_phik_peer_destroy(eb_phik_peer *g);
eb_status eb_phik_execute_allreduce_dev(eb_phik_plan *p, eb_phik_peer *g, const double *phi_dev, double *phik_dev,
                                        double *phi_sum_dev /* may be NULL */);

/* ---- map-derived target (SURVEY.md section 8f-4) ------------------------------
 * Density from an occupancy grid: Phi[i][j] = entropy(cell / 100) (numerics.hpp:164-179 over GridMap::getCell,
 * grid.cpp:177-184; -1 = unknown), sampled at the cell centres of the map frame [0, xsize * res] x [0, ysize * res],
 * normalised like Target::fill (target.cpp:87) and contracted like Basis::spatialCoeff (basis.cpp:122-133).
 * One execute per map update; phik_dev can be handed to eb_set_phik_dev without a host round trip.
 * Large maps whose width is a multiple of 16 cells run as ONE kernel (the bytes are staged by TMA, the entropy table
 * is looked up in shared memory, folded DMMA tiles): the density itself is then never written;
 * eb_map_target_density_dev materialises it on demand from the cells of the last execute (which must still be alive). */
typedef struct eb_map_target eb_map_target;
eb_status eb_map_target_create(int device, unsigned int xsize, unsigned int ysize, double resolution, int nb,
                               eb_map_target **out);
void eb_map_target_destroy(eb_map_target *m);
eb_status eb_map_target_set_stream(eb_map_target *m, void *cuda_stream);
eb_status eb_map_target_execute_dev(eb_map_target *m, const signed char *cells_dev, double *phik_dev,
                                    double *phi_sum_dev /* may be NULL */);
eb_status eb_map_target_execute_host(eb_map_target *m, const signed char *cells, double *phik, double *phi_sum);
double *eb_map_target_density_dev(eb_map_target *m); /* un-normalised entropy density of the last execute, [ysize][xsize]; NULL on failure */
eb_status eb_map_target_extent(const eb_map_target *m, double *lx, double *ly);
long long eb_map_target_launch_count(const eb_map_target *m);
/* phik_ <- a device buffer of K doubles (stream-ordered copy), basis extent (lx, ly) */
eb_status eb_set_phik_dev(eb_controller *c, const double *phik_dev, double lx, double ly);

/* ---- per-instance targets ----------------------------------------------------------------------------------------
 * Every instance owns its target, phi_k and map frame, as B reference ErgodicControl objects each driven with its own
 * GridMap would.  The first of these calls switches the controller to per-instance mode; from then on the shared target
 * calls (eb_set_target_gaussians, eb_config_target, eb_set_phik, eb_set_phik_dev, eb_get_phik, eb_control_host / _dev)
 * return EB_ERR_INVALID_ARGUMENT and eb_control_dev_gather[_wait] EB_ERR_UNSUPPORTED (eb_control_batch_dev_gather[_wait]
 * below gather per-instance twists).  Layouts are column-major
 * (Armadillo): instance i owns column i.
 * eb_set_target_gaussians_batch: Target::setTarget per instance; counts[i] <= max_n <= 256 Gaussians of instance i in
 *   columns of mu / sigma (2 x max_n x B).  Does not rebuild phi_k by itself.
 * eb_config_target_batch_dev: configTarget (ergodic_control.hpp:363-416) of every instance in one launch, bounds_dev
 *   4 x B {xmin xmax ymin ymax}.  The origin is always recorded; phi_k is rebuilt where the extent moved by >= 1e-12
 *   (rebuilt_dev[i] = 1).  A moved extent without Gaussians or a non-positive one is reported by the next synchronising
 *   call (eb_check_status, eb_control_batch_host) as EB_ERR_INVALID_ARGUMENT.
 * eb_set_phik_batch_dev: phi_k rows (K x B, device) and extents (2 x B {lx, ly}, device); origins are kept.  Map-derived
 *   rows are simpler through eb_set_map_targets_batch_dev / _host below.
 * eb_control_batch_dev / _host: eb_control_dev / _host with per-instance bounds (4 x B, device / host).  bounds NULL:
 *   the frames of the last configure are used and no frame launch is made (the per-tick fast path). */
eb_status eb_set_target_gaussians_batch(eb_controller *c, int max_n, const int *counts /* B */,
                                        const double *mu /* 2 x max_n x B */, const double *sigma /* 2 x max_n x B */);
eb_status eb_set_phik_batch_dev(eb_controller *c, const double *phik_dev /* K x B */,
                                const double *extent_dev /* 2 x B: lx, ly */);
eb_status eb_get_phik_batch(const eb_controller *c, double *phik /* K x B, may be NULL */,
                            double *extent /* 2 x B, may be NULL */);
eb_status eb_config_target_batch_dev(eb_controller *c, const double *bounds_dev /* 4 x B: xmin xmax ymin ymax */,
                                     int *rebuilt_dev /* B, may be NULL */);
eb_status eb_control_batch_dev(eb_controller *c, const double *bounds_dev, const double *x_dev, const int *mem_idx_dev,
                               double *u0_dev, double *metric_dev);
eb_status eb_control_batch_host(eb_controller *c, const double *bounds, const double *x, const int *mem_idx,
                                double *u0, double *metric);
/* Map-derived (entropy) target per instance, ONE kernel launch for the whole batch.  For every instance i with
 * update[i] != 0 (update NULL: all):
 *   phi_k row i  <- the entropy target of map i, what eb_map_target_create(xsize[i], ysize[i], resolution[i], nb) +
 *                   eb_map_target_execute compute (cell centres, Target::fill normalisation, spatialCoeff), to rounding;
 *                   row i depends on map i alone (bit-identical whatever else is in the batch)
 *   frame i      <- origin (origin[2i], origin[2i+1]) = the GridMap's xmin / ymin,
 *                   extent (xsize[i] * resolution[i], ysize[i] * resolution[i])
 *   the replay cosines of instance i are re-derived if its frame moved (as eb_config_target_batch_dev does).
 * Rows, frames and replay cosines of the other instances are not touched.  Switches the controller to per-instance
 * mode like every eb_*_batch target call.  xsize, ysize, resolution, origin (2 x B) and update are host arrays; cells
 * holds B pointers (host array) to ysize[i] x xsize[i] int8 cells in GridMap layout (row-major, x fastest): device
 * pointers for _dev (stream-ordered, returns at once; the cells must stay alive until the launch has run), host
 * pointers for _host (packed into pinned memory, copied, run, synchronised).  The pointer of an instance that is not
 * flagged is not read and may be NULL.  No flagged instance: nothing is launched.
 * EB_ERR_INVALID_ARGUMENT, before anything is launched, for a flagged map with a zero size, a resolution <= 0 or
 * non-finite, more than 2^31 - 1 cells, or a NULL cells pointer.
 * Afterwards eb_control_batch_* runs with bounds NULL (once every instance has a frame), or with the maps' own bounds
 * {xmin, xmin + xsize * res, ymin, ymin + ysize * res}: their extent is almost_equal to the frame's, so nothing is
 * rebuilt (the rule the single-map flow relies on).  A later configure whose extent really moves rebuilds that instance
 * from its Gaussians (eb_set_target_gaussians_batch), as for any per-instance target. */
eb_status eb_set_map_targets_batch_dev(eb_controller *c, const signed char *const *cells_dev, const unsigned *xsize,
                                       const unsigned *ysize, const double *resolution, const double *origin /* 2 x B */,
                                       const int *update /* B or NULL */);
eb_status eb_set_map_targets_batch_host(eb_controller *c, const signed char *const *cells, const unsigned *xsize,
                                        const unsigned *ysize, const double *resolution, const double *origin,
                                        const int *update);
/* The same targets from the maps of an eb_grid_batch, without a second upload: for every flagged instance i
 * (update NULL: all) the row, the frame and the replay cosines equal, bit for bit, what eb_set_map_targets_batch_dev
 * returns for map i's cells, geometry and origin, with the same rules (per-instance mode, unflagged instances not
 * touched).  row_begin / row_count NULL: whole maps.  Otherwise (host arrays of B) they declare the rows of map i that
 * changed since this controller last derived instance i from this grid batch: the arrays given to
 * eb_grid_batch_set_rows_*, or their union over several such calls.  The controller keeps each derived instance's raw
 * nb x nb block of every 64-row unit of its map, and recomputes only the units that meet the declared rows; the row is
 * then the sum of all kept blocks in unit order, as in the full call.  An instance is recomputed whole when it has no
 * kept blocks yet, when they came from another grid batch or from a map of another xsize, ysize or resolution, or when
 * its map was replaced by eb_grid_batch_set_maps_* since.  A flagged instance with nothing to recompute keeps the row
 * and frame it was last derived with.
 * The kept blocks take K doubles per unit: for 4096 maps of 160-640 rows (about 27.6 k units) 22 MB at nb 10, 57 MB at
 * nb 16, 226 MB at nb 32 and 0.9 GB at nb 64, plus up to a quarter of headroom for a map that grew (its slot then
 * takes its units and a quarter more, so a growing map rarely moves the blocks).
 * Stream-ordered on the controller's stream, after the work enqueued on the grid batch's stream, with one kernel
 * launch (none when no unit needs work); the grid batch's next set or rows call waits for it.
 * EB_ERR_INVALID_ARGUMENT, before anything is launched: a NULL handle, a grid batch of another B or on another device,
 * a flagged instance without a map, row_begin + row_count > ysize_i, or only one of row_begin / row_count NULL. */
eb_status eb_set_map_targets_from_grid_batch(eb_controller *c, eb_grid_batch *g,
                                             const unsigned *row_begin /* B or NULL */,
                                             const unsigned *row_count /* B or NULL */, const int *update /* B or NULL */);

/* ---- safe control tick of B robots on B maps -----------------------------------------------------------------------
 * The reference loop's arbitration between the ergodic twist and the safety planner (exploration.hpp:238-247) for a
 * per-instance controller and an eb_grid_batch of the same B on the same device, as one stream-ordered call with no
 * host synchronisation.  For every robot i:
 *   1. u0_i = what eb_control_batch_dev(c, bounds, x, mem_idx, u0, metric) returns; the controller's state (ut_, pose,
 *      replay sampling) advances exactly as in that call, and metric (NULL: not written) is that call's;
 *   2. ok_i = eb_validate_control_batch_dev of (x_i, u0_i) on map i with col, val_dt and val_horizon;
 *   3. ok_i: u_i = u0_i, branch_i = 0.  Otherwise (found_i, ud_i) = eb_dwa_control_traj_batch_dev on map i with col, dwa,
 *      vb_i and robot i's optTraj() (eb_opt_traj_dev, ncols = N, dt_ref = the controller's dt) as the reference;
 *      found: u_i = ud_i, branch_i = 1; not found: u_i = 0, branch_i = 2.
 * Every output equals that composition of calls bit for bit, and robot i's results depend on robot i alone.  The
 * dynamic window runs only for the robots whose twist fails validation; the B x N x 3 optTraj is never written.
 * Work runs on the controller's stream, after the work already enqueued on the grid batch's stream (an event: a
 * eb_grid_batch_set_maps_dev followed by a tick needs no synchronisation), and the grid batch's next set call waits for
 * the last tick before it writes or frees a map.  With bounds_dev NULL a tick is exactly three kernel launches, counted
 * by eb_launch_count (solve, validate + compaction, dynamic window over the failing robots) plus a cudaMemsetAsync of a
 * counter; given bounds add eb_control_batch_dev's frame launch.  Device-side faults of the solve surface as for
 * eb_control_batch_dev (eb_check_status); _host copies x, vb, bounds and mem_idx in, runs, copies u, branch and metric
 * out and synchronises.
 * Refused before anything is launched or copied, so an error leaves the controller as it was: EB_ERR_INVALID_ARGUMENT
 * for a NULL argument, a controller without per-instance targets (a shared target, or no eb_*_batch target call yet),
 * bounds NULL before any frame was configured, a grid batch of another B or on another device, an instance without a
 * map, an eb_collision the Collision constructor refuses, val_dt == 0 or dwa->dt == 0; EB_ERR_OUT_OF_RANGE when the
 * window's rollout outlasts the N-column optTraj (as eb_dwa_control_traj_*).
 * Not covered: the reference loop's policy of following the planner for a while once it took over, and replanning
 * (ROS-loop policy; branch lets a caller build it). */
eb_status eb_control_safe_batch_dev(eb_controller *c, eb_grid_batch *g, const eb_collision *col, const eb_dwa *dwa,
                                    double val_dt, double val_horizon, const double *bounds_dev /* 4 x B or NULL */,
                                    const double *x_dev /* 3 x B */, const int *mem_idx_dev, const double *vb_dev /* 3 x B */,
                                    double *u_dev /* 3 x B */, int *branch_dev /* B */, double *metric_dev /* B or NULL */);
eb_status eb_control_safe_batch_host(eb_controller *c, eb_grid_batch *g, const eb_collision *col, const eb_dwa *dwa,
                                     double val_dt, double val_horizon, const double *bounds, const double *x,
                                     const int *mem_idx, const double *vb, double *u, int *branch, double *metric);

/* ---- per-instance control and the safe tick on several GPUs ------------------------------------------------------
 * The per-instance counterparts of eb_control_dev_gather[_wait]: each rank of an eb_peer_group (elems = 3 * B, created
 * on the controller's device) runs its B robots, and the twists land in every rank's gathered buffer over peer memory,
 * with no collective call.  Each call is one step of the group (eb_peer_group_steps advances by one; a group's steps may
 * mix these calls and eb_peer_group_wait), and after it rows [rank * B, (rank + 1) * B) of eb_peer_gathered_dev(pg,
 * step) on every rank hold, bit for bit, what this rank's
 *   eb_control_batch_dev_gather[_wait]:      eb_control_batch_dev(c, bounds_dev, x_dev, mem_idx_dev, u0, metric_dev)
 *   eb_control_safe_batch_dev_gather[_wait]: eb_control_safe_batch_dev(c, g, col, dwa, ..., u, branch_dev, metric_dev)
 * returns as u0 / u.  The controller's state advances exactly as in that call; branch_dev (B) and metric_dev (B, may be
 * NULL) are this rank's local outputs.  Plain forms: the rows are here after eb_peer_group_wait(pg, c, step).  _wait
 * forms: when the enqueued work has run, every rank's rows of the step are here; everything runs on the controller's
 * stream.  The buffers rotate and are reused as for eb_control_dev_gather.
 * eb_control_batch_dev_gather[_wait] publish as eb_control_dev_gather[_wait] do for the same batch size: from inside the
 * solve kernel (batch >= eb_gather_fuse_min_batch()), else through peer_publish_kernel on the group's stream (or
 * peer_publish_wait_kernel behind the solve kernel for _wait).  eb_control_safe_batch_dev_gather[_wait] are the safe
 * tick's three launches (plus its counter memset): the solve writes to controller scratch, the validation stores the
 * rows of the valid robots to every rank, the dynamic window those of the failing ones, raises the arrival flags and,
 * for _wait, waits for every rank's.  Given bounds add one frame launch, as in the single-GPU calls.
 * Refused, with nothing launched and the step counter unchanged: whatever the single-GPU call refuses, a NULL or
 * unconnected group or one sized for another batch (as eb_control_dev_gather), and a group on another device than the
 * controller (EB_ERR_INVALID_ARGUMENT). */
eb_status eb_control_batch_dev_gather(eb_controller *c, eb_peer_group *pg, const double *bounds_dev /* 4 x B or NULL */,
                                      const double *x_dev, const int *mem_idx_dev, double *metric_dev);
eb_status eb_control_batch_dev_gather_wait(eb_controller *c, eb_peer_group *pg, const double *bounds_dev,
                                           const double *x_dev, const int *mem_idx_dev, double *metric_dev);
eb_status eb_control_safe_batch_dev_gather(eb_controller *c, eb_peer_group *pg, eb_grid_batch *g, const eb_collision *col,
                                           const eb_dwa *dwa, double val_dt, double val_horizon,
                                           const double *bounds_dev /* 4 x B or NULL */, const double *x_dev,
                                           const int *mem_idx_dev, const double *vb_dev, int *branch_dev,
                                           double *metric_dev);
eb_status eb_control_safe_batch_dev_gather_wait(eb_controller *c, eb_peer_group *pg, eb_grid_batch *g,
                                                const eb_collision *col, const eb_dwa *dwa, double val_dt,
                                                double val_horizon, const double *bounds_dev, const double *x_dev,
                                                const int *mem_idx_dev, const double *vb_dev, int *branch_dev,
                                                double *metric_dev);

/* ---- kinematic models and the forward integrator (SURVEY.md section 8 rows a8 / a9) ----
 * model: 0 SimpleCart, 1 Omni (models/cart.hpp:152-206, models/omni.hpp:164-215), 2 Cart (cart.hpp:60-145;
 * params = { wheel_radius, wheel_base }; 2 wheel velocities), 3 Mecanum (omni.hpp:59-157; params = { wheel_radius,
 * wheel_base_x, wheel_base_y }; 4 wheel velocities).  eb_rk4_solve = RungeKutta::solve (integrator.hpp:135-152):
 * x0 3 x count, ut nu x steps (one signal for all instances) or nu x steps x count (per_instance), xt 3 x steps x count,
 * steps = |horizon / dt|, heading wrapped after every step.  SimpleCart with a y-velocity: EB_ERR_INVALID_ARGUMENT
 * (cart.hpp:167-170) from the _host call, bit 0 of *fault_dev from the _dev call. */
int eb_model_controls(int model);
eb_status eb_rk4_solve_host(int device, int model, const double *params, double dt, double horizon, const double *x0,
                            const double *ut, int per_instance, int count, double *xt);
eb_status eb_rk4_solve_dev(int device, int model, const double *params, double dt, double horizon,
                           const double *x0_dev, const double *ut_dev, int per_instance, int count, double *xt_dev,
                           int *fault_dev, void *cuda_stream);
/* operator() -> f (3 x count), fdx -> A (3 x 3 x count), fdu -> B (3 x nu x count), wheels2Twist -> vb (3 x count);
 * outputs may be NULL */
eb_status eb_model_eval_host(int device, int model, const double *params, const double *x, const double *u, int count,
                             double *f, double *A, double *B, double *vb);

/* ---- measurement helpers --------------------------------------------------
 * eb_l2_gather_peak: measured rate (G sectors/s) of random 1-byte loads over a 16 MB L2-resident buffer -- the
 * roofline denominator of the collision / DynamicWindow kernels. */
eb_status eb_l2_gather_peak(int device, double *gsectors_per_s);
/*
 * Measured FP64 throughput of the device (TFLOP/s, 2 flop per FMA): a
 * register-resident DFMA loop and an mma.sync m8n8k4 f64 (DMMA) loop.  Used
 * as the FP64 roofline denominator (MEASURED_PEAKS.json has no FP64 figure). */
eb_status eb_fp64_peak(int device, double *dfma_tflops, double *dmma_tflops);

#ifdef __cplusplus
}
#endif
#endif /* ERGODIC_B200_H */

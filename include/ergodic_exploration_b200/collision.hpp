/**
 * @file collision.hpp
 * @brief Header-only C++ adapter for the batched occupancy-grid collision checks
 *        of libergodic_b200 (include/ergodic_b200.h, eb_grid_* / eb_collision_check_* /
 *        eb_validate_control_*).
 *
 * Mirrors, in namespace ergodic_exploration::b200, what the exploration loop calls right
 * after ErgodicControl::control() on every tick (exploration.hpp:238):
 *   Collision::collisionCheck(grid, pose)                     collision.cpp:126-143
 *   validate_control(collision, grid, x0, u, dt, horizon)     numerics.hpp:312-330
 *   DynamicWindow::control(grid, x0, vb, vref | xt_ref)       dynamic_window.cpp:93-187
 * for one pose / twist (the reference's signatures), for a 3 x B batch sharing one map (DeviceGrid), or for B
 * instances on B maps (DeviceGridBatch: instance i is checked against map i, one kernel launch per call); controlSafe
 * runs the whole tick of B robots on B maps (control, validate_control, DynamicWindow where needed) as one call.
 * The grid type is anything with the reference GridMap's getters
 * (gridData(), xsize(), ysize(), resolution(), xmin(), ymin(); grid.hpp:201-255).
 * The reference's Collision keeps its radii private (collision.hpp:159-163), so the
 * four constructor arguments are given to this class directly; it throws where the
 * reference constructor throws (collision.cpp:52-63).  Armadillo in, Armadillo / std out.
 */
#ifndef ERGODIC_EXPLORATION_B200_COLLISION_HPP
#define ERGODIC_EXPLORATION_B200_COLLISION_HPP

#include <memory>
#include <cmath>
#include <stdexcept>
#include <string>
#include <tuple>
#include <vector>

#include <armadillo>

#include <ergodic_b200.h>
#include <ergodic_exploration_b200/ergodic_control.hpp>

namespace ergodic_exploration
{
namespace b200
{
/** @brief An occupancy grid resident on the GPU (copy of a GridMap's cells and geometry) */
class DeviceGrid
{
public:
  template <class GridT>
  explicit DeviceGrid(const GridT& grid)
    : xsize_(grid.xsize()), ysize_(grid.ysize()), resolution_(grid.resolution()), xmin_(grid.xmin()), ymin_(grid.ymin())
  {
    eb_grid* g = nullptr;
    check(eb_grid_create(default_device(), reinterpret_cast<const signed char*>(grid.gridData().data()), xsize_,
                         ysize_, resolution_, xmin_, ymin_, &g));
    h_.reset(g, eb_grid_destroy);
  }

  /** @brief GridMap::update (grid.cpp:84-94): new cells; a new geometry re-creates the device copy */
  template <class GridT>
  void update(const GridT& grid)
  {
    if (grid.xsize() != xsize_ || grid.ysize() != ysize_ || grid.resolution() != resolution_ ||
        grid.xmin() != xmin_ || grid.ymin() != ymin_)
    {
      *this = DeviceGrid(grid);
      return;
    }
    check(eb_grid_update(h_.get(), reinterpret_cast<const signed char*>(grid.gridData().data())));
  }

  eb_grid* handle() const { return h_.get(); }

private:
  unsigned int xsize_, ysize_;
  double resolution_, xmin_, ymin_;
  std::shared_ptr<eb_grid> h_;
};

/**
 * @brief B occupancy grids resident on the GPU, one per instance (eb_grid_batch): every map has its own shape,
 * resolution and origin.  Built from and updated with the same GridMap-like objects as
 * BatchedErgodicControl::setMapTargets, so one vector of grids per map update feeds both.
 */
class DeviceGridBatch
{
public:
  template <class GridT>
  explicit DeviceGridBatch(const std::vector<GridT>& grids)
    : batch_(static_cast<unsigned int>(grids.size())), xsize_(grids.size(), 0)
  {
    if (grids.empty()) throw std::logic_error("DeviceGridBatch: need at least one grid");
    eb_grid_batch* g = nullptr;
    check(eb_grid_batch_create(default_device(), int(batch_), &g));
    h_.reset(g, eb_grid_batch_destroy);
    update(grids);
  }

  /** @brief instance i gets grids[i]'s cells and geometry when (*update)[i] (nullptr: all); the others keep theirs */
  template <class GridT>
  void update(const std::vector<GridT>& grids, const std::vector<bool>* update = nullptr)
  {
    if (grids.size() != batch_) throw std::logic_error("DeviceGridBatch::update: need B grids");
    if (update && update->size() != batch_) throw std::logic_error("DeviceGridBatch::update: update needs B flags");
    std::vector<const signed char*> cells(batch_, nullptr);
    std::vector<unsigned> xs(batch_), ys(batch_);
    std::vector<double> res(batch_), origin(2 * size_t(batch_));
    std::vector<int> upd(batch_, 1);
    for (unsigned int i = 0; i < batch_; i++)
    {
      if (update) upd[i] = (*update)[i] ? 1 : 0;
      if (upd[i]) cells[i] = reinterpret_cast<const signed char*>(grids[i].gridData().data());
      xs[i] = static_cast<unsigned>(grids[i].xsize());
      ys[i] = static_cast<unsigned>(grids[i].ysize());
      res[i] = grids[i].resolution();
      origin[2 * i + 0] = grids[i].xmin();
      origin[2 * i + 1] = grids[i].ymin();
    }
    check(eb_grid_batch_set_maps_host(h_.get(), cells.data(), xs.data(), ys.data(), res.data(), origin.data(),
                                      upd.data()));
    for (unsigned int i = 0; i < batch_; i++)
      if (upd[i]) xsize_[i] = xs[i];
  }

  /**
   * @brief rows [row_begin[i], row_begin[i] + n_i) of map i <- bands[i] (n_i x xsize_i cells, GridMap layout) when
   * (*update)[i] (nullptr: all); shapes and origins do not change.  Pass row_begin and the n_i to setMapTargets.
   */
  void updateRows(const std::vector<std::vector<signed char>>& bands, const std::vector<unsigned>& row_begin,
                  const std::vector<bool>* update = nullptr)
  {
    if (bands.size() != batch_ || row_begin.size() != batch_)
      throw std::logic_error("DeviceGridBatch::updateRows: need B bands and B row_begin");
    if (update && update->size() != batch_) throw std::logic_error("DeviceGridBatch::updateRows: update needs B flags");
    std::vector<const signed char*> rows(batch_, nullptr);
    std::vector<unsigned> count(batch_, 0);
    std::vector<int> upd(batch_, 1);
    for (unsigned int i = 0; i < batch_; i++)
    {
      if (update) upd[i] = (*update)[i] ? 1 : 0;
      if (!upd[i] || bands[i].empty()) continue;
      if (xsize_[i] == 0 || bands[i].size() % xsize_[i] != 0)
        throw std::logic_error("DeviceGridBatch::updateRows: band " + std::to_string(i) + " is not whole rows of its map");
      rows[i] = bands[i].data();
      count[i] = static_cast<unsigned>(bands[i].size() / xsize_[i]);
    }
    check(eb_grid_batch_set_rows_host(h_.get(), rows.data(), row_begin.data(), count.data(), upd.data()));
  }

  eb_grid_batch* handle() const { return h_.get(); }
  unsigned int batch() const { return batch_; }

  /** @brief rows per instance of a 3 x (per * B) matrix */
  int per(const arma::mat& m, const char* what) const
  {
    if (m.n_rows != 3 || m.n_cols == 0 || m.n_cols % batch_ != 0)
      throw std::logic_error(std::string(what) + ": must be 3 x (per * B)");
    return static_cast<int>(m.n_cols / batch_);
  }

private:
  unsigned int batch_;
  std::vector<unsigned> xsize_;  // of each map set so far (0: none)
  std::shared_ptr<eb_grid_batch> h_;
};

/** @brief Collision (collision.hpp:85-165) evaluated on the GPU, one pose or a batch */
class Collision
{
public:
  Collision(double boundary_radius, double search_radius, double obstacle_threshold, double occupied_threshold)
    : cfg_{ boundary_radius, search_radius, obstacle_threshold, occupied_threshold }
  {
    if (search_radius < boundary_radius)  // collision.cpp:52-56
      throw std::invalid_argument("Search radius must be at least the same size as the boundary radius");
    if (occupied_threshold > 100.0 || occupied_threshold < 0.0)  // collision.cpp:58-62
      throw std::invalid_argument("Occupied threshold must be between 0 and 100");
  }

  double totalPadding() const { return cfg_.boundary_radius + cfg_.obstacle_threshold; }  // collision.cpp:145-148

  /** @brief collision.cpp:126-143 */
  bool collisionCheck(const DeviceGrid& grid, const arma::vec& pose) const
  {
    if (pose.n_elem != 3) throw std::logic_error("collisionCheck: pose must have 3 elements");
    int hit = 0;
    check(eb_collision_check_host(grid.handle(), &cfg_, pose.memptr(), 1, &hit));
    return hit != 0;
  }

  /** @brief batch: poses is 3 x B; returns B flags, 1 = collision */
  std::vector<int> collisionCheck(const DeviceGrid& grid, const arma::mat& poses) const
  {
    if (poses.n_rows != 3) throw std::logic_error("collisionCheck: poses must be 3 x B");
    std::vector<int> hit(poses.n_cols);
    check(eb_collision_check_host(grid.handle(), &cfg_, poses.memptr(), static_cast<int>(poses.n_cols), hit.data()));
    return hit;
  }

  /** @brief per-instance maps: poses is 3 x (per * B), instance-major; pose p is checked against map p / per */
  std::vector<int> collisionCheck(const DeviceGridBatch& grids, const arma::mat& poses) const
  {
    const int per = grids.per(poses, "collisionCheck: poses");
    std::vector<int> hit(poses.n_cols);
    check(eb_collision_check_batch_host(grids.handle(), &cfg_, poses.memptr(), per, hit.data()));
    return hit;
  }

  const eb_collision& config() const { return cfg_; }

private:
  eb_collision cfg_;
};

/** @brief numerics.hpp:312-330: true if the constant twist is collision free over the horizon */
inline bool validate_control(const Collision& collision, const DeviceGrid& grid, const arma::vec& x0,
                             const arma::vec& u, double dt, double horizon)
{
  if (x0.n_elem != 3 || u.n_elem != 3) throw std::logic_error("validate_control: x0 and u must have 3 elements");
  int valid = 0;
  check(eb_validate_control_host(grid.handle(), &collision.config(), x0.memptr(), u.memptr(), 1, dt, horizon, &valid));
  return valid != 0;
}

/** @brief batch: x0 and u are 3 x B (B start poses / candidate twists on one map) */
inline std::vector<int> validate_control(const Collision& collision, const DeviceGrid& grid, const arma::mat& x0,
                                         const arma::mat& u, double dt, double horizon)
{
  if (x0.n_rows != 3 || u.n_rows != 3 || x0.n_cols != u.n_cols)
    throw std::logic_error("validate_control: x0 and u must be 3 x B");
  std::vector<int> valid(x0.n_cols);
  check(eb_validate_control_host(grid.handle(), &collision.config(), x0.memptr(), u.memptr(),
                                 static_cast<int>(x0.n_cols), dt, horizon, valid.data()));
  return valid;
}
/** @brief per-instance maps: x0 and u are 3 x (per * B), instance-major; row p is checked against map p / per */
inline std::vector<int> validate_control(const Collision& collision, const DeviceGridBatch& grids, const arma::mat& x0,
                                         const arma::mat& u, double dt, double horizon)
{
  const int per = grids.per(x0, "validate_control: x0");
  if (u.n_rows != 3 || u.n_cols != x0.n_cols) throw std::logic_error("validate_control: x0 and u must be 3 x (per * B)");
  std::vector<int> valid(x0.n_cols);
  check(eb_validate_control_batch_host(grids.handle(), &collision.config(), x0.memptr(), u.memptr(), per, dt, horizon,
                                       valid.data()));
  return valid;
}

/** @brief DynamicWindow (dynamic_window.hpp:60-172) evaluated on the GPU, one robot or a batch */
class DynamicWindow
{
public:
  /** @brief same argument order as dynamic_window.hpp:60-65 */
  DynamicWindow(const Collision& collision, double dt, double horizon, double acc_dt, double acc_lim_x,
                double acc_lim_y, double acc_lim_th, double max_vel_x, double min_vel_x, double max_vel_y,
                double min_vel_y, double max_rot_vel, double min_rot_vel, unsigned int vx_samples,
                unsigned int vy_samples, unsigned int vth_samples)
    : collision_(collision)
    , cfg_{ dt,        horizon,   acc_dt,    acc_lim_x,   acc_lim_y,   acc_lim_th, max_vel_x,  min_vel_x,
            max_vel_y, min_vel_y, max_rot_vel, min_rot_vel, vx_samples, vy_samples, vth_samples }
  {
  }

  /** @brief dynamic_window.cpp:93-139: (collision-free twist found, optimal twist) */
  std::tuple<bool, arma::vec> control(const DeviceGrid& grid, const arma::vec& x0, const arma::vec& vb,
                                      const arma::vec& vref) const
  {
    if (x0.n_elem != 3 || vb.n_elem != 3 || vref.n_elem != 3) throw std::logic_error("DynamicWindow::control: 3-vectors");
    int found = 0;
    arma::vec u(3);
    check(eb_dwa_control_twist_host(grid.handle(), &collision_.config(), &cfg_, x0.memptr(), vb.memptr(),
                                    vref.memptr(), 1, &found, u.memptr(), nullptr));
    return std::make_tuple(found != 0, u);
  }

  /** @brief dynamic_window.cpp:141-187: follow a reference trajectory (3 x n, time step dt_ref) */
  std::tuple<bool, arma::vec> control(const DeviceGrid& grid, const arma::vec& x0, const arma::vec& vb,
                                      const arma::mat& xt_ref, double dt_ref) const
  {
    if (x0.n_elem != 3 || vb.n_elem != 3 || xt_ref.n_rows != 3 || xt_ref.n_cols < 1)
      throw std::logic_error("DynamicWindow::control: x0, vb 3-vectors and xt_ref 3 x n");
    int found = 0;
    arma::vec u(3);
    check(eb_dwa_control_traj_host(grid.handle(), &collision_.config(), &cfg_, x0.memptr(), vb.memptr(),
                                   xt_ref.memptr(), static_cast<int>(xt_ref.n_cols), 0, dt_ref, 1, &found, u.memptr(),
                                   nullptr));
    return std::make_tuple(found != 0, u);
  }

  /** @brief batch: x0, vb, vref are 3 x B; returns the B found flags and the 3 x B optimal twists */
  std::tuple<std::vector<int>, arma::mat> controlBatch(const DeviceGrid& grid, const arma::mat& x0, const arma::mat& vb,
                                                      const arma::mat& vref) const
  {
    if (x0.n_rows != 3 || vb.n_rows != 3 || vref.n_rows != 3 || x0.n_cols != vb.n_cols || x0.n_cols != vref.n_cols)
      throw std::logic_error("DynamicWindow::controlBatch: x0, vb, vref must be 3 x B");
    std::vector<int> found(x0.n_cols);
    arma::mat u(3, x0.n_cols);
    check(eb_dwa_control_twist_host(grid.handle(), &collision_.config(), &cfg_, x0.memptr(), vb.memptr(),
                                    vref.memptr(), static_cast<int>(x0.n_cols), found.data(), u.memptr(), nullptr));
    return std::make_tuple(found, u);
  }

  /** @brief per-instance maps: robot i (column i of the 3 x B x0, vb, vref) on map i */
  std::tuple<std::vector<int>, arma::mat> controlBatch(const DeviceGridBatch& grids, const arma::mat& x0,
                                                       const arma::mat& vb, const arma::mat& vref) const
  {
    const unsigned int B = grids.batch();
    if (x0.n_rows != 3 || vb.n_rows != 3 || vref.n_rows != 3 || x0.n_cols != B || vb.n_cols != B || vref.n_cols != B)
      throw std::logic_error("DynamicWindow::controlBatch: x0, vb, vref must be 3 x B");
    std::vector<int> found(B);
    arma::mat u(3, B);
    check(eb_dwa_control_twist_batch_host(grids.handle(), &collision_.config(), &cfg_, x0.memptr(), vb.memptr(),
                                          vref.memptr(), found.data(), u.memptr(), nullptr));
    return std::make_tuple(found, u);
  }

  /**
   * @brief per-instance maps and reference trajectories: robot i on map i follows columns [i * n, (i + 1) * n) of
   * xt_ref (3 x (n * B), time step dt_ref), the layout BatchedErgodicControl::optTraj() returns
   */
  std::tuple<std::vector<int>, arma::mat> controlBatch(const DeviceGridBatch& grids, const arma::mat& x0,
                                                       const arma::mat& vb, const arma::mat& xt_ref, double dt_ref) const
  {
    const unsigned int B = grids.batch();
    if (x0.n_rows != 3 || vb.n_rows != 3 || x0.n_cols != B || vb.n_cols != B)
      throw std::logic_error("DynamicWindow::controlBatch: x0, vb must be 3 x B");
    const int ncols = grids.per(xt_ref, "DynamicWindow::controlBatch: xt_ref");
    std::vector<int> found(B);
    arma::mat u(3, B);
    check(eb_dwa_control_traj_batch_host(grids.handle(), &collision_.config(), &cfg_, x0.memptr(), vb.memptr(),
                                         xt_ref.memptr(), ncols, 1, dt_ref, found.data(), u.memptr(), nullptr));
    return std::make_tuple(found, u);
  }

  double timeStep() const { return cfg_.dt; }
  double horizon() const { return cfg_.horizon; }
  unsigned int steps() const { return static_cast<unsigned int>(std::abs(cfg_.horizon / cfg_.dt)); }
  const eb_dwa& config() const { return cfg_; }

private:
  Collision collision_;
  eb_dwa cfg_;
};

/**
 * @brief One safe control tick of B robots on B maps (eb_control_safe_batch_host), the reference loop's arbitration
 * (exploration.hpp:238-247): u = ctl.control(grids, X); where validate_control(collision, grids, X, u, val_dt,
 * val_horizon) fails, dwa.controlBatch(grids, X, VB, ctl.optTraj(), ctl's time step) takes over, and a robot whose
 * window finds nothing gets the zero twist.  The window runs only for the robots that need it.  ctl must hold
 * per-instance frames (setMapTargets or control(grids, x) before); they are used as they are.
 * @return the 3 x B twists and the B branches (0 ergodic twist, 1 dynamic window, 2 nothing found)
 */
template <class ModelT>
std::tuple<arma::mat, std::vector<int>> controlSafe(BatchedErgodicControl<ModelT>& ctl, const DeviceGridBatch& grids,
                                                    const Collision& collision, const DynamicWindow& dwa,
                                                    const arma::mat& X, const arma::mat& VB, double val_dt,
                                                    double val_horizon)
{
  const unsigned int B = grids.batch();
  if (ctl.batch() != B) throw std::logic_error("controlSafe: the controller and the grid batch need the same B");
  if (X.n_rows != 3 || VB.n_rows != 3 || X.n_cols != B || VB.n_cols != B)
    throw std::logic_error("controlSafe: X and VB must be 3 x B");
  arma::mat u(3, B);
  std::vector<int> branch(B);
  check(eb_control_safe_batch_host(ctl.handle(), grids.handle(), &collision.config(), &dwa.config(), val_dt,
                                   val_horizon, nullptr, X.memptr(), nullptr, VB.memptr(), u.memptr(), branch.data(),
                                   nullptr));
  return std::make_tuple(u, branch);
}

/**
 * @brief ErgodicControl::setMapTargets of every flagged instance i from map i of grids, without uploading the cells
 * again: bit for bit the target of map i's cells and geometry.  row_begin / row_count (both or neither; nullptr: whole
 * maps) declare the rows of map i changed since ctl last derived instance i from grids (what updateRows was given);
 * only the 64-row units that meet them are recomputed.
 */
template <class ModelT>
void setMapTargets(BatchedErgodicControl<ModelT>& ctl, DeviceGridBatch& grids,
                   const std::vector<unsigned>* row_begin = nullptr, const std::vector<unsigned>* row_count = nullptr,
                   const std::vector<bool>* update = nullptr)
{
  const unsigned int B = grids.batch();
  if (ctl.batch() != B) throw std::logic_error("setMapTargets: the controller and the grid batch need the same B");
  if ((row_begin && row_begin->size() != B) || (row_count && row_count->size() != B) || (update && update->size() != B))
    throw std::logic_error("setMapTargets: row_begin, row_count and update need B entries");
  std::vector<int> upd(B, 1);
  if (update)
    for (unsigned int i = 0; i < B; i++) upd[i] = (*update)[i] ? 1 : 0;
  check(eb_set_map_targets_from_grid_batch(ctl.handle(), grids.handle(), row_begin ? row_begin->data() : nullptr,
                                           row_count ? row_count->data() : nullptr, upd.data()));
}
}  // namespace b200
}  // namespace ergodic_exploration
#endif

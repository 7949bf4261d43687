/**
 * ergodic_exploration_b200/ergodic_control.hpp
 *
 * Header-only drop-in for the reference's hot-path C++ API, backed by the
 * sm_100a CUDA kernels behind include/ergodic_b200.h.  Armadillo in,
 * Armadillo out; same names, argument meaning and exception types as
 *   ergodic_exploration/ergodic_control.hpp:72-185   ErgodicControl<ModelT>
 *   ergodic_exploration/basis.hpp:50-106             Basis
 *   ergodic_exploration/target.hpp:56-161            Gaussian, Target
 *   ergodic_exploration/models/{cart,omni}.hpp       Cart, SimpleCart, Mecanum, Omni
 * so a node main (exploration_{cart,omni}_node.cpp) switches by changing its
 * include path and linking libergodic_b200.so (see INTEGRATION.md).
 *
 * What stays with the caller: GridMap and Collision (the controller reads only
 * xmin/xmax/ymin/ymax of the grid and never touches the collision object,
 * SURVEY App. B-11), hence control()/configTarget() accept any type with those
 * four getters and the constructor takes `const Collision&` for any Collision.
 * ROS message producers (path(), Target::markers()) are compiled only when
 * ERGODIC_B200_WITH_ROS is defined (they need nav_msgs / tf2 /
 * visualization_msgs headers).
 *
 * All arithmetic of control(), optTraj(), configTarget(), Basis::* and
 * Target::fill runs on the GPU; nothing here falls back to the CPU.  The model
 * structs keep their small host-side operator()/fdx/fdu (they are the model
 * definitions users pass around), the controller itself only uses their type.
 */
#ifndef ERGODIC_EXPLORATION_B200_ERGODIC_CONTROL_HPP
#define ERGODIC_EXPLORATION_B200_ERGODIC_CONTROL_HPP

#include <cmath>
#include <cstring>
#include <stdexcept>
#include <string>
#include <type_traits>
#include <utility>
#include <algorithm>
#include <vector>

#include <armadillo>

#include "../ergodic_b200.h"

#ifdef ERGODIC_B200_WITH_ROS
#include <nav_msgs/Path.h>
#include <tf2/LinearMath/Quaternion.h>
#include <visualization_msgs/MarkerArray.h>
#endif

namespace ergodic_exploration
{
using arma::imat;
using arma::mat;
using arma::vec;

constexpr double PI = 3.14159265358979323846;  // numerics.hpp:58

class Collision;  // stays with the caller; only its reference is taken

namespace b200
{
/** @brief eb_status -> the exception type the reference would have thrown */
inline void check(eb_status st)
{
  if (st == EB_OK) return;
  const std::string msg = eb_last_error();
  if (st == EB_ERR_INVALID_ARGUMENT) throw std::invalid_argument(msg);
  if (st == EB_ERR_OUT_OF_RANGE) throw std::out_of_range(msg);
  throw std::runtime_error(msg);
}

/** @brief CUDA device used by objects constructed afterwards (default 0) */
inline int& default_device()
{
  static int device = 0;
  return device;
}
}  // namespace b200

// ---------------------------------------------------------------------------
// numerics.hpp (the two helpers the hot path's callers use)
// ---------------------------------------------------------------------------
inline bool almost_equal(double d1, double d2, double epsilon = 1.0e-12)  // numerics.hpp:67-70
{
  return std::fabs(d1 - d2) < epsilon;
}

inline double normalize_angle_PI(double rad)  // numerics.hpp:77-89
{
  const auto q = std::floor((rad + PI) / (2.0 * PI));
  rad = (rad + PI) - q * 2.0 * PI;
  if (rad < 0.0) rad += 2.0 * PI;
  return rad - PI;
}

// ---------------------------------------------------------------------------
// models (models/cart.hpp, models/omni.hpp)
// ---------------------------------------------------------------------------
namespace models
{
/** @brief 2 wheel differential drive, controls [uL, uR] (cart.hpp:60-145) */
struct Cart
{
  Cart(double wheel_radius, double wheel_base) : wheel_radius(wheel_radius), wheel_base(wheel_base), state_space(3) {}

  vec wheels2Twist(const vec u) const
  {
    return { wheel_radius / 2.0 * (u(0) + u(1)), 0.0, wheel_radius / (2.0 * wheel_base) * (u(1) - u(0)) };
  }
  vec operator()(const vec x, const vec u) const
  {
    const double f = wheel_radius / 2.0;
    return { f * ((u(0) + u(1)) * std::cos(x(2))), f * ((u(0) + u(1)) * std::sin(x(2))),
             f * ((u(1) - u(0)) / wheel_base) };
  }
  mat fdx(const vec x, const vec u) const
  {
    mat A(3, 3, arma::fill::zeros);
    A(0, 2) = -(wheel_radius / 2.0) * (u(0) + u(1)) * std::sin(x(2));
    A(1, 2) = (wheel_radius / 2.0) * (u(0) + u(1)) * std::cos(x(2));
    return A;
  }
  mat fdu(const vec x) const
  {
    const double f = wheel_radius / 2.0;
    mat B(3, 2);
    B(0, 0) = B(0, 1) = f * std::cos(x(2));
    B(1, 0) = B(1, 1) = f * std::sin(x(2));
    B(2, 0) = f * (-1.0 / wheel_base);
    B(2, 1) = f * (1.0 / wheel_base);
    return B;
  }
  double wheel_radius, wheel_base;
  unsigned int state_space;
};

/** @brief differential drive driven by a body twist [vx, vy, w] (cart.hpp:152-206) */
struct SimpleCart
{
  SimpleCart() : state_space(3) {}
  vec operator()(const vec x, const vec u) const
  {
    if (!almost_equal(u(1), 0.0)) throw std::invalid_argument("Invalid twist y-velocity must be 0.");
    return { u(0) * std::cos(x(2)), u(0) * std::sin(x(2)), u(2) };
  }
  mat fdx(const vec x, const vec u) const
  {
    mat A(3, 3, arma::fill::zeros);
    A(0, 2) = -u(0) * std::sin(x(2));
    A(1, 2) = u(0) * std::cos(x(2));
    return A;
  }
  mat fdu(const vec x) const
  {
    mat B(3, 3, arma::fill::zeros);
    B(0, 0) = std::cos(x(2));
    B(1, 0) = std::sin(x(2));
    B(2, 2) = 1.0;
    return B;
  }
  unsigned int state_space;
};

/** @brief 4 mecanum wheels, controls are wheel velocities (omni.hpp:59-157) */
struct Mecanum
{
  Mecanum(double wheel_radius, double wheel_base_x, double wheel_base_y)
    : wheel_radius(wheel_radius), wheel_base_x(wheel_base_x), wheel_base_y(wheel_base_y), state_space(3)
  {
  }
  vec wheels2Twist(const vec u) const
  {
    const double l = 1.0 / (wheel_base_x + wheel_base_y), f = wheel_radius / 4.0;
    return { f * (u(0) + u(1) + u(2) + u(3)), f * (-u(0) + u(1) - u(2) + u(3)),
             f * (-l * u(0) + l * u(1) + l * u(2) - l * u(3)) };
  }
  vec operator()(const vec x, const vec u) const
  {
    const double s = (wheel_radius / 4.0) * std::sin(x(2)), c = (wheel_radius / 4.0) * std::cos(x(2));
    const double l = wheel_radius / (4.0 * (wheel_base_x + wheel_base_y));
    return { u(0) * (s + c) + u(1) * (-s + c) + u(2) * (s + c) + u(3) * (-s + c),
             u(0) * (s - c) + u(1) * (s + c) + u(2) * (s - c) + u(3) * (s + c),
             -u(0) * l + u(1) * l + u(2) * l - u(3) * l };
  }
  mat fdx(const vec x, const vec u) const
  {
    const double s = (wheel_radius / 4.0) * std::sin(x(2)), c = (wheel_radius / 4.0) * std::cos(x(2));
    mat A(3, 3, arma::fill::zeros);
    A(0, 2) = u(0) * (-s + c) + u(1) * (-s - c) + u(2) * (-s + c) + u(3) * (-s - c);
    A(1, 2) = u(0) * (s + c) + u(1) * (-s + c) + u(2) * (s + c) + u(3) * (-s + c);
    return A;
  }
  mat fdu(const vec x) const
  {
    const double s = (wheel_radius / 4.0) * std::sin(x(2)), c = (wheel_radius / 4.0) * std::cos(x(2));
    const double l = wheel_radius / (4.0 * (wheel_base_x + wheel_base_y));
    return { { s + c, -s + c, s + c, -s + c }, { s - c, s + c, s - c, s + c }, { -l, l, l, -l } };
  }
  double wheel_radius, wheel_base_x, wheel_base_y;
  unsigned int state_space;
};

/** @brief omni-directional robot driven by a body twist [vx, vy, w] (omni.hpp:164-215) */
struct Omni
{
  Omni() : state_space(3) {}
  vec operator()(const vec x, const vec u) const
  {
    return { u(0) * std::cos(x(2)) - u(1) * std::sin(x(2)), u(0) * std::sin(x(2)) + u(1) * std::cos(x(2)), u(2) };
  }
  mat fdx(const vec x, const vec u) const
  {
    mat A(3, 3, arma::fill::zeros);
    A(0, 2) = -u(0) * std::sin(x(2)) - u(1) * std::cos(x(2));
    A(1, 2) = u(0) * std::cos(x(2)) - u(1) * std::sin(x(2));
    return A;
  }
  mat fdu(const vec x) const
  {
    return { { std::cos(x(2)), -std::sin(x(2)), 0.0 }, { std::sin(x(2)), std::cos(x(2)), 0.0 }, { 0.0, 0.0, 1.0 } };
  }
  unsigned int state_space;
};
}  // namespace models

namespace b200
{
/** @brief model type -> eb_model.  Only the 3-twist models can be driven by
 * ErgodicControl (ut_ has 3 rows, ergodic_control.hpp:201,447-449). */
template <class ModelT>
struct model_id
{
  static_assert(sizeof(ModelT) == 0, "ErgodicControl needs a 3-twist model: models::SimpleCart or models::Omni");
};
template <>
struct model_id<models::SimpleCart>
{
  static constexpr int value = EB_MODEL_SIMPLE_CART;
};
template <>
struct model_id<models::Omni>
{
  static constexpr int value = EB_MODEL_OMNI;
};
// model id + parameter block of the forward integrator (all four models)
template <class ModelT>
struct rk_model;
template <>
struct rk_model<models::SimpleCart>
{
  static constexpr int id = EB_MODEL_SIMPLE_CART;
  static void params(const models::SimpleCart&, double*) {}
};
template <>
struct rk_model<models::Omni>
{
  static constexpr int id = EB_MODEL_OMNI;
  static void params(const models::Omni&, double*) {}
};
template <>
struct rk_model<models::Cart>
{
  static constexpr int id = EB_MODEL_CART;
  static void params(const models::Cart& m, double* p)
  {
    p[0] = m.wheel_radius;
    p[1] = m.wheel_base;
  }
};
template <>
struct rk_model<models::Mecanum>
{
  static constexpr int id = EB_MODEL_MECANUM;
  static void params(const models::Mecanum& m, double* p)
  {
    p[0] = m.wheel_radius;
    p[1] = m.wheel_base_x;
    p[2] = m.wheel_base_y;
  }
};
}  // namespace b200

// ---------------------------------------------------------------------------
// RungeKutta, forward problem (integrator.hpp:60-152, 176-184)
// ---------------------------------------------------------------------------
/** @brief 4th order Runge-Kutta forward integration of a kinematic model on the GPU (rk4_solve_kernel).
 *  The co-state overload of the reference (integrator.hpp:154-174) lives inside the fused control() kernel. */
class RungeKutta
{
public:
  explicit RungeKutta(double dt) : dt_(dt) {}

  /** @brief Simulate the dynamics forward in time (integrator.hpp:135-152): xt is 3 x steps, headings wrapped */
  template <class ModelT>
  mat solve(const ModelT& model, const vec& x0, const mat& ut, double horizon) const
  {
    const auto steps = static_cast<unsigned int>(std::abs(horizon / dt_));
    if (x0.n_elem != 3 || ut.n_cols < steps || ut.n_rows != static_cast<arma::uword>(eb_model_controls(b200::rk_model<ModelT>::id)))
      throw std::logic_error("RungeKutta::solve: x0 must have 3 rows and ut one column of wheel / twist controls per step");
    double par[3] = { 0.0, 0.0, 0.0 };
    b200::rk_model<ModelT>::params(model, par);
    mat xt(3, steps);
    const eb_status st = eb_rk4_solve_host(0, b200::rk_model<ModelT>::id, par, dt_, horizon, x0.memptr(), ut.memptr(), 0, 1, xt.memptr());
    if (st == EB_ERR_INVALID_ARGUMENT) throw std::invalid_argument(eb_last_error());  // cart.hpp:167-170
    if (st != EB_OK) throw std::runtime_error(eb_last_error());
    return xt;
  }

private:
  double dt_;
};

// ---------------------------------------------------------------------------
// Basis (basis.hpp:50-106)
// ---------------------------------------------------------------------------
class Basis
{
public:
  Basis(double lx, double ly, unsigned int num_basis)
    : lx_(lx), ly_(ly), num_basis_(num_basis), total_basis_(num_basis * num_basis), lamdak_(total_basis_), k_(2, total_basis_)
  {
    unsigned int col = 0;  // basis.cpp:58-67: index = ky * nb + kx
    for (unsigned int i = 0; i < num_basis; i++)
      for (unsigned int j = 0; j < num_basis; j++)
      {
        k_(0, col) = j;
        k_(1, col) = i;
        col++;
      }
    for (unsigned int i = 0; i < total_basis_; i++)  // basis.cpp:72-75
      lamdak_(i) = 1.0 / std::pow(1.0 + std::sqrt(double(k_(0, i) * k_(0, i) + k_(1, i) * k_(1, i))), 1.5);
  }

  /** @brief cosine basis functions at x = [x y] (num_basis^2 x 1) */
  vec fourierBasis(const vec& x) const
  {
    vec fk(total_basis_);
    const double pt[2] = { x(0), x(1) };
    b200::check(eb_basis_traj_coeff_host(b200::default_device(), lx_, ly_, int(num_basis_), pt, 2, 1, fk.memptr()));
    return fk;
  }

  /** @brief gradient of each basis function (2 x num_basis^2) */
  mat gradFourierBasis(const vec& x) const
  {
    mat dfk(2, total_basis_);
    const double pt[2] = { x(0), x(1) };
    b200::check(eb_basis_grad_host(b200::default_device(), lx_, ly_, int(num_basis_), pt, dfk.memptr()));
    return dfk;
  }

  /** @brief trajectory fourier coefficients; xt holds one state per column */
  vec trajCoeff(const mat& xt) const
  {
    vec ck(total_basis_);
    b200::check(eb_basis_traj_coeff_host(b200::default_device(), lx_, ly_, int(num_basis_), xt.memptr(),
                                         int(xt.n_rows), int(xt.n_cols), ck.memptr()));
    return ck;
  }

  /** @brief spatial fourier coefficients of phi_vals sampled at the columns of phi_grid */
  vec spatialCoeff(const vec& phi_vals, const mat& phi_grid) const
  {
    if (phi_grid.n_rows != 2 || phi_grid.n_cols != phi_vals.n_elem)
      throw std::logic_error("Basis::spatialCoeff: phi_grid must be 2 x G with G = phi_vals.n_elem");
    vec phik(total_basis_);
    b200::check(eb_basis_spatial_coeff_host(b200::default_device(), lx_, ly_, int(num_basis_), phi_vals.memptr(),
                                            phi_grid.memptr(), (long long)phi_vals.n_elem, phik.memptr()));
    return phik;
  }

  const vec& lamdak() const { return lamdak_; }
  const imat& k() const { return k_; }

private:
  double lx_, ly_;
  unsigned int num_basis_, total_basis_;
  vec lamdak_;
  imat k_;
};

// ---------------------------------------------------------------------------
// Gaussian, Target (target.hpp:56-161)
// ---------------------------------------------------------------------------
struct Gaussian
{
  Gaussian() {}
  Gaussian(const vec& mu, const vec& sigmas) : mu(mu), sigmas(sigmas), cov(2, 2, arma::fill::zeros), cov_inv(2, 2, arma::fill::zeros)
  {
    cov(0, 0) = sigmas(0) * sigmas(0);  // diagmat(square(sigmas)), target.hpp:69
    cov(1, 1) = sigmas(1) * sigmas(1);
    const double det = cov(0, 0) * cov(1, 1);  // inv() of the diagonal 2x2
    cov_inv(0, 0) = cov(1, 1) / det;
    cov_inv(1, 1) = cov(0, 0) / det;
  }
  double operator()(const vec& pt) const { return (*this)(pt, vec({ 0.0, 0.0 })); }
  /** @param trans - translation from map frame to fourier domain (target.hpp:91-102) */
  double operator()(const vec& pt, const vec& trans) const
  {
    const double d0 = pt(0) - (mu(0) - trans(0)), d1 = pt(1) - (mu(1) - trans(1));
    return std::exp(-0.5 * ((d0 * cov_inv(0, 0)) * d0 + (d1 * cov_inv(1, 1)) * d1));
  }
  vec mu, sigmas;
  mat cov, cov_inv;
};
typedef std::vector<Gaussian> GaussianList;

class Target
{
public:
  Target() {}
  Target(const GaussianList& gaussians) : gaussians_(gaussians) {}
  void addGaussian(const Gaussian& g) { gaussians_.emplace_back(g); }
  void deleteGaussian(unsigned int idx) { gaussians_.erase(gaussians_.begin() + idx); }

  /** @brief value of the mixture at pt (target.cpp:68-76) */
  double evaluate(const vec& pt, const vec& trans) const
  {
    double val = 0.0;
    for (const auto& g : gaussians_) val += g(pt, trans);
    return val;
  }

  /** @brief target evaluated at every column of phi_grid, normalised to sum to 1 (target.cpp:78-89) */
  vec fill(const vec& trans, const mat& phi_grid) const
  {
    std::vector<double> mu, sg;
    pack(mu, sg);
    vec phi_vals(phi_grid.n_cols);
    const double tr[2] = { trans(0), trans(1) };
    b200::check(eb_target_fill_host(b200::default_device(), int(gaussians_.size()), mu.data(), sg.data(), tr,
                                    phi_grid.memptr(), (long long)phi_grid.n_cols, phi_vals.memptr()));
    return phi_vals;
  }

#ifdef ERGODIC_B200_WITH_ROS
  /** @brief the targets as ellipses (target.cpp:91-119) */
  visualization_msgs::MarkerArray markers(const std::string& frame) const
  {
    visualization_msgs::MarkerArray ma;
    ma.markers.resize(gaussians_.size());
    for (unsigned int i = 0; i < gaussians_.size(); i++)
    {
      auto& m = ma.markers.at(i);
      const double e0 = std::min(gaussians_.at(i).cov(0, 0), gaussians_.at(i).cov(1, 1));
      const double e1 = std::max(gaussians_.at(i).cov(0, 0), gaussians_.at(i).cov(1, 1));
      m.header.frame_id = frame;
      m.id = i;
      m.type = visualization_msgs::Marker::SPHERE;
      m.action = visualization_msgs::Marker::ADD;
      m.pose.position.x = gaussians_.at(i).mu(0);
      m.pose.position.y = gaussians_.at(i).mu(1);
      m.pose.orientation.w = 1.0;
      m.scale.x = 2.0 * e0;
      m.scale.y = 2.0 * e1;
      m.scale.z = 0.01;
      m.color.r = 1.0;
      m.color.g = 1.0;
      m.color.b = 0.6;
      m.color.a = 0.5;
    }
    return ma;
  }
#endif

  const GaussianList& gaussians() const { return gaussians_; }
  /** @brief flat (2 x n, column-major) means and sigmas for the C ABI */
  void pack(std::vector<double>& mu, std::vector<double>& sigma) const
  {
    mu.clear();
    sigma.clear();
    for (const auto& g : gaussians_)
    {
      mu.push_back(g.mu(0));
      mu.push_back(g.mu(1));
      sigma.push_back(g.sigmas(0));
      sigma.push_back(g.sigmas(1));
    }
  }

private:
  GaussianList gaussians_;
};

// ---------------------------------------------------------------------------
// ErgodicControl (ergodic_control.hpp:72-185)
// ---------------------------------------------------------------------------
namespace b200
{
/** @brief owning wrapper of an eb_controller handle with value semantics
 * (the reference object is copied by value into Exploration,
 * exploration.hpp:137-138: copies are deep, eb_clone) */
class Handle
{
public:
  Handle() : h_(nullptr) {}
  explicit Handle(const eb_config& cfg) : h_(nullptr) { check(eb_create(&cfg, &h_)); }
  Handle(const Handle& o) : h_(nullptr)
  {
    if (o.h_) check(eb_clone(o.h_, &h_));
  }
  Handle(Handle&& o) noexcept : h_(o.h_) { o.h_ = nullptr; }
  Handle& operator=(Handle o) noexcept
  {
    std::swap(h_, o.h_);
    return *this;
  }
  ~Handle() { eb_destroy(h_); }
  eb_controller* get() const { return h_; }

private:
  eb_controller* h_;
};

inline eb_config make_config(int model, int batch, double dt, double horizon, double resolution,
                             double exploration_weight, unsigned int num_basis, unsigned int buffer_size,
                             unsigned int batch_size, const mat& Rinv, const vec& umin, const vec& umax)
{
  if (Rinv.n_rows != 3 || Rinv.n_cols != 3 || umin.n_elem != 3 || umax.n_elem != 3)
    throw std::logic_error("ErgodicControl: Rinv must be 3x3 and umin/umax must have 3 elements");
  eb_config cfg;
  eb_config_defaults(&cfg, model);
  cfg.batch = batch;
  cfg.device = default_device();
  cfg.dt = dt;
  cfg.horizon = horizon;
  cfg.resolution = resolution;
  cfg.expl_weight = exploration_weight;
  cfg.num_basis = num_basis;
  cfg.buffer_size = buffer_size;
  cfg.batch_size = batch_size;
  std::memcpy(cfg.Rinv, Rinv.memptr(), sizeof(cfg.Rinv));  // column-major on both sides
  std::memcpy(cfg.umin, umin.memptr(), sizeof(cfg.umin));
  std::memcpy(cfg.umax, umax.memptr(), sizeof(cfg.umax));
  return cfg;
}
}  // namespace b200

/** @brief Receding horizon ergodic trajectory optimization (single robot) */
template <class ModelT>
class ErgodicControl
{
public:
  /** same argument list as ergodic_control.hpp:90-94 (CTAD-deducible) */
  template <class CollisionT = Collision>
  ErgodicControl(const ModelT& model, const CollisionT& /*collision: stored but never used by the reference*/,
                 double dt, double horizon, double resolution, double exploration_weight, unsigned int num_basis,
                 unsigned int buffer_size, unsigned int batch_size, const mat& Rinv, const vec& umin, const vec& umax)
    : model_(model)
    , dt_(dt)
    , horizon_(horizon)
    , steps_(static_cast<unsigned int>(std::abs(horizon / dt)))
    , h_(b200::make_config(b200::model_id<ModelT>::value, 1, dt, horizon, resolution, exploration_weight, num_basis,
                           buffer_size, batch_size, Rinv, umin, umax))
  {
  }

  /**
   * @brief Update the control signal (ergodic_control.hpp:225-311)
   * @param grid - anything with xmin()/xmax()/ymin()/ymax() (the reference's GridMap)
   * @param x - current state [x, y, theta]
   * @return first twist in the updated control signal [vx, vy, w]
   */
  template <class GridT>
  vec control(const GridT& grid, const vec& x)
  {
    if (x.n_elem != 3) throw std::logic_error("ErgodicControl::control: x must have 3 elements");
    vec u0(3);
    b200::check(eb_control_host(h_.get(), grid.xmin(), grid.xmax(), grid.ymin(), grid.ymax(), x.memptr(), nullptr,
                                u0.memptr(), nullptr));
    return u0;
  }

  /** @brief optimized trajectory, 3 x steps (ergodic_control.hpp:314-317) */
  mat optTraj() const
  {
    mat xt(3, steps_);
    b200::check(eb_opt_traj_host(h_.get(), xt.memptr()));
    return xt;
  }

#ifdef ERGODIC_B200_WITH_ROS
  /** @brief optimized trajectory as a path message (ergodic_control.hpp:320-342) */
  nav_msgs::Path path(const std::string& map_frame_id) const
  {
    nav_msgs::Path path;
    path.header.frame_id = map_frame_id;
    path.poses.resize(steps_);
    const mat opt_traj = optTraj();
    for (unsigned int i = 0; i < opt_traj.n_cols; i++)
    {
      path.poses.at(i).pose.position.x = opt_traj(0, i);
      path.poses.at(i).pose.position.y = opt_traj(1, i);
      tf2::Quaternion quat;
      quat.setRPY(0.0, 0.0, normalize_angle_PI(opt_traj(2, i)));
      path.poses.at(i).pose.orientation.x = quat.x();
      path.poses.at(i).pose.orientation.y = quat.y();
      path.poses.at(i).pose.orientation.z = quat.z();
      path.poses.at(i).pose.orientation.w = quat.w();
    }
    return path;
  }
#endif

  /** @brief add the robot's state to memory (ergodic_control.hpp:345-348) */
  void addStateMemory(const vec& x)
  {
    if (x.n_elem != 3) throw std::logic_error("ErgodicControl::addStateMemory: x must have 3 elements");
    b200::check(eb_add_state_memory_host(h_.get(), x.memptr()));
  }

  double timeStep() const { return dt_; }

  /** @brief set the target distribution (ergodic_control.hpp:357-360) */
  void setTarget(const Target& target)
  {
    std::vector<double> mu, sg;
    target.pack(mu, sg);
    b200::check(eb_set_target_gaussians(h_.get(), int(target.gaussians().size()), mu.data(), sg.data()));
  }

  /** @brief rebuild the target coefficients if the map extent changed (ergodic_control.hpp:363-416) */
  template <class GridT>
  void configTarget(const GridT& grid)
  {
    b200::check(eb_config_target(h_.get(), grid.xmin(), grid.xmax(), grid.ymin(), grid.ymax(), nullptr));
  }

  // ---- beyond the reference: state access for checkpoint / teacher forcing
  mat controlSignal() const
  {
    mat ut(3, steps_);
    b200::check(eb_get_ut(h_.get(), ut.memptr()));
    return ut;
  }
  void setControlSignal(const mat& ut)
  {
    if (ut.n_rows != 3 || ut.n_cols != steps_) throw std::logic_error("setControlSignal: ut must be 3 x steps");
    b200::check(eb_set_ut(h_.get(), ut.memptr()));
  }
  vec trajectoryCoefficients() const
  {
    vec ck(eb_num_coeff(h_.get()));
    b200::check(eb_get_ck(h_.get(), ck.memptr()));
    return ck;
  }
  vec targetCoefficients() const
  {
    vec phik(eb_num_coeff(h_.get()));
    b200::check(eb_get_phik(h_.get(), phik.memptr(), nullptr, nullptr));
    return phik;
  }
  eb_controller* handle() const { return h_.get(); }

private:
  ModelT model_;
  double dt_, horizon_;
  unsigned int steps_;
  b200::Handle h_;
};

/** @brief B independent controllers advanced by ONE kernel launch per
 * control() -- the batched face of the same hot path (3 x B in, 3 x B out). */
template <class ModelT>
class BatchedErgodicControl
{
public:
  BatchedErgodicControl(const ModelT& model, unsigned int batch, double dt, double horizon, double resolution,
                        double exploration_weight, unsigned int num_basis, unsigned int buffer_size,
                        unsigned int batch_size, const mat& Rinv, const vec& umin, const vec& umax)
    : model_(model)
    , batch_(batch)
    , steps_(static_cast<unsigned int>(std::abs(horizon / dt)))
    , h_(b200::make_config(b200::model_id<ModelT>::value, int(batch), dt, horizon, resolution, exploration_weight,
                           num_basis, buffer_size, batch_size, Rinv, umin, umax))
  {
  }

  /** @param x - 3 x B current states; @return 3 x B first twists; metric (optional) receives B ergodic metrics */
  template <class GridT>
  mat control(const GridT& grid, const mat& x, vec* metric = nullptr)
  {
    if (x.n_rows != 3 || x.n_cols != batch_) throw std::logic_error("BatchedErgodicControl::control: x must be 3 x B");
    mat u0(3, batch_);
    if (metric) metric->set_size(batch_);
    b200::check(eb_control_host(h_.get(), grid.xmin(), grid.xmax(), grid.ymin(), grid.ymax(), x.memptr(), nullptr,
                                u0.memptr(), metric ? metric->memptr() : nullptr));
    return u0;
  }
  void addStateMemory(const mat& x)
  {
    if (x.n_rows != 3 || x.n_cols != batch_) throw std::logic_error("addStateMemory: x must be 3 x B");
    b200::check(eb_add_state_memory_host(h_.get(), x.memptr()));
  }
  void setTarget(const Target& target)
  {
    std::vector<double> mu, sg;
    target.pack(mu, sg);
    b200::check(eb_set_target_gaussians(h_.get(), int(target.gaussians().size()), mu.data(), sg.data()));
  }
  /** @brief one target per instance (targets.size() == B); switches the controller to per-instance targets */
  void setTargets(const std::vector<Target>& targets)
  {
    if (targets.size() != batch_) throw std::logic_error("BatchedErgodicControl::setTargets: need B targets");
    int max_n = 1;
    for (const Target& t : targets) max_n = std::max(max_n, int(t.gaussians().size()));
    std::vector<int> counts(batch_);
    std::vector<double> mu(2 * size_t(max_n) * batch_, 0.0), sg(2 * size_t(max_n) * batch_, 1.0);
    for (unsigned int i = 0; i < batch_; i++)
    {
      std::vector<double> m, s;
      targets[i].pack(m, s);
      counts[i] = int(targets[i].gaussians().size());
      std::copy(m.begin(), m.end(), mu.begin() + 2 * size_t(max_n) * i);
      std::copy(s.begin(), s.end(), sg.begin() + 2 * size_t(max_n) * i);
    }
    b200::check(eb_set_target_gaussians_batch(h_.get(), max_n, counts.data(), mu.data(), sg.data()));
  }
  /**
   * @brief map-derived (entropy) target per instance from its occupancy grid, one kernel launch for the batch
   * @param grids B grids with the GridMap getters gridData() / xsize() / ysize() / resolution() / xmin() / ymin()
   * @param update instance i is updated when (*update)[i] (nullptr: all)
   * @details instance i gets the phi_k of grids[i]'s entropy density and grids[i]'s frame; control(grids, x) then
   * drives every robot in its own map.  Switches the controller to per-instance targets.
   */
  template <class GridT>
  void setMapTargets(const std::vector<GridT>& grids, const std::vector<bool>* update = nullptr)
  {
    if (grids.size() != batch_) throw std::logic_error("BatchedErgodicControl::setMapTargets: need B grids");
    if (update && update->size() != batch_)
      throw std::logic_error("BatchedErgodicControl::setMapTargets: update needs B flags");
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
    b200::check(eb_set_map_targets_batch_host(h_.get(), cells.data(), xs.data(), ys.data(), res.data(), origin.data(),
                                              upd.data()));
  }
  /** @brief per-instance maps: instance i is driven in grids[i]'s frame (after setTargets or setMapTargets) */
  template <class GridT>
  mat control(const std::vector<GridT>& grids, const mat& x, vec* metric = nullptr)
  {
    if (x.n_rows != 3 || x.n_cols != batch_) throw std::logic_error("BatchedErgodicControl::control: x must be 3 x B");
    if (grids.size() != batch_) throw std::logic_error("BatchedErgodicControl::control: need B grids");
    std::vector<double> bounds(4 * size_t(batch_));
    for (unsigned int i = 0; i < batch_; i++)
    {
      bounds[4 * i + 0] = grids[i].xmin();
      bounds[4 * i + 1] = grids[i].xmax();
      bounds[4 * i + 2] = grids[i].ymin();
      bounds[4 * i + 3] = grids[i].ymax();
    }
    mat u0(3, batch_);
    if (metric) metric->set_size(batch_);
    b200::check(eb_control_batch_host(h_.get(), bounds.data(), x.memptr(), nullptr, u0.memptr(),
                                      metric ? metric->memptr() : nullptr));
    return u0;
  }
  /** @brief 3 x (steps * B): instance i occupies columns [i*steps, (i+1)*steps) */
  mat optTraj() const
  {
    mat xt(3, size_t(steps_) * batch_);
    b200::check(eb_opt_traj_host(h_.get(), xt.memptr()));
    return xt;
  }
  unsigned int batch() const { return batch_; }
  unsigned int steps() const { return steps_; }
  eb_controller* handle() const { return h_.get(); }

private:
  ModelT model_;
  unsigned int batch_, steps_;
  b200::Handle h_;
};
}  // namespace ergodic_exploration
#endif

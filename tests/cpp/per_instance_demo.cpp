// tests/cpp/per_instance_demo.cpp -- BatchedErgodicControl with one target and one map per robot: three robots on
// maps with their own origins and extents (one of them grows after two ticks) in a closed loop.  Built against the
// test-only Armadillo stand-in (oracle/shim).  Prints, per tick, each robot's map bounds, pose and first twist for
// tests/test_cpp_per_instance.py to replay on the oracle.
#include <cstdio>
#include <vector>

#include <ergodic_exploration_b200/ergodic_control.hpp>

using namespace ergodic_exploration;

struct Bounds
{
  double x0, x1, y0, y1;
  double xmin() const { return x0; }
  double xmax() const { return x1; }
  double ymin() const { return y0; }
  double ymax() const { return y1; }
};

static void print_vec(const char* name, int i, const double* p, size_t n)
{
  std::printf("%s %d", name, i);
  for (size_t k = 0; k < n; k++) std::printf(" %.17g", p[k]);
  std::printf("\n");
}

int main()
{
  mat Rinv(3, 3, arma::fill::zeros);
  Rinv(0, 0) = 1.0;
  Rinv(1, 1) = 1.0;
  Rinv(2, 2) = 2.0;
  const unsigned B = 3;
  BatchedErgodicControl<models::Omni> bec(models::Omni(), B, 0.1, 5.0, 0.1, 1.0, 10, 1000, 100, Rinv,
                                          vec({ -1.0, -1.0, -2.0 }), vec({ 1.0, 1.0, 2.0 }));
  std::vector<Bounds> grids = { { 0.0, 10.0, 0.0, 10.0 }, { -8.35, 11.55, -13.95, 17.85 }, { 3.0, 15.0, -2.0, 6.0 } };
  std::vector<Target> targets;
  targets.emplace_back(GaussianList{ Gaussian(vec({ 2.5, 2.5 }), vec({ 1.5, 1.5 })), Gaussian(vec({ 8.5, 2.5 }), vec({ 1.5, 1.5 })) });
  targets.emplace_back(GaussianList{ Gaussian(vec({ 0.0, 5.0 }), vec({ 2.0, 1.0 })) });
  targets.emplace_back(GaussianList{ Gaussian(vec({ 6.0, 1.0 }), vec({ 1.0, 1.0 })), Gaussian(vec({ 12.0, 4.0 }), vec({ 1.5, 0.8 })),
                                     Gaussian(vec({ 9.0, 0.0 }), vec({ 1.2, 1.2 })) });
  bec.setTargets(targets);
  mat x(3, B);
  for (unsigned i = 0; i < B; i++)
  {
    x(0, i) = grids[i].x0 + 2.0 + i;
    x(1, i) = grids[i].y0 + 3.0;
    x(2, i) = 0.4 * i;
  }
  for (int step = 0; step < 4; step++)
  {
    if (step == 2) grids[2].x1 += 2.0;  // robot 2's map grows
    bec.addStateMemory(x);
    vec metric;
    const mat u = bec.control(grids, x, &metric);
    for (unsigned i = 0; i < B; i++)
    {
      const double b[4] = { grids[i].x0, grids[i].x1, grids[i].y0, grids[i].y1 };
      print_vec("bounds", int(i), b, 4);
      print_vec("x", int(i), x.colptr(i), 3);
      print_vec("u0", int(i), u.colptr(i), 3);
      print_vec("metric", int(i), &metric(i), 1);
    }
    for (unsigned i = 0; i < B; i++)
    {
      x(0, i) += 0.1 * u(0, i);  // any plant will do: the Python side replays the printed poses
      x(1, i) += 0.1 * u(1, i);
      x(2, i) += 0.1 * u(2, i);
    }
  }
  std::printf("OK\n");
  return 0;
}

// tests/cpp/map_targets_demo.cpp -- BatchedErgodicControl with a map-derived target per robot: three robots on
// GridMap-like occupancy maps with their own origins, targets set by setMapTargets and driven by control(grids, x);
// robot 1's map grows after two ticks (new cells, larger xsize).  Built against the test-only Armadillo stand-in
// (oracle/shim).  Prints, per tick, each robot's map geometry, pose and first twist for
// tests/test_cpp_map_targets.py to replay on the oracle (the cells follow cell_value below).
#include <cstdint>
#include <cstdio>
#include <vector>

#include <ergodic_exploration_b200/ergodic_control.hpp>

using namespace ergodic_exploration;

// the getters of the reference's GridMap (grid.hpp:201-255) that the adapter reads
struct Grid
{
  std::vector<int8_t> data;
  unsigned xs, ys;
  double res, x0, y0;
  const std::vector<int8_t>& gridData() const { return data; }
  unsigned xsize() const { return xs; }
  unsigned ysize() const { return ys; }
  double resolution() const { return res; }
  double xmin() const { return x0; }
  double ymin() const { return y0; }
  double xmax() const { return x0 + xs * res; }
  double ymax() const { return y0 + ys * res; }
};

// occupancy of cell (row i, column j) of robot r's map, generation gen: -1 (unknown) .. 100
static int8_t cell_value(unsigned i, unsigned j, unsigned r, unsigned gen)
{
  return static_cast<int8_t>(int((i * 31u + j * 17u + r * 7u + gen * 13u + (i * j) % 5u) % 102u) - 1);
}

static Grid make_grid(unsigned r, unsigned gen, unsigned xs, unsigned ys, double res, double x0, double y0)
{
  Grid g{ std::vector<int8_t>(size_t(xs) * ys), xs, ys, res, x0, y0 };
  for (unsigned i = 0; i < ys; i++)
    for (unsigned j = 0; j < xs; j++) g.data[size_t(i) * xs + j] = cell_value(i, j, r, gen);
  return g;
}

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
  std::vector<Grid> grids = { make_grid(0, 0, 120, 90, 0.05, 0.0, 0.0), make_grid(1, 0, 80, 61, 0.1, -8.350015, -13.950030),
                              make_grid(2, 0, 37, 150, 0.1, 3.0, -2.0) };
  std::vector<unsigned> gen = { 0, 0, 0 };
  bec.setMapTargets(grids);
  mat x(3, B);
  for (unsigned i = 0; i < B; i++)
  {
    x(0, i) = grids[i].x0 + 1.0 + 0.5 * i;
    x(1, i) = grids[i].y0 + 2.0;
    x(2, i) = 0.4 * i;
  }
  for (int step = 0; step < 4; step++)
  {
    if (step == 2)
    {
      grids[1] = make_grid(1, 1, 95, 61, 0.1, -8.350015, -13.950030);  // robot 1's map grows
      gen[1] = 1;
      const std::vector<bool> update = { false, true, false };
      bec.setMapTargets(grids, &update);
    }
    bec.addStateMemory(x);
    vec metric;
    const mat u = bec.control(grids, x, &metric);
    for (unsigned i = 0; i < B; i++)
    {
      const double g[6] = { double(grids[i].xs), double(grids[i].ys), grids[i].res, grids[i].x0, grids[i].y0,
                            double(gen[i]) };
      print_vec("grid", int(i), g, 6);
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

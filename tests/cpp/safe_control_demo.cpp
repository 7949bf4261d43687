// tests/cpp/safe_control_demo.cpp -- the exploration loop's safe tick for three robots, each on its own occupancy map,
// through b200::controlSafe: the ergodic twist where it validates on the robot's map, the dynamic window following the
// robot's optTraj() where it does not, the zero twist where the window finds nothing.  Robot 1's map grows after two
// ticks (new cells, larger xsize: the grid batch moves every map to a new arena).  Built against the test-only
// Armadillo stand-in (oracle/shim).  Prints, per tick and robot, the map geometry, the inputs and the results for
// tests/test_cpp_safe_control.py to replay through the composed Python calls (the cells follow cell_value below).
#include <cstdint>
#include <cstdio>
#include <vector>

#include <ergodic_exploration_b200/collision.hpp>

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

// occupancy of cell (row i, column j) of robot r's map, generation gen: mostly free, some obstacles and unknown cells
static int8_t cell_value(unsigned i, unsigned j, unsigned r, unsigned gen)
{
  const unsigned h = i * 31u + j * 17u + r * 7u + gen * 13u + (i * j) % 5u;
  return h % 41u == 0 ? int8_t(100) : (h % 23u == 0 ? int8_t(-1) : int8_t(0));
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
  // explore_omni.yaml radii and window (tests/test_dwa_cpu.py COL, DWA_OMNI)
  const b200::Collision collision(0.2, 1.0, 0.05, 0.65);
  const b200::DynamicWindow dwa(collision, 0.1, 2.0, 0.2, 1.0, 1.0, 2.0, 1.0, -1.0, 1.0, -1.0, 2.0, -2.0, 3, 8, 5);
  std::vector<Grid> grids = { make_grid(0, 0, 120, 90, 0.05, 0.0, 0.0), make_grid(1, 0, 80, 61, 0.1, -8.350015, -13.950030),
                              make_grid(2, 0, 37, 150, 0.1, 3.0, -2.0) };
  std::vector<unsigned> gen = { 0, 0, 0 };
  std::vector<bool> upd = { true, true, true };
  b200::DeviceGridBatch grid_batch(grids);
  mat x(3, B), vb(3, B, arma::fill::zeros);
  for (unsigned i = 0; i < B; i++)
  {
    x(0, i) = grids[i].x0 + 1.0 + 0.5 * i;
    x(1, i) = grids[i].y0 + 2.0;
    x(2, i) = 0.4 * i;
  }
  for (int step = 0; step < 6; step++)
  {
    if (step == 2)
    {
      grids[1] = make_grid(1, 1, 95, 61, 0.1, -8.350015, -13.950030);  // robot 1's map grows
      gen[1] = 1;
      upd = { false, true, false };
    }
    bec.setMapTargets(grids, &upd);
    grid_batch.update(grids, &upd);
    bec.addStateMemory(x);
    const auto [u, branch] = b200::controlSafe(bec, grid_batch, collision, dwa, x, vb, 0.1, 1.0);
    for (unsigned i = 0; i < B; i++)
    {
      const double g[6] = { double(grids[i].xs), double(grids[i].ys), grids[i].res, grids[i].x0, grids[i].y0,
                            double(gen[i]) };
      print_vec("grid", int(i), g, 6);
      print_vec("x", int(i), x.colptr(i), 3);
      print_vec("vb", int(i), vb.colptr(i), 3);
      print_vec("u", int(i), u.colptr(i), 3);
      const double b = branch[i];
      print_vec("branch", int(i), &b, 1);
    }
    for (unsigned i = 0; i < B; i++)
    {
      for (unsigned k = 0; k < 3; k++)  // any plant will do: the Python side replays the printed poses
      {
        x(k, i) += 0.1 * u(k, i);
        vb(k, i) = u(k, i);
      }
    }
    upd = { false, false, false };
  }
  std::printf("OK\n");
  return 0;
}

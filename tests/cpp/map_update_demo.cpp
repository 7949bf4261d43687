// tests/cpp/map_update_demo.cpp -- the row-band map update through the C++ adapter: three maps in a
// b200::DeviceGridBatch take bands of changed rows with updateRows, and b200::setMapTargets derives the entropy targets
// from the grid batch, recomputing only the changed rows.  A second controller gets the whole maps through
// BatchedErgodicControl::setMapTargets after every step; the two controllers' phi_k rows and extents must be equal bit
// for bit.  Built against the test-only Armadillo stand-in (oracle/shim); tests/test_cpp_map_update.py runs it.
#include <cstdint>
#include <cstdio>
#include <cstring>
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
};

static int8_t cell_value(unsigned i, unsigned j, unsigned r, unsigned gen)
{
  const unsigned h = i * 31u + j * 17u + r * 7u + gen * 13u + (i * j) % 5u;
  return h % 41u == 0 ? int8_t(100) : (h % 23u == 0 ? int8_t(-1) : int8_t(h % 7u == 0 ? 50 : 0));
}

static Grid make_grid(unsigned r, unsigned xs, unsigned ys, double res, double x0, double y0)
{
  Grid g{ std::vector<int8_t>(size_t(xs) * ys), xs, ys, res, x0, y0 };
  for (unsigned i = 0; i < ys; i++)
    for (unsigned j = 0; j < xs; j++) g.data[size_t(i) * xs + j] = cell_value(i, j, r, 0);
  return g;
}

int main()
{
  mat Rinv(3, 3, arma::fill::zeros);
  Rinv(0, 0) = 1.0;
  Rinv(1, 1) = 1.0;
  Rinv(2, 2) = 2.0;
  const unsigned B = 3, nb = 10, K = nb * nb;
  auto make_ctl = [&] {
    return BatchedErgodicControl<models::Omni>(models::Omni(), B, 0.1, 5.0, 0.1, 1.0, nb, 1000, 100, Rinv,
                                               vec({ -1.0, -1.0, -2.0 }), vec({ 1.0, 1.0, 2.0 }));
  };
  auto full = make_ctl(), rows = make_ctl();
  std::vector<Grid> grids = { make_grid(0, 120, 200, 0.05, 0.0, 0.0), make_grid(1, 80, 61, 0.1, -8.35, -13.95),
                              make_grid(2, 37, 150, 0.1, 3.0, -2.0) };
  b200::DeviceGridBatch grid_batch(grids);
  b200::setMapTargets(rows, grid_batch);  // first derivation: whole maps
  // steps of (first row, rows) per map; a band of 0 rows leaves the map as it is
  const unsigned bands[4][3][2] = { { { 70, 3 }, { 0, 0 }, { 149, 1 } },
                                    { { 0, 200 }, { 10, 51 }, { 0, 0 } },
                                    { { 127, 2 }, { 60, 1 }, { 63, 66 } },
                                    { { 199, 1 }, { 0, 61 }, { 64, 64 } } };
  int mismatches = 0;
  for (unsigned step = 0; step < 4; step++)
  {
    std::vector<std::vector<signed char>> band(B);
    std::vector<unsigned> rb(B), rc(B);
    for (unsigned i = 0; i < B; i++)
    {
      Grid& g = grids[i];
      rb[i] = bands[step][i][0];
      rc[i] = bands[step][i][1];
      for (unsigned r = rb[i]; r < rb[i] + rc[i]; r++)
        for (unsigned j = 0; j < g.xs; j++) g.data[size_t(r) * g.xs + j] = cell_value(r, j, i, step + 1);
      const signed char* src = reinterpret_cast<const signed char*>(g.data.data()) + size_t(rb[i]) * g.xs;
      band[i].assign(src, src + size_t(rc[i]) * g.xs);
    }
    grid_batch.updateRows(band, rb);
    b200::setMapTargets(rows, grid_batch, &rb, &rc);
    full.setMapTargets(grids);
    std::vector<double> pa(size_t(K) * B), pb(size_t(K) * B), ea(2 * B), eb(2 * B);
    b200::check(eb_get_phik_batch(full.handle(), pa.data(), ea.data()));
    b200::check(eb_get_phik_batch(rows.handle(), pb.data(), eb.data()));
    const bool same = std::memcmp(pa.data(), pb.data(), sizeof(double) * pa.size()) == 0 &&
                      std::memcmp(ea.data(), eb.data(), sizeof(double) * ea.size()) == 0;
    std::printf("step %u %s\n", step, same ? "equal" : "DIFFERENT");
    mismatches += same ? 0 : 1;
  }
  if (mismatches) return 1;
  std::printf("OK\n");
  return 0;
}

// Drop-in demonstration: the pipeline of /root/reference/examples/embedder.cpp:213-228 (Galerkin
// coarse graphs -> timed partition::embed -> NaN check) written against the reference's own
// interface, compiled against graph-embed_b200's headers and linked with libgraphembed_b200.so.
// The only source-level difference from a reference build is the include directory.
#include <cassert>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <string>

#include "embed.hpp"
#include "export.hpp"

namespace {

// nx x ny 4-neighbour grid (BASELINE config 1 uses 100 x 100)
SparseMatrix grid(int nx, int ny) {
  linalgcpp::CooMatrix<double> coo(nx * ny, nx * ny);
  for (int x = 0; x < nx; ++x)
    for (int y = 0; y < ny; ++y) {
      const int v = x * ny + y;
      if (x + 1 < nx) { coo.Add(v, v + ny, 1.0); coo.Add(v + ny, v, 1.0); }
      if (y + 1 < ny) { coo.Add(v, v + 1, 1.0); coo.Add(v + 1, v, 1.0); }
    }
  return coo.ToSparse();
}

// Aggregates of 2 x 2 cells: a stand-in for partition::partition, which stays on the host and
// is an input to the hot path.
SparseMatrix blocks(int nx, int ny) {
  const int bx = (nx + 1) / 2, by = (ny + 1) / 2;
  linalgcpp::CooMatrix<double> coo(bx * by, nx * ny);
  for (int x = 0; x < nx; ++x)
    for (int y = 0; y < ny; ++y) coo.Add((x / 2) * by + (y / 2), x * ny + y, 1.0);
  return coo.ToSparse();
}

}  // namespace

// `--gpus N`: partition::forceAtlas (include/forceatlas.hpp:89-305) on a 200 x 200 grid, sharded
// over N GPUs of this box by the library (one process, NCCL inside the context).
int flat_on_gpus(int gpus, int dimension) {
  ge_b200::options().gpus = gpus;
  ge_b200::options().seed = 7;
  const SparseMatrix A = grid(200, 200);
  std::vector<std::vector<double>> coords(0);
  linalgcpp::Timer timer(linalgcpp::Timer::Start::True);
  partition::forceAtlas(A, dimension, coords, 20);
  timer.Click();
  std::cout << "forceAtlas: " << A.Rows() << " vertices, 20 iterations on "
            << ge_context_device_count(ge_b200::default_context()) << " GPU(s) in " << timer[0] << "s"
            << std::endl;
  double sum = 0.0;
  for (size_t i = 0; i < coords.size(); i++)
    for (int k = 0; k < dimension; k++) {
      if (std::isnan(coords[i][k])) return 1;
      sum += coords[i][k];
    }
  std::cout.precision(17);
  std::cout << "checksum " << sum << std::endl;
  return 0;
}

// `--coarsen`: graph -> hierarchy built on the device (ge_b200::coarsen) -> partition::embed.
int coarsen_then_embed(int nx, int dimension) {
  ge_b200::options().seed = 3;
  std::vector<SparseMatrix> As;
  linalgcpp::Timer timer(linalgcpp::Timer::Start::True);
  const std::vector<SparseMatrix> hierarchy = ge_b200::coarsen(grid(nx, nx), 0.25, 64, &As);
  timer.Click();
  std::cout << "coarsen: " << hierarchy.size() << " levels in " << timer[0] << "s:";
  for (const auto& A : As) std::cout << " " << A.Rows();
  std::cout << std::endl;
  linalgcpp::Timer t2(linalgcpp::Timer::Start::True);
  std::vector<std::vector<double>> coords = partition::embed(As, hierarchy, dimension);
  t2.Click();
  std::cout << "embedded! in time " << t2[0] << "s" << std::endl;
  for (size_t i = 0; i < coords.size(); i++)
    for (int k = 0; k < dimension; k++)
      if (std::isnan(coords[i][k])) {
        std::cerr << "NaN at vertex " << i << std::endl;
        return 1;
      }
  return coords.size() == static_cast<size_t>(nx) * nx ? 0 : 2;
}

// `--layout`: a grid with isolated vertices and a small second component appended, laid out in one
// call (ge_b200::layout: largest component -> hierarchy -> embed, on the device).
int layout_raw_graph(int nx, int dimension) {
  ge_b200::options().seed = 3;
  const int g = nx * nx, isolated = 50, tail = 10, n = g + isolated + tail;
  const SparseMatrix G = grid(nx, nx);
  linalgcpp::CooMatrix<double> coo(n, n);
  for (int i = 0; i < G.Rows(); ++i)
    for (int e = G.GetIndptr()[i]; e < G.GetIndptr()[i + 1]; ++e) coo.Add(i, G.GetIndices()[e], 1.0);
  for (int v = g + isolated; v + 1 < n; ++v) {  // a path of `tail` vertices
    coo.Add(v, v + 1, 1.0);
    coo.Add(v + 1, v, 1.0);
  }
  const SparseMatrix A = coo.ToSparse();
  std::vector<int> vertices;
  ge_layout_stats stats;
  linalgcpp::Timer timer(linalgcpp::Timer::Start::True);
  std::vector<std::vector<double>> coords = ge_b200::layout(A, dimension, 0.25, 64, &vertices, &stats);
  timer.Click();
  std::cout << "layout: " << vertices.size() << " of " << n << " vertices kept (" << stats.components
            << " components), " << stats.levels << " levels" << std::endl;
  std::cout << "embedded! in time " << timer[0] << "s" << std::endl;
  for (size_t i = 0; i < coords.size(); i++)
    for (int k = 0; k < dimension; k++)
      if (std::isnan(coords[i][k])) {
        std::cerr << "NaN at vertex " << vertices[i] << std::endl;
        return 1;
      }
  return coords.size() == static_cast<size_t>(g) && vertices.back() == g - 1 ? 0 : 2;
}

// `--edges`: a grid's edge list with every edge listed twice (once reversed), self-loops and real
// weights.  ge_b200::fromEdges must equal linalgcpp's CooMatrix built from the same calls, bit for
// bit; then the edge list is laid out in one call (ge_b200::layoutEdges).
int layout_edge_list(int nx, int dimension) {
  ge_b200::options().seed = 3;
  const int n = nx * nx;
  std::vector<int> src, dst;
  std::vector<double> w;
  auto edge = [&](int a, int b, double x) {
    src.push_back(a);
    dst.push_back(b);
    w.push_back(x);
  };
  for (int x = 0; x < nx; ++x)
    for (int y = 0; y < nx; ++y) {
      const int v = x * nx + y;
      // weights that round differently depending on the order they are added in
      if (x + 1 < nx) {
        edge(v, v + nx, 1.0 + v * 1e-3);
        edge(v + nx, v, 1e-17 * (y + 1));
      }
      if (y + 1 < nx) {
        edge(v, v + 1, 0.1 * (x + 1));
        edge(v + 1, v, 0.7);
      }
      if (v % 7 == 0) edge(v, v, 2.0);
    }
  ge_edges_options opt;
  ge_edges_options_default(&opt);
  linalgcpp::CooMatrix<double> coo(n, n);
  for (size_t e = 0; e < src.size(); ++e) {
    if (src[e] == dst[e]) continue;
    coo.Add(src[e], dst[e], w[e]);
    coo.Add(dst[e], src[e], w[e]);
  }
  const SparseMatrix ref = coo.ToSparse();
  const SparseMatrix A = ge_b200::fromEdges(n, src, dst, &w, &opt);
  if (A.GetIndptr() != ref.GetIndptr() || A.GetIndices() != ref.GetIndices() ||
      A.GetData().size() != ref.GetData().size() ||
      std::memcmp(A.GetData().data(), ref.GetData().data(), sizeof(double) * ref.GetData().size()) != 0) {
    std::cerr << "fromEdges differs from CooMatrix::ToSparse()" << std::endl;
    return 3;
  }
  std::cout << "fromEdges: " << src.size() << " edges -> " << A.GetIndices().size()
            << " entries, equal to CooMatrix" << std::endl;
  std::vector<int> vertices;
  ge_layout_stats stats;
  linalgcpp::Timer timer(linalgcpp::Timer::Start::True);
  std::vector<std::vector<double>> coords =
      ge_b200::layoutEdges(n, src, dst, &w, dimension, 0.25, 64, &vertices, &opt, &stats);
  timer.Click();
  std::cout << "layoutEdges: " << vertices.size() << " vertices, " << stats.levels << " levels" << std::endl;
  std::cout << "embedded! in time " << timer[0] << "s" << std::endl;
  for (size_t i = 0; i < coords.size(); i++)
    for (int k = 0; k < dimension; k++)
      if (std::isnan(coords[i][k])) {
        std::cerr << "NaN at vertex " << vertices[i] << std::endl;
        return 1;
      }
  return coords.size() == static_cast<size_t>(n) ? 0 : 2;
}

int main(int argc, char** argv) {
  std::string outdir;  // --out DIR: write the layout and the plot inputs like examples/embedder.cpp:230-289
  bool coarsen = false, layout = false, edges = false;
  for (int a = 1; a < argc; ++a) {
    if (a + 1 < argc && std::string(argv[a]) == "--gpus") return flat_on_gpus(std::atoi(argv[a + 1]), 2);
    if (a + 1 < argc && std::string(argv[a]) == "--out") outdir = argv[a + 1];
    if (std::string(argv[a]) == "--coarsen") coarsen = true;
    if (std::string(argv[a]) == "--layout") layout = true;
    if (std::string(argv[a]) == "--edges") edges = true;
  }
  int nx = argc > 1 ? std::atoi(argv[1]) : 64, ny = nx;
  const int dimension = argc > 2 ? std::atoi(argv[2]) : 2;
  if (coarsen) return coarsen_then_embed(nx, dimension);
  if (layout) return layout_raw_graph(nx, dimension);
  if (edges) return layout_edge_list(nx, dimension);
  std::vector<SparseMatrix> As = {grid(nx, ny)}, hierarchy;
  while (nx * ny > 40) {
    hierarchy.push_back(blocks(nx, ny));
    const SparseMatrix& P = hierarchy.back();
    As.push_back(P.Mult(As.back()).Mult(P.Transpose()));  // examples/embedder.cpp:215
    // the same product on the device (ge_galerkin) must give the same matrix, entry for entry
    const SparseMatrix G = ge_b200::galerkin(As[As.size() - 2], P);
    if (G.GetIndptr() != As.back().GetIndptr() || G.GetIndices() != As.back().GetIndices() ||
        G.GetData() != As.back().GetData()) {
      std::cerr << "device Galerkin product differs from P.Mult(A).Mult(P.Transpose())" << std::endl;
      return 3;
    }
    nx = (nx + 1) / 2;
    ny = (ny + 1) / 2;
  }
  std::cout << "levels:";
  for (const auto& A : As) std::cout << " " << A.Rows();
  std::cout << std::endl << "starting embedding: " << std::endl;
  linalgcpp::Timer timer(linalgcpp::Timer::Start::True);
  std::vector<std::vector<double>> coords = partition::embed(As, hierarchy, dimension);
  timer.Click();
  std::cout << "embedded! in time " << timer[0] << "s" << std::endl;
  for (size_t i = 0; i < coords.size(); i++)
    for (int k = 0; k < dimension; k++)
      if (std::isnan(coords[i][k])) {  // examples/embedder.cpp:224-228
        std::cerr << "NaN at vertex " << i << std::endl;
        return 1;
      }
  // the plugin interface (include/embed.hpp:40-49) with the B200 solver as the functor
  std::vector<std::vector<double>> via =
      partition::embedVia(As, hierarchy, dimension, partition::forceAtlasMultilevelEmbedder());
  if (via.size() != coords.size()) return 2;
  std::cout << "embedVia ok: " << via.size() << " vertices" << std::endl;
  if (!outdir.empty()) {
    partition::writeCoords(coords, outdir + "/coords.txt");  // include/export.hpp:23
    ge_b200::writePlotInputs(As[0], hierarchy, coords, dimension, outdir + "/part.temp",
                             outdir + "/coords.temp", outdir + "/mat.temp");
    std::cout << "wrote " << outdir << "/{coords.txt,part.temp,coords.temp,mat.temp}" << std::endl;
  }
  return 0;
}

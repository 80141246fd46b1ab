// graph-embed_b200 drop-in :: glue between the reference's C++ types and the C ABI.
#ifndef GE_B200_RUNTIME_HPP
#define GE_B200_RUNTIME_HPP

#include <algorithm>
#include <cstdlib>
#include <stdexcept>
#include <string>
#include <vector>

#include "graph_embed_b200.h"
#include "matrixutils.hpp"

namespace ge_b200 {

// Knobs the reference does not have (precision, seed, GPU count); change before the first call
// into the library (the GPU count is read once, when the process-wide context is created).
struct Options {
  int precision = GE_F64;
  unsigned seed = 0;   // 0: std::random_device like the reference
  bool verbose = true; // print the reference's "embedding layer N" progress lines
  int gpus = 0;        // 0: the environment variable GE_GPUS, else 1.  > 1: partition::forceAtlas on
                       // graphs of >= 32768 vertices is sharded over that many GPUs of the box
};
inline Options& options() {
  static Options o;
  return o;
}

// Process-wide context (the reference keeps no state either; the context only owns streams, the
// device memory pools and, with several GPUs, the NCCL communicator).
inline ge_context* default_context() {
  struct Holder {
    ge_context* ctx = nullptr;
    Holder() {
      int gpus = options().gpus;
      if (gpus <= 0) {
        const char* e = std::getenv("GE_GPUS");
        gpus = e ? std::atoi(e) : 1;
      }
      const ge_status st = gpus > 1 ? ge_context_create_multi(gpus, nullptr, &ctx)
                                    : ge_context_create(-1, nullptr, &ctx);
      if (st != GE_OK) throw std::runtime_error(std::string("graph-embed_b200: ") + ge_last_error());
    }
    ~Holder() { ge_context_destroy(ctx); }
  };
  static Holder h;
  return h.ctx;
}

// The reference reports problems through assert() only (src/embed.cpp:564-570); the drop-in
// throws instead of continuing with garbage, because there is no CPU path to fall back to.
inline void check(ge_status st) {
  if (st != GE_OK) throw std::runtime_error(std::string("graph-embed_b200: ") + ge_last_error());
}

inline ge_csr view(const SparseMatrix& A) {
  ge_csr c;
  c.rows = A.Rows();
  c.cols = A.Cols();
  c.nnz = static_cast<int64_t>(A.GetIndices().size());
  c.indptr = A.GetIndptr().data();
  c.indices = A.GetIndices().data();
  c.data = A.GetData().data();
  return c;
}

inline std::vector<double> flatten(const std::vector<std::vector<double>>& c, int d) {
  std::vector<double> x(c.size() * static_cast<size_t>(d));
  for (size_t i = 0; i < c.size(); ++i)
    for (int k = 0; k < d; ++k) x[i * d + k] = c[i][k];
  return x;
}

inline std::vector<std::vector<double>> unflatten(const std::vector<double>& x, int n, int d) {
  std::vector<std::vector<double>> c(n, std::vector<double>(d));
  for (int i = 0; i < n; ++i)
    for (int k = 0; k < d; ++k) c[i][k] = x[static_cast<size_t>(i) * d + k];
  return c;
}

// A_{l+1} = P_T * A_l * P_T^T on the device: the line every caller of partition::embed writes as
//   As.push_back(P.Mult(As.back()).Mult(P.Transpose()));   (examples/embedder.cpp:213-216)
// becomes  As.push_back(ge_b200::galerkin(As.back(), P));
inline SparseMatrix galerkin(const SparseMatrix& A, const SparseMatrix& P_T) {
  const ge_csr a = view(A), p = view(P_T);
  std::vector<int> indptr(static_cast<size_t>(P_T.Rows()) + 1), indices(A.GetIndices().size());
  std::vector<double> data(A.GetIndices().size());
  int64_t nnz = 0;
  check(ge_galerkin(default_context(), &a, &p, indptr.data(), indices.data(), data.data(),
                    static_cast<int64_t>(indices.size()), &nnz, nullptr));
  indices.resize(static_cast<size_t>(nnz));
  data.resize(static_cast<size_t>(nnz));
  return SparseMatrix(std::move(indptr), std::move(indices), std::move(data), P_T.Rows(), P_T.Rows());
}

// The multilevel hierarchy built on the device (ge_coarsen: random-mate matching, NOT the
// reference's partitioner).  Returns the P_T of every level, the shape partition::partition
// returns; As (when not null) receives the graphs {A, A_1, ..., A_L}, ready for partition::embed.
inline std::vector<SparseMatrix> coarsen(const SparseMatrix& A, double coarseningFactor, int minCoarse,
                                         std::vector<SparseMatrix>* As = nullptr) {
  const ge_csr a = view(A);
  ge_coarsen_options opt;
  ge_coarsen_options_default(&opt);
  opt.coarsening_factor = coarseningFactor;
  opt.min_coarse = minCoarse;
  opt.seed = options().seed;
  ge_hierarchy* h = nullptr;
  check(ge_coarsen(default_context(), &a, &opt, &h, nullptr));
  struct Owner {
    ge_hierarchy* h;
    ~Owner() { ge_hierarchy_destroy(h); }
  } owner{h};
  auto copy = [](const ge_csr& c) {
    const int64_t nnz = c.nnz;
    return SparseMatrix(std::vector<int>(c.indptr, c.indptr + c.rows + 1),
                        std::vector<int>(c.indices, c.indices + nnz), std::vector<double>(c.data, c.data + nnz),
                        c.rows, c.cols);
  };
  const int L = ge_hierarchy_levels(h);
  std::vector<SparseMatrix> P_Ts;
  if (As) {
    As->clear();
    As->push_back(A);
  }
  for (int l = 0; l < L; ++l) {
    ge_csr c;
    check(ge_hierarchy_aggregation(h, l, &c));
    P_Ts.push_back(copy(c));
    if (As) {
      check(ge_hierarchy_graph(h, l + 1, &c));
      As->push_back(copy(c));
    }
  }
  return P_Ts;
}

// examples/embedder.cpp:156 (largestComponent) on the device: the largest connected component of
// A; vertices (when not null) receives the original id of each of its rows.
inline SparseMatrix largestComponent(const SparseMatrix& A, std::vector<int>* vertices = nullptr) {
  const ge_csr a = view(A);
  const size_t n = static_cast<size_t>(A.Rows());
  std::vector<int> vert(n), indptr(n + 1), indices(A.GetIndices().size());
  std::vector<double> data(A.GetIndices().size());
  int32_t k = 0;
  int64_t nnz = 0;
  check(ge_largest_component(default_context(), &a, vert.data(), &k, indptr.data(), indices.data(), data.data(),
                             static_cast<int64_t>(indices.size()), &nnz, nullptr));
  vert.resize(static_cast<size_t>(k));
  indptr.resize(static_cast<size_t>(k) + 1);
  indices.resize(static_cast<size_t>(nnz));
  data.resize(static_cast<size_t>(nnz));
  if (vertices) *vertices = vert;
  return SparseMatrix(std::move(indptr), std::move(indices), std::move(data), k, k);
}

// A graph in, coordinates out: its largest component, the device-built hierarchy (ge_coarsen) and
// partition::embed in one call (ge_layout_graph).  Row i of the result is the vertex (*vertices)[i]
// of A; stats (when not null) receives the call's counters.
inline std::vector<std::vector<double>> layout(const SparseMatrix& A, int d, double coarseningFactor,
                                               int minCoarse, std::vector<int>* vertices = nullptr,
                                               ge_layout_stats* stats = nullptr) {
  const ge_csr a = view(A);
  ge_coarsen_options copt;
  ge_coarsen_options_default(&copt);
  copt.coarsening_factor = coarseningFactor;
  copt.min_coarse = minCoarse;
  copt.seed = options().seed;
  ge_embed_options eopt;
  ge_embed_options_default(&eopt);
  eopt.precision = options().precision;
  eopt.seed = options().seed;
  eopt.verbose = options().verbose;
  const size_t n = static_cast<size_t>(A.Rows());
  std::vector<double> x(n * static_cast<size_t>(d));
  std::vector<int> vert(n);
  int32_t k = 0;
  check(ge_layout_graph(default_context(), &a, d, 1, &copt, &eopt, x.data(), vert.data(), &k, stats));
  vert.resize(static_cast<size_t>(k));
  if (vertices) *vertices = vert;
  x.resize(static_cast<size_t>(k) * d);
  return unflatten(x, k, d);
}

// An edge list -> the SparseMatrix that linalgcpp's CooMatrix builds from it (ge_graph_from_edges):
// Add(src[e], dst[e], w) for every edge, and Add(dst[e], src[e], w) too when symmetrising; duplicates
// summed in that order; self-loops dropped unless edgeOptions->keep_self_loops.  weights null: 1.0;
// edgeOptions null: symmetrise, drop self-loops, sum the weights.
inline SparseMatrix fromEdges(int n, const std::vector<int>& src, const std::vector<int>& dst,
                              const std::vector<double>* weights = nullptr,
                              const ge_edges_options* edgeOptions = nullptr) {
  if (src.size() != dst.size() || (weights && weights->size() != src.size()))
    throw std::invalid_argument("graph-embed_b200: edge arrays differ in length");
  const int64_t E = static_cast<int64_t>(src.size());
  const bool sym = edgeOptions ? edgeOptions->symmetrize != 0 : true;
  const size_t cap = static_cast<size_t>(std::max<int64_t>(E * (sym ? 2 : 1), 1));
  std::vector<int> indptr(static_cast<size_t>(n) + 1), indices(cap);
  std::vector<double> data(cap);
  int64_t nnz = 0;
  check(ge_graph_from_edges(default_context(), n, E, src.data(), dst.data(), weights ? weights->data() : nullptr,
                            edgeOptions, indptr.data(), indices.data(), data.data(), static_cast<int64_t>(cap), &nnz,
                            nullptr));
  indices.resize(static_cast<size_t>(nnz));
  data.resize(static_cast<size_t>(nnz));
  return SparseMatrix(std::move(indptr), std::move(indices), std::move(data), n, n);
}

// ge_b200::layout from an edge list (ge_layout_edges): the graph fromEdges would return is built on
// the device and laid out there without crossing PCIe.
inline std::vector<std::vector<double>> layoutEdges(int n, const std::vector<int>& src, const std::vector<int>& dst,
                                                    const std::vector<double>* weights, int d,
                                                    double coarseningFactor, int minCoarse,
                                                    std::vector<int>* vertices = nullptr,
                                                    const ge_edges_options* edgeOptions = nullptr,
                                                    ge_layout_stats* stats = nullptr) {
  if (src.size() != dst.size() || (weights && weights->size() != src.size()))
    throw std::invalid_argument("graph-embed_b200: edge arrays differ in length");
  ge_coarsen_options copt;
  ge_coarsen_options_default(&copt);
  copt.coarsening_factor = coarseningFactor;
  copt.min_coarse = minCoarse;
  copt.seed = options().seed;
  ge_embed_options eopt;
  ge_embed_options_default(&eopt);
  eopt.precision = options().precision;
  eopt.seed = options().seed;
  eopt.verbose = options().verbose;
  const size_t nn = static_cast<size_t>(std::max(n, 0));
  std::vector<double> x(nn * static_cast<size_t>(d));
  std::vector<int> vert(nn);
  int32_t k = 0;
  check(ge_layout_edges(default_context(), n, static_cast<int64_t>(src.size()), src.data(), dst.data(),
                        weights ? weights->data() : nullptr, edgeOptions, d, 1, &copt, &eopt, x.data(), vert.data(), &k,
                        nullptr, stats));
  vert.resize(static_cast<size_t>(k));
  if (vertices) *vertices = vert;
  x.resize(static_cast<size_t>(k) * d);
  return unflatten(x, k, d);
}

}  // namespace ge_b200

#endif

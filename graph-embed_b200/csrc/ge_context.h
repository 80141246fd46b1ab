// graph-embed_b200 :: context, device buffers, host-side helpers shared by the .cu files.
#ifndef GE_CONTEXT_H
#define GE_CONTEXT_H

#include <cuda_runtime.h>

#include <chrono>
#include <cstddef>
#include <cstdint>
#include <memory>
#include <vector>

#include "ge_common.cuh"

namespace ge {
struct Stager;      // pinned staging ring for large host->device copies (ge_capi.cu)
struct MultiState;  // sub-contexts of the other devices + NCCL communicator (ge_multi.cu)
}

struct ge_context {
  ge::Stager* stager = nullptr;
  // second stream + staging ring: ge_embed uploads the level graphs on it from a helper thread
  // while the coarsest-level solve occupies the main stream
  cudaStream_t copy_stream = nullptr;
  ge::Stager* stager2 = nullptr;
  int device = 0;
  int sm_count = 0;
  size_t smem_optin = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  int64_t launches = 0;
  double h2d_bytes = 0, d2h_bytes = 0;
  // device time of the large-aggregate (multi-CTA) tier of the per-aggregate solver, accumulated
  // over the levels of one ge_embed call (CUDA events on the context stream)
  double grid_tier_ms = 0;
  double radii_ms = 0;  // device time of the ball-radius / rescale kernels
  ge::MultiState* multi = nullptr;  // ge_context_create_multi: this context drives several devices
};

namespace ge {

inline double now_ms() {
  return std::chrono::duration<double, std::milli>(
             std::chrono::steady_clock::now().time_since_epoch())
      .count();
}

// Host -> device copy on the context stream.  Large copies from pageable caller memory go through
// a ring of pinned buffers filled by a few host threads (the driver's own pageable path is
// single-threaded, ~12 GB/s on this box; the staged path overlaps four memcpy streams with the DMA).
void host_to_device(ge_context* ctx, void* dst, const void* src, size_t bytes);

// Owning device allocation from the stream-ordered memory pool of the context's device
// (cudaMallocAsync / cudaFreeAsync on the context stream; the pool's release threshold is raised at
// context creation so that repeated solves reuse memory instead of paying cudaMalloc / cudaFree,
// which cost milliseconds and synchronise the device).  Movable, not copyable.
template <typename T>
class DevBuf {
 public:
  DevBuf() = default;
  DevBuf(ge_context* ctx, size_t n) { alloc(ctx, n); }
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : p_(o.p_), n_(o.n_), stream_(o.stream_) { o.p_ = nullptr; o.n_ = 0; }
  DevBuf& operator=(DevBuf&& o) noexcept {
    if (this != &o) {
      release();
      p_ = o.p_;
      n_ = o.n_;
      stream_ = o.stream_;
      o.p_ = nullptr;
      o.n_ = 0;
    }
    return *this;
  }
  ~DevBuf() { release(); }
  void alloc(ge_context* ctx, size_t n) {
    release();
    n_ = n;
    stream_ = ctx->stream;
    if (n) GE_CUDA(cudaMallocAsync(&p_, n * sizeof(T), stream_));
  }
  void release() {
    if (p_) cudaFreeAsync(p_, stream_);
    p_ = nullptr;
    n_ = 0;
  }
  void zero(cudaStream_t s) {
    if (n_) GE_CUDA(cudaMemsetAsync(p_, 0, n_ * sizeof(T), s));
  }
  void upload(ge_context* ctx, const T* host, size_t n) {
    if (n) host_to_device(ctx, p_, host, n * sizeof(T));
    ctx->h2d_bytes += double(n * sizeof(T));
  }
  void download(ge_context* ctx, T* host, size_t n) const {
    if (n) GE_CUDA(cudaMemcpyAsync(host, p_, n * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
    ctx->d2h_bytes += double(n * sizeof(T));
  }
  T* get() const { return p_; }
  size_t size() const { return n_; }

 private:
  T* p_ = nullptr;
  size_t n_ = 0;
  cudaStream_t stream_ = nullptr;
};

// ---- ge_flat.cu ------------------------------------------------------------------------------
// Type-erased device-resident flat solver (rows [row_begin,row_end) of one graph).
class FlatSolver {
 public:
  virtual ~FlatSolver() {}
  virtual int64_t ld() const = 0;
  virtual int elem_size() const = 0;
  virtual void bind_coords(void* b0, void* b1) = 0;
  virtual void upload_coords(const double* aos) = 0;
  virtual void download_coords(double* aos) = 0;
  virtual void download_forces(double* aos) = 0;  // owned rows x dim (forces_prev)
  virtual void* cur_coords() = 0;
  virtual void* next_coords() = 0;
  virtual void launch_iteration(bool update) = 0;  // = launch_repulsion + launch_step
  virtual void launch_repulsion() = 0;
  virtual void launch_step(bool update) = 0;
  // symmetric sweep (ge_flat_sym.cu): raw pair sums [dim][ld]; a multi-rank caller binds its own
  // buffer and adds the ranks' sums between launch_repulsion and launch_step
  virtual bool symmetric() const = 0;
  virtual void bind_pair_sums(void* full) = 0;
  virtual void* pair_sums() = 0;
  virtual void swap() = 0;
  virtual void normalize() = 0;  // include/forceatlas.hpp:272-303 (single rank)
  virtual void select_kernels(int mask) = 0;
  virtual void profile(bool enable) = 0;
  virtual void profile_get(double* rep_ms, int64_t* rep_n, double* step_ms, int64_t* step_n) = 0;
  ge_context* ctx = nullptr;
};
// part / parts: rank of a symmetric multi-rank solve (rows must be that rank's row block)
// shared_deg: the row sums of every row (flat_degrees), computed once by a caller that builds
// several plans of the same graph; nullptr: the plan computes them
FlatSolver* make_flat_solver(ge_context* ctx, const ge_csr& A, int dim, const ge_params& p,
                             int row_begin, int row_end, int part = 0, int parts = 1,
                             const double* shared_deg = nullptr);
void flat_degrees(const ge_csr& A, const ge_params& p, std::vector<double>& deg);

// ---- ge_onchip.cu ----------------------------------------------------------------------------
// Small flat solve entirely inside one CTA (coarsest level: n ~ 30-100, 100 000 iterations).
constexpr int kOnchipMaxThreads = 1024;
constexpr int kOnchipMaxVertices = 1024;
void onchip_flat_solve(ge_context* ctx, const ge_csr& A, int dim, const ge_params& p,
                       double* coords /* n x dim in/out */, double* forces_out /* or null */,
                       bool forces_only, DevBuf<double>* keep_on_device = nullptr /* [n][dim]: no download */);

// ---- ge_multilevel.cu ------------------------------------------------------------------------
// A level graph already on the device (uploaded ahead of time on another stream); `ready` is
// recorded after the last copy.
struct LevelLayout;  // slot layout of a level (ge_multilevel.cu): depends on P_T only
LevelLayout* make_level_layout(ge_context* ctx, const ge_csr& P_T, int n, int agg_begin = 0,
                               int agg_end = -1, bool members = true,
                               const std::vector<int>* owned = nullptr);
void free_level_layout(LevelLayout* layout);
struct PrefetchedGraph {
  DevBuf<int> I, J;
  DevBuf<double> Dw;  // empty when A.data == nullptr
  LevelLayout* layout = nullptr;
  cudaEvent_t ready = nullptr;
  ~PrefetchedGraph() {
    if (ready) cudaEventDestroy(ready);
    free_level_layout(layout);
  }
};
// Device-resident inputs / outputs of one level (ge_embed keeps the coordinates on the device
// between the levels): when d_coords_A / d_r_A are set the host pointers coords_A / r_A of
// multilevel_solve are ignored; keep_out receives the level's coordinates [n][dim]; download =
// false skips the copy to coords_out.
struct LevelIO {
  const double* d_coords_A = nullptr;
  const double* d_r_A = nullptr;
  DevBuf<double>* keep_out = nullptr;
  bool download = true;
  const std::vector<int>* owned = nullptr;  // solve exactly these aggregates (overrides the range)
};
void multilevel_solve(ge_context* ctx, const ge_csr& A, const ge_csr& P_T, const int32_t* v_A,
                      const double* coords_A, const double* r_A, const double* init,
                      double* coords_out, int dim, const ge_params& p, bool forces_only,
                      double* pairs_out, int agg_begin = 0, int agg_end = -1,
                      const PrefetchedGraph* pre = nullptr, const LevelIO* io = nullptr);

// ---- ge_radii.cu --------------------------------------------------------------------------------
// Ball radii + rescale on the device (src/embed.cpp:615-778).  d_x [m][dim] in/out, d_r [m] out.
// lv == nullptr: base case (all pairs of the m vertices, :616-679).  Otherwise the general case
// (:680-777): lv describes the level whose m vertices these are -- its graph (I, J), the vertex ->
// family map `parent`, the families' member lists (PI, PJ: the CSR of its aggregation, mc rows) --
// and d_xc [mc][dim] / d_rc [mc] are the centres and radii of the families' balls.
constexpr int kRadiiBaseMax = 4096;
struct RadiiLevel {
  const int* I;
  const int* J;
  const int* parent;
  const int* PI;
  const int* PJ;
  int mc;
};
void level_radii_device(ge_context* ctx, int m, int dim, double* d_x, double* d_r,
                        const RadiiLevel* lv, const double* d_xc, const double* d_rc);
// The RadiiLevel view of a level whose graph and slot layout are on the device.
RadiiLevel radii_level_of(const PrefetchedGraph& g, int mc);

// ---- ge_galerkin.cu ----------------------------------------------------------------------------
int64_t galerkin(ge_context* ctx, const ge_csr& A, const ge_csr& P_T, int32_t* c_indptr,
                 int32_t* c_indices, double* c_data, int64_t capacity, ge_galerkin_stats* stats);
// A graph and its aggregation already on the device (every pointer is a device pointer).
// Segment a of the product is the entries of the rows of aggregate a's members, in P_T order:
// segoff [m+1] = first entry of each segment, rowoff [n] = offset of row i inside its segment.
struct GalerkinInput {
  int n = 0, m = 0;
  const int* I = nullptr;
  const int* J = nullptr;
  const double* W = nullptr;  // nullptr: unit weights
  const int* vA = nullptr;    // vertex -> aggregate [n]
  const int* Pptr = nullptr;  // P_T.indptr [m+1]
  const int* Pidx = nullptr;  // P_T.indices [n]
  const int* rowoff = nullptr;
  const int* segoff = nullptr;
};
// The product on the device.  segoff_host: host copy of in.segoff (the size classes of the segments
// are sorted out on the host).  outptr receives the row pointers [m+1]; when nnz(A_c) <= capacity,
// outcol / outval receive the columns and values.  c_indptr (host, may be null) receives a copy of
// the row pointers.  Returns nnz(A_c) (synchronises the stream once); stats: the segment counts and
// nnz_out only.  start (optional) is recorded after the size classes are uploaded, just before the
// first kernel.
int64_t galerkin_device(ge_context* ctx, const GalerkinInput& in, const int* segoff_host,
                        int32_t* c_indptr, DevBuf<int>& outptr, DevBuf<int>& outcol,
                        DevBuf<double>& outval, int64_t capacity, ge_galerkin_stats* stats,
                        cudaEvent_t start = nullptr);
// Exclusive prefix sum of d_in [n] into d_out [n+1] (d_out[n] = total), on the context stream.
void exclusive_scan(ge_context* ctx, const int* d_in, int n, int* d_out);

// ---- ge_coarsen.cu ---------------------------------------------------------------------------
// Builds the hierarchy of ge_coarsen (include/graph_embed_b200.h) on the context's device.
struct HostHierarchy {
  struct Csr {
    int rows = 0, cols = 0;
    std::vector<int> indptr, indices;
    std::vector<double> data;
  };
  std::vector<Csr> graphs;  // As[1..L]
  std::vector<Csr> aggs;    // P_T[0..L-1]
};
void coarsen(ge_context* ctx, const ge_csr& A, const ge_coarsen_options& opt, HostHierarchy& out,
             ge_coarsen_stats* stats);
void check_coarsen_options(const ge_coarsen_options& opt);

// A square CSR graph on the device.
struct DevGraph {
  int n = 0, nnz = 0;
  DevBuf<int> I, J;
  DevBuf<double> W;  // empty: unit weights
  const double* w() const { return W.size() ? W.get() : nullptr; }
};
struct DevAgg {  // P_T of one level: m aggregates of n vertices, members ascending per row
  int m = 0, n = 0;
  DevBuf<int> ptr, idx;
};
// The levels of ge_coarsen left on the device: graphs[0] is the input, graphs[l] = As[l].
struct DeviceHierarchy {
  std::vector<std::unique_ptr<DevGraph>> graphs;
  std::vector<std::unique_ptr<DevAgg>> aggs;
  int levels() const { return (int)aggs.size(); }
};
// A on the device (square; the arrays as given, no check of the entries).
void upload_graph(ge_context* ctx, const ge_csr& A, DevGraph& G);
// GE_ERR_INVALID unless G.I is ascending and every column lies in [0, n).
void check_graph(ge_context* ctx, const DevGraph& G);
// Builds the hierarchy of the graph h.graphs[0] into h (check: run check_graph first).
// rounds: matching rounds, all levels.
void coarsen_device(ge_context* ctx, DeviceHierarchy& h, const ge_coarsen_options& opt, bool check,
                    int64_t* rounds);

// ---- ge_components.cu ------------------------------------------------------------------------
// The largest weakly connected component of A (ties to the component with the smallest vertex) on
// the device.  Returns the number of components.  With more than one, out receives the subgraph
// A[vertices][:, vertices] (entry order kept, columns renumbered, weights copied; unit weights
// become ones) and vertices its original ids, ascending; with one, out and vertices stay empty.
int64_t largest_component_device(ge_context* ctx, const DevGraph& A, DevGraph& out, DevBuf<int>& vertices);
// Unit weights made explicit: G.W = ones when it is empty.
void unit_weights(ge_context* ctx, DevGraph& G);

// ---- ge_edges.cu -----------------------------------------------------------------------------
// GE_ERR_INVALID unless n and E are in range and the slots of E edges fit int32 row pointers.
void check_edges_args(int64_t n, int64_t E, const int32_t* src, const int32_t* dst, const ge_edges_options& opt);
// The graph of ge_graph_from_edges (include/graph_embed_b200.h) built on the device from host edge
// arrays (uploaded here).  out.W is always explicit.  stats: every field but total_ms.
void edges_to_graph_device(ge_context* ctx, int n, int64_t E, const int32_t* src, const int32_t* dst,
                           const double* w, const ge_edges_options& opt, DevGraph& out, ge_edges_stats* stats);

// ---- ge_multi.cu ---------------------------------------------------------------------------------
void multi_attach(ge_context* ctx, int ndev, const int* devices);
void multi_destroy(MultiState* m);
int multi_size(const ge_context* ctx);
void multi_flat_solve(ge_context* ctx, const ge_csr& A, int dim, double* coords, const ge_params& p);
ge_context* multi_device(ge_context* ctx, int r);  // sub-context of device r (0: ctx itself)
// bufs[r]: a buffer of `count` doubles on device r.  Enqueued on the devices' streams.
void multi_broadcast_f64(ge_context* ctx, const std::vector<double*>& bufs, size_t count, int root);
void multi_allreduce_sum_f64(ge_context* ctx, const std::vector<double*>& bufs, size_t count);
void multi_sync(ge_context* ctx);                // every device's stream
void multi_collect_counters(ge_context* ctx);    // fold the sub-contexts' counters into ctx

// ---- ge_capi.cu (host-side level driver) -------------------------------------------------------
void level_radii(int m, int dim, double* coords_A, double* r_A, const ge_csr* A_c,
                 const ge_csr* P_T_c, const double* coords_Ac, const double* r_Ac);
void reference_uniform(uint32_t seed, int64_t count, double* out);
void level_init_stream(uint32_t seed, const ge_csr& P_T, int dim, double* init_by_vertex);
uint32_t resolve_seed(uint32_t seed);

}  // namespace ge

#endif  // GE_CONTEXT_H

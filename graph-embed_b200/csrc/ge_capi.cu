// graph-embed_b200 :: the C ABI (include/graph_embed_b200.h) and the host-side level driver.
//
// Host logic restated here, from scratch, for the drop-in:
//   ge_embed        <- partition::embed / embedMultilevel, /root/reference/src/embed.cpp:561-796
//   level_radii     <- the ball-radius and rescale step, src/embed.cpp:615-778
//   reference_uniform <- the reference's generator, include/forceatlas.hpp:104-108
// Everything numerical that iterates runs on the device; there is no CPU fallback.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <memory>
#include <random>
#include <atomic>
#include <string>
#include <thread>
#include <tuple>
#include <vector>

#include "ge_context.h"
#include "ge_flat.cuh"

namespace ge {

static thread_local std::string g_error;
void set_error(const std::string& msg) { g_error = msg; }

// ---------------------------------------------------------------------------------------------
// staged host -> device copies
// ---------------------------------------------------------------------------------------------
struct Stager {
  static constexpr size_t kChunk = size_t(4) << 20;
  static constexpr int kThreads = 4, kSlotsPerThread = 2;
  void* pinned[kThreads * kSlotsPerThread] = {};
  cudaEvent_t ev[kThreads * kSlotsPerThread] = {};
  bool ok = false;
  Stager() {
    ok = true;
    for (int i = 0; i < kThreads * kSlotsPerThread; ++i) {
      if (cudaHostAlloc(&pinned[i], kChunk, cudaHostAllocDefault) != cudaSuccess ||
          cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming) != cudaSuccess) {
        cudaGetLastError();
        ok = false;
        break;
      }
    }
  }
  ~Stager() {
    for (int i = 0; i < kThreads * kSlotsPerThread; ++i) {
      if (ev[i]) cudaEventDestroy(ev[i]);
      if (pinned[i]) cudaFreeHost(pinned[i]);
    }
  }
};

void host_to_device(ge_context* ctx, void* dst, const void* src, size_t bytes) {
  bool direct = bytes < 4 * Stager::kChunk || std::getenv("GE_NO_STAGING") != nullptr;
  if (!direct) {  // already page-locked (cudaHostAlloc / cudaHostRegister): the DMA engine reads it directly
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, src) == cudaSuccess && attr.type == cudaMemoryTypeHost) direct = true;
    cudaGetLastError();
  }
  if (direct) {
    GE_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return;
  }
  if (!ctx->stager) ctx->stager = new Stager();
  Stager& st = *ctx->stager;
  if (!st.ok) {
    GE_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return;
  }
  const size_t nchunks = (bytes + Stager::kChunk - 1) / Stager::kChunk;
  std::atomic<int> failed(0);
  auto worker = [&](int t) {
    if (cudaSetDevice(ctx->device) != cudaSuccess) {
      failed = 1;
      return;
    }
    int turn = 0;
    for (size_t c = t; c < nchunks; c += Stager::kThreads, ++turn) {
      const int slot = t * Stager::kSlotsPerThread + (turn % Stager::kSlotsPerThread);
      const size_t off = c * Stager::kChunk, sz = std::min(Stager::kChunk, bytes - off);
      // the previous DMA out of this pinned buffer must have drained before it is refilled
      if (cudaEventSynchronize(st.ev[slot]) != cudaSuccess) failed = 1;
      std::memcpy(st.pinned[slot], (const char*)src + off, sz);
      if (cudaMemcpyAsync((char*)dst + off, st.pinned[slot], sz, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess ||
          cudaEventRecord(st.ev[slot], ctx->stream) != cudaSuccess)
        failed = 1;
    }
  };
  std::vector<std::thread> pool;
  for (int t = 1; t < Stager::kThreads; ++t) pool.emplace_back(worker, t);
  worker(0);
  for (auto& th : pool) th.join();
  if (failed) {
    cudaGetLastError();
    set_error("staged host->device copy failed");
    throw Fail{GE_ERR_CUDA};
  }
}

uint32_t resolve_seed(uint32_t seed) {
  if (seed != 0) return seed;
  std::random_device rd;  // what the reference does for every generator
  return rd();
}

// uniform_real_distribution<double>(-1,1) over std::mt19937 as libstdc++ evaluates it
// (generate_canonical<double,53>: two 32-bit draws, low word first, divided by 2^64; then
// a + (b-a)*u), written out so that it runs at the speed of the raw engine (~3x faster than going
// through the distribution object); bit-identical to it (tests/test_capi_host.py).
void reference_uniform(uint32_t seed, int64_t count, double* out) {
  std::mt19937 gen(seed);
  for (int64_t c = 0; c < count; ++c) {
    const double lo = (double)gen();
    const double hi = (double)gen();
    double u = (lo + hi * 4294967296.0) / 18446744073709551616.0;
    if (u >= 1.0) u = std::nextafter(1.0, 0.0);
    out[c] = u * (1.0 - (-1.0)) + (-1.0);
  }
}

// The reference's draw order for the local initial coordinates of one level
// (include/forceatlas.hpp:341, 356-358): aggregate-major, member-major, k-minor.
void level_init_stream(uint32_t seed, const ge_csr& P_T, int dim, double* init_by_vertex) {
  const int64_t n = P_T.indptr[P_T.rows];
  std::vector<double> stream((size_t)n * dim);
  reference_uniform(seed, n * dim, stream.data());
  for (int64_t c = 0; c < n; ++c)
    for (int k = 0; k < dim; ++k) init_by_vertex[(size_t)P_T.indices[c] * dim + k] = stream[c * dim + k];
}

// ---------------------------------------------------------------------------------------------
// Ball radii (src/embed.cpp:615-778).  Every pair (base case) or intra-super-aggregate coarse
// edge (general case) is an event "the two growing balls touch" at time -t; events are served
// latest-key-first in the lexicographic (t, i, j) order the reference obtains by sorting a
// vector of tuples and popping its back.  A max-heap gives the same service order without the
// reference's full re-sort after every freeze.
// ---------------------------------------------------------------------------------------------
namespace {
struct Event {
  double t;
  int i, j;
  bool operator<(const Event& o) const { return std::tie(t, i, j) < std::tie(o.t, o.i, o.j); }
};

inline double dist(const double* a, const double* b, int dim) {
  double sum = 0.0;
  for (int k = 0; k < dim; ++k) {
    const double d = b[k] - a[k];
    sum += d * d;
  }
  return std::sqrt(sum);
}

// ev: the events of one family; every vertex id in them has local[id] in [0, nloc).
// Service order = repeatedly the largest (t, i, j) among the current keys, exactly the reference's
// sort + pop_back; but only events incident to a vertex that just froze change key, and an event
// whose two endpoints are frozen can never act again, so a lazy-deletion heap over per-vertex
// incidence lists does it in O(E log E) instead of the reference's O(V E log E).
struct HeapItem {
  Event e;
  int idx, ver;
  bool operator<(const HeapItem& o) const { return e < o.e; }
};

void grow_balls(std::vector<Event>& ev, double* r_A, int m, const int* local, int nloc,
                std::vector<int>& inc_ptr, std::vector<int>& inc, std::vector<int>& ver,
                std::vector<HeapItem>& heap) {
  static thread_local std::vector<int> fill;  // scratch: families are many and small
  const int E = (int)ev.size();
  inc_ptr.assign(nloc + 1, 0);
  for (const Event& e : ev) {
    inc_ptr[local[e.i] + 1]++;
    inc_ptr[local[e.j] + 1]++;
  }
  for (int v = 0; v < nloc; ++v) inc_ptr[v + 1] += inc_ptr[v];
  inc.resize(2 * (size_t)E);
  {
    fill.assign(inc_ptr.begin(), inc_ptr.end() - 1);
    for (int x = 0; x < E; ++x) {
      inc[fill[local[ev[x].i]]++] = x;
      inc[fill[local[ev[x].j]]++] = x;
    }
  }
  ver.assign(E, 0);
  heap.clear();
  heap.reserve(2 * (size_t)E);
  for (int x = 0; x < E; ++x) heap.push_back(HeapItem{ev[x], x, 0});
  std::make_heap(heap.begin(), heap.end());
  int count = 0;
  while (count < m && !heap.empty()) {
    std::pop_heap(heap.begin(), heap.end());
    const HeapItem top = heap.back();
    heap.pop_back();
    if (top.ver != ver[top.idx]) continue;  // superseded key
    ver[top.idx] = -1;                       // served
    const int i = top.e.i, j = top.e.j;
    const bool live_i = r_A[i] <= 0.0, live_j = r_A[j] <= 0.0;
    if (!live_i && !live_j) continue;
    const double reach = -top.e.t;
    if (live_i) r_A[i] = reach;
    if (live_j) r_A[j] = reach;
    // a frozen ball stops growing: the partner must cover the remaining gap alone
    for (int side = 0; side < 2; ++side) {
      if (!(side == 0 ? live_i : live_j)) continue;
      const int v = local[side == 0 ? i : j];
      for (int q = inc_ptr[v]; q < inc_ptr[v + 1]; ++q) {
        const int x = inc[q];
        if (ver[x] < 0) continue;
        Event& e = ev[x];
        if (side == 1 && live_i && (e.i == i || e.j == i)) continue;  // already re-keyed once
        e.t = -(2 * (-e.t) - (-top.e.t));
        const int other = (e.i == (side == 0 ? i : j)) ? e.j : e.i;
        if (r_A[other] > 0.0) {  // both ends frozen now: can never act again
          ver[x] = -1;
          continue;
        }
        heap.push_back(HeapItem{e, x, ++ver[x]});
        std::push_heap(heap.begin(), heap.end());
      }
    }
    count += (live_i ? 1 : 0) + (live_j ? 1 : 0);
  }
}
}  // namespace

void level_radii(int m, int dim, double* coords_A, double* r_A, const ge_csr* A_c,
                 const ge_csr* P_T_c, const double* coords_Ac, const double* r_Ac) {
  std::fill(r_A, r_A + m, 0.0);
  std::vector<int> inc_ptr, inc, ver, local(std::max(m, 1));
  std::vector<HeapItem> heap;
  if (P_T_c == nullptr) {  // :616-679
    std::vector<Event> ev;
    ev.reserve((size_t)m * (m > 0 ? m - 1 : 0) / 2);
    for (int i = 0; i < m; ++i) {
      local[i] = i;
      for (int j = i + 1; j < m; ++j)
        ev.push_back(Event{-dist(coords_A + (size_t)i * dim, coords_A + (size_t)j * dim, dim) / 2, i, j});
    }
    grow_balls(ev, r_A, m, local.data(), m, inc_ptr, inc, ver, heap);
    return;
  }
  const int mc = P_T_c->rows;
  const int32_t* PI = P_T_c->indptr;
  const int32_t* PJ = P_T_c->indices;
  // a few host threads pull blocks of families off a counter (every loop below touches only the
  // members of its own families, so the results do not depend on the schedule)
  const int kBlock = 512;
  const int nthreads = (int)std::max(1u, std::min({std::thread::hardware_concurrency(), 16u,
                                                   (unsigned)((mc + kBlock - 1) / kBlock)}));
  auto for_family_blocks = [&](const std::function<void(int, int)>& body) {
    if (nthreads <= 1) {
      body(0, mc);
      return;
    }
    std::atomic<int> next(0);
    std::vector<std::thread> pool;
    for (int t = 0; t < nthreads; ++t)
      pool.emplace_back([&] {
        for (;;) {
          const int b0 = next.fetch_add(kBlock);
          if (b0 >= mc) break;
          body(b0, std::min(mc, b0 + kBlock));
        }
      });
    for (auto& th : pool) th.join();
  };
  std::vector<int> parent(m, -1);  // :684
  for_family_blocks([&](int b0, int b1) {
    for (int b = b0; b < b1; ++b)
      for (int c = PI[b]; c < PI[b + 1]; ++c) parent[PJ[c]] = b;
  });
  // :686-756: the families are independent (the reference runs this loop under `omp parallel
  // for`, src/embed.cpp:685).
  auto families = [&](int b0, int b1) {
    static thread_local std::vector<Event> ev;
    static thread_local std::vector<int> ip, in, vr, loc;
    static thread_local std::vector<HeapItem> hp;
    if ((int)loc.size() < m) loc.resize(m);
    for (int b = b0; b < b1; ++b) {
      const int s = PI[b + 1] - PI[b];
      if (s == 1) {
        r_A[PJ[PI[b]]] = r_Ac[b];
        continue;
      }
      ev.clear();
      for (int c = PI[b]; c < PI[b + 1]; ++c) loc[PJ[c]] = c - PI[b];
      for (int c = PI[b]; c < PI[b + 1]; ++c) {
        const int a = PJ[c];
        for (int kk = A_c->indptr[a]; kk < A_c->indptr[a + 1]; ++kk) {
          const int j = A_c->indices[kk];
          if (a < j && parent[j] == parent[a])
            ev.push_back(Event{-dist(coords_A + (size_t)a * dim, coords_A + (size_t)j * dim, dim) / 2, a, j});
        }
      }
      grow_balls(ev, r_A, m, loc.data(), s, ip, in, vr, hp);
    }
  };
  for_family_blocks(families);
  for_family_blocks([&](int b0, int b1) {  // :757-777 shrink each family into its parent ball
    for (int b = b0; b < b1; ++b) {
      const double* cb = coords_Ac + (size_t)b * dim;
      double alpha = 0.0;
      for (int c = PI[b]; c < PI[b + 1]; ++c) {
        const int a = PJ[c];
        alpha = std::max(alpha, dist(cb, coords_A + (size_t)a * dim, dim) + r_A[a]);
      }
      if (alpha < 0.000001) alpha = 0.000001;
      const double scale = r_Ac[b] / alpha;
      for (int c = PI[b]; c < PI[b + 1]; ++c) {
        const int a = PJ[c];
        for (int k = 0; k < dim; ++k)
          coords_A[(size_t)a * dim + k] = cb[k] + scale * (coords_A[(size_t)a * dim + k] - cb[k]);
        r_A[a] = scale * r_A[a];
      }
    }
  });
}

namespace {

// Independent register-resident FMA chains: the FP-pipe roofline the repulsion kernels are
// measured against (SURVEY.md section 8d asks for a measured, not derived, denominator).
template <typename T>
__global__ void __launch_bounds__(512) k_fma_peak(T* out, int iters, T b, T c) {
  T a[8];
#pragma unroll
  for (int u = 0; u < 8; ++u) a[u] = (T)(threadIdx.x + u) * (T)1e-3;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int u = 0; u < 8; ++u) a[u] = fma(a[u], b, c);
  }
  T s = (T)0;
#pragma unroll
  for (int u = 0; u < 8; ++u) s += a[u];
  out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

template <typename T>
double fma_peak(ge_context* ctx) {
  const int threads = 512, ctas = ctx->sm_count * 4, iters = 1 << 15;
  DevBuf<T> out(ctx, (size_t)threads * ctas);
  cudaEvent_t e0, e1;
  GE_CUDA(cudaEventCreate(&e0));
  GE_CUDA(cudaEventCreate(&e1));
  double best = 0.0;
  for (int rep = 0; rep < 4; ++rep) {
    GE_CUDA(cudaEventRecord(e0, ctx->stream));
    k_fma_peak<T><<<ctas, threads, 0, ctx->stream>>>(out.get(), iters, (T)0.999999, (T)1e-6);
    GE_CUDA(cudaEventRecord(e1, ctx->stream));
    GE_CUDA(cudaEventSynchronize(e1));
    ctx->launches++;
    float ms = 0;
    GE_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    const double flops = 2.0 * 8.0 * iters * double(threads) * ctas;
    if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  return best;
}

int onchip_threshold() {
  const char* v = std::getenv("GE_ONCHIP_MAX");
  // measured crossover between the cluster on-chip solve and the per-iteration launches of the
  // tiled kernels: n = 600 -> 10.7 vs ~17 us, n = 1000 -> 23.6 vs 20 us per iteration
  return v ? std::min(std::atoi(v), kOnchipMaxVertices) : 800;
}

void check_csr(const ge_csr* A, const char* what) {
  GE_REQUIRE(A != nullptr, std::string(what) + " is null");
  GE_REQUIRE(A->rows >= 0 && A->cols >= 0, std::string(what) + " has negative shape");
  GE_REQUIRE(A->indptr != nullptr, std::string(what) + ".indptr is null");
  GE_REQUIRE(A->indptr[A->rows] == 0 || A->indices != nullptr, std::string(what) + ".indices is null");
  GE_REQUIRE((int64_t)A->indptr[A->rows] == A->nnz, std::string(what) + ".nnz != indptr[rows]");
}

void flat_solve(ge_context* ctx, const ge_csr& A, int dim, double* coords, const ge_params& p,
                int path) {
  const bool onchip = path == 2 || (path == 0 && A.rows <= onchip_threshold());
  if (A.rows == 0) return;
  if (onchip) {
    onchip_flat_solve(ctx, A, dim, p, coords, nullptr, false);
    return;
  }
  // a multi-device context shards the iteration (graphs too small for the symmetric sweep stay on
  // the context's first device: nothing to share out)
  if (path == 0 && multi_size(ctx) > 1 && A.rows >= 32768 && std::getenv("GE_REP_SYM") == nullptr) {
    multi_flat_solve(ctx, A, dim, coords, p);
    return;
  }
  std::unique_ptr<FlatSolver> s(make_flat_solver(ctx, A, dim, p, 0, A.rows));
  s->upload_coords(coords);
  int it = 0;
  // Long runs on mid-size graphs are launch-bound (3 small kernels per iteration): after two
  // eager iterations (which also settle the one-time buffer refreshes) the steady-state pair of
  // iterations -- the coordinate buffers ping-pong, so the pattern has period 2 -- is captured
  // into a CUDA graph and replayed.
  const bool use_graph = p.iterations >= 64 && A.rows < 100000 && std::getenv("GE_NO_GRAPH") == nullptr;
  if (use_graph) {
    for (; it < 2; ++it) {
      s->launch_iteration(true);
      s->swap();
    }
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    GE_CUDA(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
    const int64_t launches_before = ctx->launches;
    for (int k = 0; k < 2; ++k) {
      s->launch_iteration(true);
      s->swap();
    }
    const int64_t per_replay = ctx->launches - launches_before;
    GE_CUDA(cudaStreamEndCapture(ctx->stream, &graph));
    GE_CUDA(cudaGraphInstantiate(&exec, graph, 0));
    ctx->launches = launches_before;  // capture launched nothing; replays are counted below
    for (; it + 2 <= p.iterations; it += 2) {
      GE_CUDA(cudaGraphLaunch(exec, ctx->stream));
      ctx->launches += per_replay;
    }
    GE_CUDA(cudaStreamSynchronize(ctx->stream));
    cudaGraphExecDestroy(exec);
    cudaGraphDestroy(graph);
  }
  for (; it < p.iterations; ++it) {
    s->launch_iteration(true);
    s->swap();
  }
  if (p.normalize) s->normalize();
  s->download_coords(coords);
}

// Cost-balanced contiguous aggregate ranges, one per device: cost(a) = s_a^2 ordered pairs + the CSR
// entries of its members' rows (SURVEY.md section 8e).  cuts: N + 1 boundaries, cuts[0] = 0,
// cuts[N] = m.  Returns the ordered intra-aggregate pairs per iteration of the level.
double aggregate_ranges(const ge_csr& A, const ge_csr& P, int N, std::vector<int>& cuts) {
  const int m = P.rows;
  std::vector<double> cost((size_t)m + 1, 0.0);
  double pairs = 0.0;
  for (int a = 0; a < m; ++a) {
    const double s = P.indptr[a + 1] - P.indptr[a];
    double nnz = 0.0;
    for (int c = P.indptr[a]; c < P.indptr[a + 1]; ++c)
      nnz += A.indptr[P.indices[c] + 1] - A.indptr[P.indices[c]];
    pairs += s * (s - 1);
    cost[a + 1] = cost[a] + s * s + nnz;
  }
  cuts.assign(N + 1, 0);
  int prev = 0;
  for (int d = 0; d < N; ++d) {
    const double target = cost[m] * (d + 1) / N;
    int cut = d == N - 1 ? m : (int)(std::lower_bound(cost.begin(), cost.end(), target) - cost.begin());
    cut = std::max(prev, std::min(cut, m));
    cuts[d + 1] = cut;
    prev = cut;
  }
  return pairs;
}

// The same as a set per device instead of a contiguous range: hierarchies of the reference
// partitioner carry a few hundred giant aggregates (one of them can be a fifth of a device's share),
// around which contiguous cuts are off by ~13 % (Delaunay 4M on 8 devices).  Heavy aggregates (cost
// above 1/64 of a device's share) are placed largest-first on the least loaded device; the light
// ones then fill the devices up in index order.  owned[d] is ascending.  Returns the ordered pairs.
double aggregate_assignment(const ge_csr& A, const ge_csr& P, int N, std::vector<std::vector<int>>& owned) {
  const int m = P.rows;
  std::vector<double> cost((size_t)std::max(m, 1), 0.0);
  double pairs = 0.0, total = 0.0;
  for (int a = 0; a < m; ++a) {
    const double s = P.indptr[a + 1] - P.indptr[a];
    double nnz = 0.0;
    for (int c = P.indptr[a]; c < P.indptr[a + 1]; ++c)
      nnz += A.indptr[P.indices[c] + 1] - A.indptr[P.indices[c]];
    pairs += s * (s - 1);
    cost[a] = s * s + nnz;
    total += cost[a];
  }
  owned.assign(N, std::vector<int>());
  std::vector<double> load(N, 0.0);
  const double heavy_min = total / N / 64.0;
  std::vector<int> heavy;
  for (int a = 0; a < m; ++a)
    if (cost[a] >= heavy_min && cost[a] > 0.0) heavy.push_back(a);
  std::stable_sort(heavy.begin(), heavy.end(), [&](int x, int y) { return cost[x] > cost[y]; });
  for (int a : heavy) {
    int best = 0;
    for (int d = 1; d < N; ++d)
      if (load[d] < load[best]) best = d;
    owned[best].push_back(a);
    load[best] += cost[a];
  }
  const double target = total / N;
  int d = 0;
  for (int a = 0; a < m; ++a) {
    if (cost[a] >= heavy_min && cost[a] > 0.0) continue;
    while (d < N - 1 && load[d] >= target) ++d;
    owned[d].push_back(a);
    load[d] += cost[a];
  }
  for (auto& o : owned) std::sort(o.begin(), o.end());
  return pairs;
}

// partition::embed on one device or, with a multi-device context, with the large levels sharded by
// aggregates (SURVEY.md section 8e: aggregates are independent, include/forceatlas.hpp:340-341).
struct EmbedRun {
  ge_context* ctx;
  int L, dim;
  const ge_csr* As;
  const ge_csr* Ps;
  ge_embed_options opt;
  ge_embed_stats st{};
  // ge_layout_graph: the graphs of levels 0..L-1 are already on device 0 and As[l] carries their row
  // pointers only.  Device 0 takes their buffers over; another device copies them from device 0
  // (dev_src: their addresses, which stay valid while device 0 owns them).
  DeviceHierarchy* on_device = nullptr;
  struct DevSrc {
    const int* I;
    const int* J;
    const double* W;
  };
  std::vector<DevSrc> dev_src;

  // Per device: the level graphs + slot layouts (inputs that do not depend on any result: a helper
  // thread uploads the large ones on the device's copy stream while the coarsest-level solve, one
  // long kernel that needs no host attention, occupies device 0), the coordinates dx[k] (n_k x dim)
  // and ball radii dr[k] (n_k) of the levels, which never leave the device, and the range of
  // aggregates [a0[l], a1[l]) the device solves at level l.
  struct Dev {
    ge_context* ctx = nullptr;
    std::vector<std::unique_ptr<PrefetchedGraph>> pre;
    std::vector<DevBuf<double>> dx, dr;
    std::vector<int> a0, a1;
    std::vector<std::vector<int>> owned;  // per sharded level: the aggregates this device solves
    std::thread prefetcher;
    std::string error;
    ge_status status = GE_OK;
    double prefetch_h2d = 0.0;
  };
  std::vector<Dev> devs;
  std::vector<char> sharded;  // per level
  static constexpr int64_t kPrefetchMinNnz = 1 << 22;  // ~50 MB of CSR: below, the upload is < 2 ms

  // Levels with at least this many ordered pairs per iteration are shared out over the devices
  // (cost-balanced contiguous aggregate ranges); smaller ones cost less than the exchange.
  void plan_ranges() {
    const int N = multi_size(ctx);
    devs.resize(N);
    sharded.assign(std::max(L, 1), 0);
    for (int d = 0; d < N; ++d) {
      devs[d].ctx = multi_device(ctx, d);
      devs[d].pre.resize(L);
      devs[d].dx.resize(L + 1);
      devs[d].dr.resize(L + 1);
      devs[d].a0.assign(L, 0);
      devs[d].a1.assign(L, 0);
      devs[d].owned.assign(L, std::vector<int>());
    }
    const char* e = std::getenv("GE_SHARD_MIN_MPAIRS");
    const double min_pairs = 1e6 * (e ? std::atof(e) : 200.0);
    for (int l = 0; l < L; ++l) {
      devs[0].a1[l] = Ps[l].rows;
      if (N == 1) continue;
      std::vector<std::vector<int>> sets;
      const double pairs = aggregate_assignment(As[l], Ps[l], N, sets);
      if (pairs < min_pairs) continue;
      sharded[l] = 1;
      for (int d = 0; d < N; ++d) {
        devs[d].owned[l] = std::move(sets[d]);
        devs[d].a0[l] = 0;
        devs[d].a1[l] = (int)devs[d].owned[l].size();  // (only "has work" below; the set decides)
      }
    }
  }

  void adopt_device_levels() {
    if (on_device == nullptr) return;
    for (int l = 0; l < L; ++l) {
      const DevGraph& G = *on_device->graphs[l];
      dev_src.push_back(DevSrc{G.I.get(), G.J.get(), G.w()});
    }
  }

  // Level l's graph on device d (context c): from the host arrays, or from the device hierarchy.
  void fetch_graph(ge_context* c, int d, int l, PrefetchedGraph& g) {
    const ge_csr& A = As[l];
    if (on_device == nullptr) {
      g.I.alloc(c, A.rows + 1);
      g.J.alloc(c, (size_t)std::max<int64_t>(A.nnz, 1));
      g.I.upload(c, A.indptr, A.rows + 1);
      g.J.upload(c, A.indices, (size_t)A.nnz);
      if (A.data != nullptr) {
        g.Dw.alloc(c, (size_t)std::max<int64_t>(A.nnz, 1));
        g.Dw.upload(c, A.data, (size_t)A.nnz);
      }
      return;
    }
    if (d == 0) {
      DevGraph& G = *on_device->graphs[l];
      g.I = std::move(G.I);
      g.J = std::move(G.J);
      g.Dw = std::move(G.W);
      return;
    }
    const DevSrc& src = dev_src[l];
    g.I.alloc(c, A.rows + 1);
    g.J.alloc(c, (size_t)std::max<int64_t>(A.nnz, 1));
    GE_CUDA(cudaMemcpyPeerAsync(g.I.get(), c->device, src.I, ctx->device, sizeof(int) * ((size_t)A.rows + 1),
                                c->stream));
    if (A.nnz)
      GE_CUDA(cudaMemcpyPeerAsync(g.J.get(), c->device, src.J, ctx->device, sizeof(int) * (size_t)A.nnz,
                                  c->stream));
    if (src.W != nullptr) {
      g.Dw.alloc(c, (size_t)std::max<int64_t>(A.nnz, 1));
      if (A.nnz)
        GE_CUDA(cudaMemcpyPeerAsync(g.Dw.get(), c->device, src.W, ctx->device, sizeof(double) * (size_t)A.nnz,
                                    c->stream));
    }
  }

  void start_prefetch() {
    if (std::getenv("GE_NO_PREFETCH")) return;
    for (size_t d = 0; d < devs.size(); ++d) {
      bool any = false;
      for (int l = 0; l < L; ++l)
        any = any || (As[l].nnz >= kPrefetchMinNnz && (d == 0 || devs[d].a1[l] > devs[d].a0[l]));
      if (!any) continue;
      Dev* dev = &devs[d];
      ge_context* c = dev->ctx;
      GE_CUDA(cudaSetDevice(c->device));
      if (!c->copy_stream) GE_CUDA(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
      dev->prefetcher = std::thread([this, dev, c, d] {
        try {
          GE_CUDA(cudaSetDevice(c->device));
          ge_context side = *c;  // same device and pool, its own stream / staging ring / counters
          side.stream = c->copy_stream;
          side.stager = c->stager2;
          side.h2d_bytes = 0;
          for (int l = 0; l < L; ++l) {  // finest first: it is the largest and the last one needed
            const ge_csr& A = As[l];
            if (A.nnz < kPrefetchMinNnz) continue;
            if (d != 0 && dev->a1[l] <= dev->a0[l]) continue;
            std::unique_ptr<PrefetchedGraph> g(new PrefetchedGraph);
            fetch_graph(&side, (int)d, l, *g);
            g->layout = sharded[l] ? make_level_layout(&side, Ps[l], A.rows, 0, -1, d == 0, &dev->owned[l])
                                   : make_level_layout(&side, Ps[l], A.rows, dev->a0[l], dev->a1[l], d == 0);
            GE_CUDA(cudaEventCreateWithFlags(&g->ready, cudaEventDisableTiming));
            GE_CUDA(cudaEventRecord(g->ready, side.stream));
            dev->pre[l] = std::move(g);
          }
          c->stager2 = side.stager;  // keep the ring for the next call
          dev->prefetch_h2d = side.h2d_bytes;
        } catch (const Fail& f) {
          dev->status = f.st;
          dev->error = ge_last_error();
        } catch (const std::exception& e) {
          dev->status = GE_ERR_INVALID;
          dev->error = e.what();
        }
      });
    }
    GE_CUDA(cudaSetDevice(ctx->device));
  }
  void join_prefetch() {
    for (auto& dev : devs) {
      if (!dev.prefetcher.joinable()) continue;
      dev.prefetcher.join();
      ctx->h2d_bytes += dev.prefetch_h2d;
      dev.prefetch_h2d = 0.0;
    }
    for (auto& dev : devs)
      if (dev.status != GE_OK) {
        set_error("level-graph prefetch: " + dev.error);
        throw Fail{dev.status};
      }
  }
  ~EmbedRun() {
    for (auto& dev : devs)
      if (dev.prefetcher.joinable()) dev.prefetcher.join();
    for (auto& dev : devs) {
      cudaSetDevice(dev.ctx->device);
      dev.dx.clear();
      dev.dr.clear();
      // the prefetched buffers were allocated on the copy stream: nothing on the main stream may
      // still read them when they are returned to the pool
      cudaStreamSynchronize(dev.ctx->stream);
      if (dev.ctx->copy_stream) cudaStreamSynchronize(dev.ctx->copy_stream);
    }
    // (device 0's level graphs are the source of the other devices' copies: freed after every sync)
    for (auto& dev : devs) {
      cudaSetDevice(dev.ctx->device);
      dev.pre.clear();
    }
    cudaSetDevice(ctx->device);
  }

  // The level graph + slot layout on device d: uploaded ahead of time by the prefetcher (large
  // levels) or here, on the device's main stream, when the level is first needed.
  const PrefetchedGraph* graph(int d, int l) {
    Dev& dev = devs[d];
    if (dev.pre[l]) return dev.pre[l].get();
    const ge_csr& A = As[l];
    std::unique_ptr<PrefetchedGraph> g(new PrefetchedGraph);
    fetch_graph(dev.ctx, d, l, *g);
    g->layout = sharded[l] ? make_level_layout(dev.ctx, Ps[l], A.rows, 0, -1, d == 0, &dev.owned[l])
                           : make_level_layout(dev.ctx, Ps[l], A.rows, dev.a0[l], dev.a1[l], d == 0);
    GE_CUDA(cudaEventCreateWithFlags(&g->ready, cudaEventDisableTiming));
    GE_CUDA(cudaEventRecord(g->ready, dev.ctx->stream));
    dev.pre[l] = std::move(g);
    return dev.pre[l].get();
  }

  // src/embed.cpp:615-778 for the vertices of level k = l + 1, on device 0.
  void radii(int k) {
    Dev& d0 = devs[0];
    const int m = As[k].rows;
    d0.dr[k].alloc(ctx, (size_t)std::max(m, 1));
    const bool base = k == L;
    const bool on_host = std::getenv("GE_HOST_RADII") != nullptr || (base && m > kRadiiBaseMax);
    if (!on_host) {
      if (base) {
        level_radii_device(ctx, m, dim, d0.dx[k].get(), d0.dr[k].get(), nullptr, nullptr, nullptr);
      } else {
        GE_CUDA(cudaStreamWaitEvent(ctx->stream, graph(0, k)->ready, 0));
        const RadiiLevel lv = radii_level_of(*graph(0, k), As[k + 1].rows);
        level_radii_device(ctx, m, dim, d0.dx[k].get(), d0.dr[k].get(), &lv, d0.dx[k + 1].get(),
                           d0.dr[k + 1].get());
      }
      return;
    }
    // host restatement (the checker of the device kernels; also the all-pairs base case of a
    // coarsest level too large for the device's event arrays)
    const double t0 = now_ms();
    std::vector<double> x((size_t)m * dim), r(m, 0.0), xc, rc;
    std::vector<int> cols;
    ge_csr Ak = As[k];
    if (!base && Ak.indices == nullptr) {  // a level on the device only: its columns come down
      const PrefetchedGraph* g = graph(0, k);
      GE_CUDA(cudaStreamWaitEvent(ctx->stream, g->ready, 0));
      cols.resize((size_t)Ak.nnz);
      g->J.download(ctx, cols.data(), cols.size());
      Ak.indices = cols.data();
    }
    d0.dx[k].download(ctx, x.data(), x.size());
    if (!base) {
      const int mc = As[k + 1].rows;
      xc.resize((size_t)mc * dim);
      rc.resize(mc);
      d0.dx[k + 1].download(ctx, xc.data(), xc.size());
      d0.dr[k + 1].download(ctx, rc.data(), rc.size());
    }
    GE_CUDA(cudaStreamSynchronize(ctx->stream));
    if (base) level_radii(m, dim, x.data(), r.data(), nullptr, nullptr, nullptr, nullptr);
    else level_radii(m, dim, x.data(), r.data(), &Ak, &Ps[k], xc.data(), rc.data());
    d0.dx[k].upload(ctx, x.data(), x.size());
    d0.dr[k].upload(ctx, r.data(), r.size());
    GE_CUDA(cudaStreamSynchronize(ctx->stream));
    st.host_radii_ms += now_ms() - t0;
  }

  // One level on one device (its range of aggregates).  Runs on the calling thread.
  void solve_level(int d, int l, const double* init, double* host_out, double* pairs) {
    Dev& dev = devs[d];
    ge_params p;
    ge_params_default_multilevel(&p);
    p.iterations = opt.level_iterations;  // :793
    p.precision = opt.precision;
    p.seed = opt.seed;
    LevelIO io;
    io.d_coords_A = dev.dx[l + 1].get();
    io.d_r_A = dev.dr[l + 1].get();
    io.keep_out = (l > 0 || sharded[l]) ? &dev.dx[l] : nullptr;
    io.download = host_out != nullptr;
    io.owned = sharded[l] ? &dev.owned[l] : nullptr;
    multilevel_solve(dev.ctx, As[l], Ps[l], nullptr, nullptr, nullptr, init, host_out, dim, p, false,
                     pairs, sharded[l] ? 0 : dev.a0[l], sharded[l] ? -1 : dev.a1[l], graph(d, l), &io);
  }

  // embedMultilevel, src/embed.cpp:576-796, unrolled from the coarsest level up.
  void run(double* coords_out, double* r_A_out, double* coords_A_out) {
    Dev& d0 = devs[0];
    const int N = (int)devs.size();
    {  // :582-587 base: forceAtlas with its defaults on the coarsest graph
      const ge_csr& A = As[L];
      const int n = A.rows;
      if (opt.verbose) std::printf("embedding layer %d: getting base coords\n", L + opt.first_layer);
      std::vector<double> coords((size_t)n * dim);
      reference_uniform(resolve_seed(opt.seed), (int64_t)n * dim, coords.data());  // forceatlas.hpp:118-125
      ge_params p;
      ge_params_default_flat(&p);
      p.iterations = opt.coarse_iterations;
      p.precision = opt.precision;
      const double t0 = now_ms();
      if (L == 0) {
        flat_solve(ctx, A, dim, coords.data(), p, 0);
        std::memcpy(coords_out, coords.data(), coords.size() * sizeof(double));
      } else if (n >= 1 && n <= onchip_threshold()) {
        onchip_flat_solve(ctx, A, dim, p, coords.data(), nullptr, false, &d0.dx[L]);
      } else {
        flat_solve(ctx, A, dim, coords.data(), p, 0);
        d0.dx[L].alloc(ctx, (size_t)std::max(n, 1) * dim);
        d0.dx[L].upload(ctx, coords.data(), coords.size());
      }
      st.coarse_ms += now_ms() - t0;
      join_prefetch();  // normally long finished: the solve above takes 0.1-0.2 s
      st.pair_interactions += double(n) * double(n - 1) * p.iterations;
      st.edge_visits += double(A.nnz) * p.iterations;
    }
    for (int l = L - 1; l >= 0; --l) {
      const ge_csr& A = As[l];
      const ge_csr& P = Ps[l];
      const int n = A.rows, m = P.rows;
      if (opt.verbose) std::printf("embeding layer %d\n", l + opt.first_layer);
      radii(l + 1);
      for (auto& dev : devs) {  // the grand-parent level is not needed any more
        if (l + 2 > L) break;
        GE_CUDA(cudaSetDevice(dev.ctx->device));
        dev.dx[l + 2].release();
        dev.dr[l + 2].release();
      }
      GE_CUDA(cudaSetDevice(ctx->device));
      // Initial local coordinates: with a fixed seed, the reference's own stream in its draw order
      // (forceatlas.hpp:341, 356-358); with seed 0 (the reference's std::random_device mode, where
      // any stream is as good as another) they are drawn on the device.
      std::vector<double> init;
      if (opt.seed != 0) {
        init.resize((size_t)n * dim);
        level_init_stream(opt.seed, P, dim, init.data());
      }
      const double* init_p = init.empty() ? nullptr : init.data();
      const double t1 = now_ms();
      double pairs = 0.0;
      if (!sharded[l]) {
        solve_level(0, l, init_p, l == 0 ? coords_out : nullptr, &pairs);
      } else {
        // parent centres and radii to every device, each device its aggregates, then one sum over
        // the devices (rows of foreign aggregates are exact zeros: x + 0 is exact)
        std::vector<double*> bx(N), br(N), bo(N);
        for (int d = 0; d < N; ++d) {
          Dev& dev = devs[d];
          GE_CUDA(cudaSetDevice(dev.ctx->device));
          if (d > 0) {
            dev.dx[l + 1].alloc(dev.ctx, (size_t)std::max(m, 1) * dim);
            dev.dr[l + 1].alloc(dev.ctx, (size_t)std::max(m, 1));
          }
          bx[d] = dev.dx[l + 1].get();
          br[d] = dev.dr[l + 1].get();
        }
        multi_broadcast_f64(ctx, bx, (size_t)m * dim, 0);
        multi_broadcast_f64(ctx, br, (size_t)m, 0);
        std::vector<std::thread> pool;
        std::vector<double> dpairs(N, 0.0);
        std::vector<ge_status> status(N, GE_OK);
        std::vector<std::string> errors(N);
        for (int d = 0; d < N; ++d)
          pool.emplace_back([&, d] {
            try {
              GE_CUDA(cudaSetDevice(devs[d].ctx->device));
              solve_level(d, l, init_p, nullptr, &dpairs[d]);
            } catch (const Fail& f) {
              status[d] = f.st;
              errors[d] = ge_last_error();
            } catch (const std::exception& e) {
              status[d] = GE_ERR_INVALID;
              errors[d] = e.what();
            }
          });
        for (auto& t : pool) t.join();
        for (int d = 0; d < N; ++d)
          if (status[d] != GE_OK) {
            set_error("device " + std::to_string(devs[d].ctx->device) + ": " + errors[d]);
            throw Fail{status[d]};
          }
        for (int d = 0; d < N; ++d) {
          pairs += dpairs[d];
          bo[d] = devs[d].dx[l].get();
        }
        multi_allreduce_sum_f64(ctx, bo, (size_t)n * dim);
        multi_sync(ctx);
        if (l == 0) {
          d0.dx[0].download(ctx, coords_out, (size_t)n * dim);
          GE_CUDA(cudaStreamSynchronize(ctx->stream));
        }
      }
      st.levels_ms += now_ms() - t1;
      st.pair_interactions += pairs * opt.level_iterations;
      st.edge_visits += double(A.nnz) * opt.level_iterations;
    }
    if (L > 0) {  // what embedMultilevel leaves in its r_A / coords_A out-parameters
      if (r_A_out) d0.dr[1].download(ctx, r_A_out, (size_t)As[1].rows);
      if (coords_A_out) d0.dx[1].download(ctx, coords_A_out, (size_t)As[1].rows * dim);
      if (r_A_out || coords_A_out) GE_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    multi_collect_counters(ctx);
  }
};

// ge_embed's driver; on_device: ge_layout_graph's hierarchy (see EmbedRun::on_device)
void embed_levels(ge_context* ctx, int L, const ge_csr* As, const ge_csr* P_Ts, int dim,
                  const ge_embed_options* opt, double* coords_out, double* r_A_out, double* coords_A_out,
                  ge_embed_stats* stats, DeviceHierarchy* on_device) {
  EmbedRun run;
  run.ctx = ctx;
  run.L = L;
  run.dim = dim;
  run.As = As;
  run.Ps = P_Ts;
  run.on_device = on_device;
  if (opt) run.opt = *opt;
  else ge_embed_options_default(&run.opt);
  const int64_t launches0 = ctx->launches;
  const double h0 = ctx->h2d_bytes, d0 = ctx->d2h_bytes;
  ctx->grid_tier_ms = 0;
  ctx->radii_ms = 0;
  const double t0 = now_ms();
  run.adopt_device_levels();
  run.plan_ranges();
  run.start_prefetch();
  run.run(coords_out, r_A_out, coords_A_out);
  run.st.total_ms = now_ms() - t0;
  run.st.kernel_launches = ctx->launches - launches0;
  run.st.h2d_bytes = ctx->h2d_bytes - h0;
  run.st.d2h_bytes = ctx->d2h_bytes - d0;
  run.st.grid_tier_ms = ctx->grid_tier_ms;
  run.st.device_radii_ms = ctx->radii_ms;
  if (stats) *stats = run.st;
}

template <typename F>
ge_status guarded(F&& body) {
  try {
    body();
    return GE_OK;
  } catch (const Fail& f) {
    return f.st;
  } catch (const std::bad_alloc&) {
    set_error("host allocation failed");
    return GE_ERR_OOM;
  } catch (const std::exception& e) {
    set_error(e.what());
    return GE_ERR_INVALID;
  }
}

// GE_ERR_NO_DEVICE without a usable device, before any argument is looked at
void require_device() {
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
    cudaGetLastError();
    set_error("no usable CUDA device (this library has no CPU fallback)");
    throw Fail{GE_ERR_NO_DEVICE};
  }
}

void require_ctx(ge_context* ctx) {
  GE_REQUIRE(ctx != nullptr, "context is null");
  GE_CUDA(cudaSetDevice(ctx->device));
}

// The body of ge_layout_graph and ge_layout_edges: a checked graph on the device -> [largest
// component] -> ge_coarsen's hierarchy -> ge_embed.  Fills st but for the whole-call counters.
void layout_device(ge_context* ctx, std::unique_ptr<DevGraph> G, int dim, int32_t largest_component,
                   const ge_coarsen_options& co, const ge_embed_options* eopt, double* coords_out,
                   int32_t* vertices_out, int32_t* n_out, ge_layout_stats& st) {
  cudaEvent_t ev[4];
  for (auto& e : ev) GE_CUDA(cudaEventCreate(&e));
  struct Events {
    cudaEvent_t* e;
    ~Events() {
      for (int i = 0; i < 4; ++i) cudaEventDestroy(e[i]);
    }
  } events{ev};
  auto elapsed = [&](int a, int b) {
    float ms = 0;
    GE_CUDA(cudaEventElapsedTime(&ms, ev[a], ev[b]));
    return (double)ms;
  };
  DeviceHierarchy h;
  DevBuf<int> kept;
  if (largest_component) {
    GE_CUDA(cudaEventRecord(ev[0], ctx->stream));
    auto C = std::make_unique<DevGraph>();
    st.components = largest_component_device(ctx, *G, *C, kept);
    if (st.components > 1) G = std::move(C);
    else unit_weights(ctx, *G);  // what ge_largest_component hands over: explicit weights
    GE_CUDA(cudaEventRecord(ev[1], ctx->stream));
  }
  h.graphs.push_back(std::move(G));
  GE_CUDA(cudaEventRecord(ev[2], ctx->stream));
  coarsen_device(ctx, h, co, false, nullptr);
  GE_CUDA(cudaEventRecord(ev[3], ctx->stream));
  // down: every P_T and every level's row pointers (O(n)), and the coarsest graph in full
  const int L = h.levels();
  std::vector<HostHierarchy::Csr> hg(L + 1), hp(L);
  for (int l = 0; l <= L; ++l) {
    const DevGraph& D = *h.graphs[l];
    HostHierarchy::Csr& g = hg[l];
    g.rows = g.cols = D.n;
    g.indptr.resize((size_t)D.n + 1);
    D.I.download(ctx, g.indptr.data(), (size_t)D.n + 1);
    if (l == L) {
      g.indices.resize(std::max(D.nnz, 1));
      D.J.download(ctx, g.indices.data(), D.nnz);
      if (D.W.size()) {
        g.data.resize(std::max(D.nnz, 1));
        D.W.download(ctx, g.data.data(), D.nnz);
      }
    }
    if (l < L) {
      const DevAgg& P = *h.aggs[l];
      HostHierarchy::Csr& p = hp[l];
      p.rows = P.m;
      p.cols = P.n;
      p.indptr.resize((size_t)P.m + 1);
      p.indices.resize(P.n);
      P.ptr.download(ctx, p.indptr.data(), (size_t)P.m + 1);
      P.idx.download(ctx, p.indices.data(), P.n);
    }
  }
  const int n = h.graphs[0]->n;
  if (vertices_out) {
    if (st.components > 1) kept.download(ctx, vertices_out, (size_t)n);
    else
      for (int v = 0; v < n; ++v) vertices_out[v] = v;
  }
  GE_CUDA(cudaStreamSynchronize(ctx->stream));
  if (largest_component) st.components_ms = elapsed(0, 1);
  st.coarsen_ms = elapsed(2, 3);
  std::vector<ge_csr> As(L + 1), Ps(std::max(L, 1));
  for (int l = 0; l <= L; ++l) {
    const HostHierarchy::Csr& g = hg[l];
    ge_csr& c = As[l];
    c.rows = c.cols = g.rows;
    c.nnz = g.indptr[g.rows];
    c.indptr = g.indptr.data();
    c.indices = l == L ? g.indices.data() : nullptr;
    c.data = l == L && !g.data.empty() ? g.data.data() : nullptr;
  }
  for (int l = 0; l < L; ++l) {
    ge_csr& c = Ps[l];
    c.rows = hp[l].rows;
    c.cols = hp[l].cols;
    c.nnz = hp[l].cols;
    c.indptr = hp[l].indptr.data();
    c.indices = hp[l].indices.data();
    c.data = nullptr;
  }
  ge_embed_options eo;
  if (eopt) eo = *eopt;
  else ge_embed_options_default(&eo);
  const double t_embed = now_ms();
  // the level graphs now move into the driver's prefetched graphs
  embed_levels(ctx, L, As.data(), Ps.data(), dim, &eo, coords_out, nullptr, nullptr, nullptr, &h);
  st.embed_ms = now_ms() - t_embed;
  *n_out = n;
  st.levels = L;
}

}  // namespace
}  // namespace ge

struct ge_flat_plan {
  std::unique_ptr<ge::FlatSolver> solver;
};

struct ge_hierarchy : ge::HostHierarchy {};

using namespace ge;

extern "C" {

const char* ge_version(void) { return "graph-embed_b200 0.1 (sm_100a)"; }
const char* ge_last_error(void) { return g_error.c_str(); }

void ge_params_default_flat(ge_params* p) {
  std::memset(p, 0, sizeof(*p));
  p->iterations = 100000;
  p->ks = 0.1;
  p->ksmax = 1.0;
  p->repel = 1.0;
  p->attract = 1.0;
  p->gravity = 1.0;
  p->delta = 1.0;
  p->tolerate = 1.0;
  p->use_weights = 1;
  p->precision = GE_F64;
}
void ge_params_default_multilevel(ge_params* p) {
  ge_params_default_flat(p);
  p->iterations = 100;
}
void ge_embed_options_default(ge_embed_options* o) {
  std::memset(o, 0, sizeof(*o));
  o->coarse_iterations = 100000;
  o->level_iterations = 100;
  o->precision = GE_F64;
  o->verbose = 1;
  o->first_layer = 1;
}

ge_status ge_context_create(int device, void* cuda_stream, ge_context** out) {
  return guarded([&] {
    GE_REQUIRE(out != nullptr, "out is null");
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
      cudaGetLastError();
      set_error("no usable CUDA device (this library has no CPU fallback)");
      throw Fail{GE_ERR_NO_DEVICE};
    }
    std::unique_ptr<ge_context> ctx(new ge_context);
    if (device < 0) GE_CUDA(cudaGetDevice(&device));
    GE_REQUIRE(device < count, "device ordinal out of range");
    ctx->device = device;
    GE_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    GE_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
      set_error("device is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) +
                "; this build contains sm_100a code only");
      throw Fail{GE_ERR_NO_DEVICE};
    }
    {  // keep freed blocks in the stream-ordered pool instead of returning them to the driver
      cudaMemPool_t pool;
      GE_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
      uint64_t keep = UINT64_MAX;
      GE_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    }
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    if (cuda_stream) {
      ctx->stream = (cudaStream_t)cuda_stream;
    } else {
      GE_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
      ctx->own_stream = true;
    }
    *out = ctx.release();
  });
}

ge_status ge_context_create_multi(int ndev, const int* devices, ge_context** out) {
  ge_context* ctx = nullptr;
  const ge_status st = guarded([&] {
    GE_REQUIRE(out != nullptr, "out is null");
    *out = nullptr;
    GE_REQUIRE(ndev >= 1 && ndev <= 64, "bad device count");
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
      cudaGetLastError();
      set_error("no usable CUDA device (this library has no CPU fallback)");
      throw Fail{GE_ERR_NO_DEVICE};
    }
    GE_REQUIRE(ndev <= count, "more devices requested than the box has");
    const ge_status s0 = ge_context_create(devices ? devices[0] : 0, nullptr, &ctx);
    if (s0 != GE_OK) throw Fail{s0};
    if (ndev > 1) multi_attach(ctx, ndev, devices);
    *out = ctx;
  });
  if (st != GE_OK && ctx != nullptr) {
    const std::string keep = g_error;
    ge_context_destroy(ctx);
    g_error = keep;
  }
  return st;
}
int32_t ge_context_device_count(const ge_context* ctx) { return ctx ? multi_size(ctx) : 0; }

void ge_context_destroy(ge_context* ctx) {
  if (!ctx) return;
  if (ctx->multi) {
    multi_destroy(ctx->multi);
    ctx->multi = nullptr;
    cudaSetDevice(ctx->device);
  }
  if (ctx->stager) {
    cudaStreamSynchronize(ctx->stream);
    delete ctx->stager;
  }
  if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
  delete ctx->stager2;
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

int64_t ge_context_launch_count(const ge_context* ctx) { return ctx ? ctx->launches : 0; }
void ge_context_bytes(const ge_context* ctx, double* h2d, double* d2h) {
  if (h2d) *h2d = ctx ? ctx->h2d_bytes : 0.0;
  if (d2h) *d2h = ctx ? ctx->d2h_bytes : 0.0;
}
ge_status ge_measure_fma_peak(ge_context* ctx, int precision, double* tflops) {
  return guarded([&] {
    require_ctx(ctx);
    GE_REQUIRE(tflops != nullptr, "tflops is null");
    *tflops = precision == GE_F32 ? fma_peak<float>(ctx) : fma_peak<double>(ctx);
  });
}

ge_status ge_flat_forceatlas(ge_context* ctx, const ge_csr* A, int dim, double* coords,
                             const ge_params* p) {
  return guarded([&] {
    require_ctx(ctx);
    check_csr(A, "A");
    GE_REQUIRE(coords != nullptr && p != nullptr, "coords / params are null");
    flat_solve(ctx, *A, dim, coords, *p, 0);
  });
}

ge_status ge_multilevel_forceatlas(ge_context* ctx, const ge_csr* A, const ge_csr* P_T,
                                   const int32_t* v_A, const double* coords_A, const double* r_A,
                                   const double* init, double* coords, int dim,
                                   const ge_params* p) {
  return guarded([&] {
    require_ctx(ctx);
    check_csr(A, "A");
    check_csr(P_T, "P_T");
    GE_REQUIRE(v_A && coords_A && r_A && coords && p, "null argument");
    std::vector<double> drawn;
    if (init == nullptr && p->seed != 0) {  // include/forceatlas.hpp:341, 356-358
      drawn.resize((size_t)A->rows * dim);
      level_init_stream(p->seed, *P_T, dim, drawn.data());
      init = drawn.data();
    }  // seed 0: drawn on the device (the reference's non-reproducible std::random_device mode)
    multilevel_solve(ctx, *A, *P_T, v_A, coords_A, r_A, init, coords, dim, *p, false, nullptr);
  });
}

ge_status ge_multilevel_forceatlas_shard(ge_context* ctx, const ge_csr* A, const ge_csr* P_T,
                                         const int32_t* v_A, const double* coords_A,
                                         const double* r_A, const double* init, double* coords,
                                         int dim, const ge_params* p, int32_t agg_begin,
                                         int32_t agg_end) {
  return guarded([&] {
    require_ctx(ctx);
    check_csr(A, "A");
    check_csr(P_T, "P_T");
    GE_REQUIRE(v_A && coords_A && r_A && coords && p, "null argument");
    std::vector<double> drawn;
    if (init == nullptr) {  // every rank draws the whole level's stream: identical on all ranks
      GE_REQUIRE(p->seed != 0, "sharded solve with init == NULL needs a fixed seed shared by all ranks");
      drawn.resize((size_t)A->rows * dim);
      level_init_stream(p->seed, *P_T, dim, drawn.data());
      init = drawn.data();
    }
    multilevel_solve(ctx, *A, *P_T, v_A, coords_A, r_A, init, coords, dim, *p, false, nullptr,
                     agg_begin, agg_end);
  });
}

ge_status ge_embed(ge_context* ctx, int n_levels, const ge_csr* As, const ge_csr* P_Ts, int dim,
                   const ge_embed_options* opt, double* coords_out, double* r_A_out,
                   double* coords_A_out, ge_embed_stats* stats) {
  return guarded([&] {
    require_ctx(ctx);
    GE_REQUIRE(n_levels >= 0 && As != nullptr && coords_out != nullptr, "null argument");
    GE_REQUIRE(n_levels == 0 || P_Ts != nullptr, "P_Ts is null");
    for (int l = 0; l <= n_levels; ++l) check_csr(&As[l], "As[l]");
    for (int l = 0; l < n_levels; ++l) {  // the asserts of src/embed.cpp:564-570
      check_csr(&P_Ts[l], "P_Ts[l]");
      GE_REQUIRE(As[l].rows == P_Ts[l].cols, "As[l].Rows() != P_Ts[l].Cols()");
      GE_REQUIRE(As[l + 1].rows == P_Ts[l].rows, "As[l+1].Rows() != P_Ts[l].Rows()");
    }
    embed_levels(ctx, n_levels, As, P_Ts, dim, opt, coords_out, r_A_out, coords_A_out, stats, nullptr);
  });
}

ge_status ge_flat_forces(ge_context* ctx, const ge_csr* A, int dim, const double* coords,
                         const ge_params* p, int path, double* forces) {
  return guarded([&] {
    require_ctx(ctx);
    check_csr(A, "A");
    GE_REQUIRE(coords && p && forces, "null argument");
    if (A->rows == 0) return;
    const bool onchip = path == 2 || (path == 0 && A->rows <= onchip_threshold());
    if (onchip) {
      std::vector<double> x(coords, coords + (size_t)A->rows * dim);
      onchip_flat_solve(ctx, *A, dim, *p, x.data(), forces, true);
      return;
    }
    std::unique_ptr<FlatSolver> s(make_flat_solver(ctx, *A, dim, *p, 0, A->rows));
    s->upload_coords(coords);
    s->launch_iteration(false);
    s->download_forces(forces);
  });
}

ge_status ge_multilevel_forces(ge_context* ctx, const ge_csr* A, const ge_csr* P_T,
                               const int32_t* v_A, const double* coords_A,
                               const double* positions, int dim, const ge_params* p,
                               double* forces) {
  return guarded([&] {
    require_ctx(ctx);
    check_csr(A, "A");
    check_csr(P_T, "P_T");
    GE_REQUIRE(v_A && coords_A && positions && p && forces, "null argument");
    std::vector<double> r_A(std::max(P_T->rows, 1), 1.0);
    multilevel_solve(ctx, *A, *P_T, v_A, coords_A, r_A.data(), positions, forces, dim, *p, true, nullptr);
  });
}

ge_status ge_level_radii(int m, int dim, double* coords_A, double* r_A, const ge_csr* A_c,
                         const ge_csr* P_T_c, const double* coords_Ac, const double* r_Ac) {
  return guarded([&] {
    GE_REQUIRE(m >= 0 && dim >= 1 && coords_A && r_A, "null argument");
    if (P_T_c != nullptr) {
      check_csr(A_c, "A_c");
      check_csr(P_T_c, "P_T_c");
      GE_REQUIRE(coords_Ac && r_Ac, "coarse centres / radii are null");
      GE_REQUIRE(P_T_c->cols == m && A_c->rows == m, "shape mismatch");
    }
    level_radii(m, dim, coords_A, r_A, A_c, P_T_c, coords_Ac, r_Ac);
  });
}

ge_status ge_level_radii_device(ge_context* ctx, int m, int dim, double* coords_A, double* r_A,
                                const ge_csr* A_c, const ge_csr* P_T_c, const double* coords_Ac,
                                const double* r_Ac) {
  return guarded([&] {
    require_ctx(ctx);
    GE_REQUIRE(m >= 0 && (dim == 2 || dim == 3) && coords_A && r_A, "bad argument");
    if (m == 0) return;
    DevBuf<double> d_x(ctx, (size_t)m * dim), d_r(ctx, (size_t)m), d_xc, d_rc;
    d_x.upload(ctx, coords_A, (size_t)m * dim);
    if (P_T_c == nullptr) {
      level_radii_device(ctx, m, dim, d_x.get(), d_r.get(), nullptr, nullptr, nullptr);
    } else {
      check_csr(A_c, "A_c");
      check_csr(P_T_c, "P_T_c");
      GE_REQUIRE(coords_Ac && r_Ac, "coarse centres / radii are null");
      GE_REQUIRE(P_T_c->cols == m && A_c->rows == m, "shape mismatch");
      GE_REQUIRE(P_T_c->indptr[P_T_c->rows] == m, "P_T_c must list every vertex exactly once");
      const int mc = P_T_c->rows;
      PrefetchedGraph g;
      g.I.alloc(ctx, (size_t)m + 1);
      g.J.alloc(ctx, (size_t)std::max<int64_t>(A_c->nnz, 1));
      g.I.upload(ctx, A_c->indptr, (size_t)m + 1);
      g.J.upload(ctx, A_c->indices, (size_t)A_c->nnz);
      g.layout = make_level_layout(ctx, *P_T_c, m);
      d_xc.alloc(ctx, (size_t)std::max(mc, 1) * dim);
      d_rc.alloc(ctx, (size_t)std::max(mc, 1));
      d_xc.upload(ctx, coords_Ac, (size_t)mc * dim);
      d_rc.upload(ctx, r_Ac, (size_t)mc);
      const RadiiLevel lv = radii_level_of(g, mc);
      level_radii_device(ctx, m, dim, d_x.get(), d_r.get(), &lv, d_xc.get(), d_rc.get());
      GE_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    d_x.download(ctx, coords_A, (size_t)m * dim);
    d_r.download(ctx, r_A, (size_t)m);
    GE_CUDA(cudaStreamSynchronize(ctx->stream));
  });
}

ge_status ge_galerkin(ge_context* ctx, const ge_csr* A, const ge_csr* P_T, int32_t* c_indptr,
                      int32_t* c_indices, double* c_data, int64_t capacity, int64_t* nnz_out,
                      ge_galerkin_stats* stats) {
  return guarded([&] {
    require_ctx(ctx);
    check_csr(A, "A");
    check_csr(P_T, "P_T");
    GE_REQUIRE(c_indptr && nnz_out, "null argument");
    *nnz_out = galerkin(ctx, *A, *P_T, c_indptr, c_indices, c_data, capacity, stats);
    GE_REQUIRE(*nnz_out <= capacity, "output capacity too small (see *nnz_out)");
  });
}

void ge_coarsen_options_default(ge_coarsen_options* opt) {
  std::memset(opt, 0, sizeof(*opt));
  opt->coarsening_factor = 0.25;
  opt->min_coarse = 64;
  opt->max_levels = 32;
  opt->seed = 0;
}

ge_status ge_coarsen(ge_context* ctx, const ge_csr* A, const ge_coarsen_options* opt,
                     ge_hierarchy** out, ge_coarsen_stats* stats) {
  return guarded([&] {
    GE_REQUIRE(out != nullptr, "out is null");
    *out = nullptr;
    require_device();
    require_ctx(ctx);  // a multi-device context: its first device
    check_csr(A, "A");
    GE_REQUIRE(opt != nullptr, "options are null");
    std::unique_ptr<ge_hierarchy> h(new ge_hierarchy);
    coarsen(ctx, *A, *opt, *h, stats);
    *out = h.release();
  });
}

ge_status ge_largest_component(ge_context* ctx, const ge_csr* A, int32_t* vertices, int32_t* n_out,
                               int32_t* c_indptr, int32_t* c_indices, double* c_data, int64_t capacity,
                               int64_t* nnz_out, int64_t* components) {
  return guarded([&] {
    require_device();
    require_ctx(ctx);  // a multi-device context: its first device
    check_csr(A, "A");
    GE_REQUIRE(A->rows == A->cols, "A must be square");
    GE_REQUIRE(vertices && n_out && c_indptr && nnz_out, "null argument");
    DevGraph G, C;
    DevBuf<int> kept;
    upload_graph(ctx, *A, G);
    check_graph(ctx, G);
    const int64_t ncomp = largest_component_device(ctx, G, C, kept);
    if (components) *components = ncomp;
    if (ncomp <= 1) {  // connected (or empty): A itself
      const int n = A->rows;
      *n_out = n;
      for (int v = 0; v < n; ++v) vertices[v] = v;
      std::memcpy(c_indptr, A->indptr, sizeof(int32_t) * ((size_t)n + 1));
      *nnz_out = A->nnz;
      GE_REQUIRE(A->nnz <= capacity, "output capacity too small (see *nnz_out)");
      GE_REQUIRE(A->nnz == 0 || (c_indices && c_data), "c_indices / c_data are null");
      if (A->nnz) std::memcpy(c_indices, A->indices, sizeof(int32_t) * (size_t)A->nnz);
      if (A->data) std::memcpy(c_data, A->data, sizeof(double) * (size_t)A->nnz);
      else std::fill(c_data, c_data + A->nnz, 1.0);
      return;
    }
    *n_out = C.n;
    *nnz_out = C.nnz;
    kept.download(ctx, vertices, (size_t)C.n);
    C.I.download(ctx, c_indptr, (size_t)C.n + 1);
    if (C.nnz <= capacity) {
      GE_REQUIRE(C.nnz == 0 || (c_indices && c_data), "c_indices / c_data are null");
      C.J.download(ctx, c_indices, (size_t)C.nnz);
      C.W.download(ctx, c_data, (size_t)C.nnz);
    }
    GE_CUDA(cudaStreamSynchronize(ctx->stream));
    GE_REQUIRE(C.nnz <= capacity, "output capacity too small (see *nnz_out)");
  });
}

ge_status ge_layout_graph(ge_context* ctx, const ge_csr* A, int dim, int32_t largest_component,
                          const ge_coarsen_options* copt, const ge_embed_options* eopt, double* coords_out,
                          int32_t* vertices_out, int32_t* n_out, ge_layout_stats* stats) {
  return guarded([&] {
    require_device();
    require_ctx(ctx);
    check_csr(A, "A");
    GE_REQUIRE(A->rows == A->cols, "A must be square");
    GE_REQUIRE(coords_out && n_out, "null argument");
    ge_coarsen_options co;
    if (copt) co = *copt;
    else ge_coarsen_options_default(&co);
    check_coarsen_options(co);
    ge_layout_stats st;
    std::memset(&st, 0, sizeof(st));
    const double t0 = now_ms();
    const int64_t launches0 = ctx->launches;
    const double h0 = ctx->h2d_bytes, d0 = ctx->d2h_bytes;
    // A goes up once; its largest component and the hierarchy stay on the device
    auto G = std::make_unique<DevGraph>();
    upload_graph(ctx, *A, *G);
    check_graph(ctx, *G);
    layout_device(ctx, std::move(G), dim, largest_component, co, eopt, coords_out, vertices_out, n_out, st);
    st.total_ms = now_ms() - t0;
    st.h2d_bytes = ctx->h2d_bytes - h0;
    st.d2h_bytes = ctx->d2h_bytes - d0;
    st.kernel_launches = ctx->launches - launches0;
    if (stats) *stats = st;
  });
}

void ge_edges_options_default(ge_edges_options* opt) {
  std::memset(opt, 0, sizeof(*opt));
  opt->symmetrize = 1;
  opt->keep_self_loops = 0;
  opt->unit_weights = 0;
}

ge_status ge_graph_from_edges(ge_context* ctx, int32_t n, int64_t E, const int32_t* src, const int32_t* dst,
                              const double* w, const ge_edges_options* opt, int32_t* c_indptr,
                              int32_t* c_indices, double* c_data, int64_t capacity, int64_t* nnz_out,
                              ge_edges_stats* stats) {
  return guarded([&] {
    require_device();
    require_ctx(ctx);  // a multi-device context: its first device
    ge_edges_options eo;
    if (opt) eo = *opt;
    else ge_edges_options_default(&eo);
    check_edges_args(n, E, src, dst, eo);
    GE_REQUIRE(c_indptr && nnz_out, "null argument");
    const double t0 = now_ms();
    ge_edges_stats st;
    std::memset(&st, 0, sizeof(st));
    DevGraph G;
    edges_to_graph_device(ctx, n, E, src, dst, w, eo, G, &st);
    *nnz_out = G.nnz;
    G.I.download(ctx, c_indptr, (size_t)n + 1);
    if (G.nnz <= capacity) {
      GE_REQUIRE(G.nnz == 0 || (c_indices && c_data), "c_indices / c_data are null");
      G.J.download(ctx, c_indices, (size_t)G.nnz);
      G.W.download(ctx, c_data, (size_t)G.nnz);
    }
    GE_CUDA(cudaStreamSynchronize(ctx->stream));
    st.total_ms = now_ms() - t0;
    if (stats) *stats = st;
    GE_REQUIRE(G.nnz <= capacity, "output capacity too small (see *nnz_out)");
  });
}

ge_status ge_layout_edges(ge_context* ctx, int32_t n, int64_t E, const int32_t* src, const int32_t* dst,
                          const double* w, const ge_edges_options* edges_opt, int dim,
                          int32_t largest_component, const ge_coarsen_options* copt,
                          const ge_embed_options* eopt, double* coords_out, int32_t* vertices_out,
                          int32_t* n_out, ge_edges_stats* edges_stats, ge_layout_stats* layout_stats) {
  return guarded([&] {
    require_device();
    require_ctx(ctx);
    ge_edges_options xo;
    if (edges_opt) xo = *edges_opt;
    else ge_edges_options_default(&xo);
    check_edges_args(n, E, src, dst, xo);
    GE_REQUIRE(coords_out && n_out, "null argument");
    ge_coarsen_options co;
    if (copt) co = *copt;
    else ge_coarsen_options_default(&co);
    check_coarsen_options(co);
    ge_layout_stats st;
    std::memset(&st, 0, sizeof(st));
    ge_edges_stats xs;
    std::memset(&xs, 0, sizeof(xs));
    const double t0 = now_ms();
    const int64_t launches0 = ctx->launches;
    const double h0 = ctx->h2d_bytes, d0 = ctx->d2h_bytes;
    // the edges go up once; the graph built from them never leaves the device
    auto G = std::make_unique<DevGraph>();
    edges_to_graph_device(ctx, n, E, src, dst, w, xo, *G, &xs);
    xs.total_ms = now_ms() - t0;
    layout_device(ctx, std::move(G), dim, largest_component, co, eopt, coords_out, vertices_out, n_out, st);
    st.total_ms = now_ms() - t0;
    st.h2d_bytes = ctx->h2d_bytes - h0;
    st.d2h_bytes = ctx->d2h_bytes - d0;
    st.kernel_launches = ctx->launches - launches0;
    if (edges_stats) *edges_stats = xs;
    if (layout_stats) *layout_stats = st;
  });
}

int32_t ge_hierarchy_levels(const ge_hierarchy* h) { return h ? (int32_t)h->aggs.size() : 0; }

namespace {
ge_csr csr_view(const HostHierarchy::Csr& c) {
  ge_csr v;
  v.rows = c.rows;
  v.cols = c.cols;
  v.nnz = (int64_t)c.indices.size();
  v.indptr = c.indptr.data();
  v.indices = c.indices.data();
  v.data = c.data.data();
  return v;
}
}  // namespace

ge_status ge_hierarchy_graph(const ge_hierarchy* h, int32_t l, ge_csr* out) {
  return guarded([&] {
    GE_REQUIRE(h != nullptr && out != nullptr, "null argument");
    GE_REQUIRE(l >= 1 && l <= (int32_t)h->graphs.size(), "level out of range (1 .. L)");
    *out = csr_view(h->graphs[l - 1]);
  });
}

ge_status ge_hierarchy_aggregation(const ge_hierarchy* h, int32_t l, ge_csr* out) {
  return guarded([&] {
    GE_REQUIRE(h != nullptr && out != nullptr, "null argument");
    GE_REQUIRE(l >= 0 && l < (int32_t)h->aggs.size(), "level out of range (0 .. L-1)");
    *out = csr_view(h->aggs[l]);
  });
}

void ge_hierarchy_destroy(ge_hierarchy* h) { delete h; }

void ge_reference_uniform(uint32_t seed, int64_t count, double* out) {
  reference_uniform(seed, count, out);
}

ge_status ge_flat_plan_create(ge_context* ctx, const ge_csr* A, int dim, const ge_params* p,
                              int32_t row_begin, int32_t row_end, ge_flat_plan** out) {
  return guarded([&] {
    require_ctx(ctx);
    check_csr(A, "A");
    GE_REQUIRE(p && out, "null argument");
    std::unique_ptr<ge_flat_plan> plan(new ge_flat_plan);
    plan->solver.reset(make_flat_solver(ctx, *A, dim, *p, row_begin, row_end));
    *out = plan.release();
  });
}
ge_status ge_flat_plan_create_symmetric(ge_context* ctx, const ge_csr* A, int dim, const ge_params* p,
                                        int32_t rank, int32_t world, ge_flat_plan** out) {
  return guarded([&] {
    require_ctx(ctx);
    check_csr(A, "A");
    GE_REQUIRE(p && out, "null argument");
    GE_REQUIRE(world >= 1 && rank >= 0 && rank < world, "bad rank / world size");
    const int64_t ld = round_up(std::max(A->rows, 1), 256 /* column tile */);
    GE_REQUIRE(ld % world == 0, "world size does not divide the padded row count");
    const int64_t R = ld / world;
    const int rb = (int)std::min<int64_t>(A->rows, rank * R);
    const int re = (int)std::min<int64_t>(A->rows, (rank + 1) * R);
    std::unique_ptr<ge_flat_plan> plan(new ge_flat_plan);
    plan->solver.reset(make_flat_solver(ctx, *A, dim, *p, rb, re, rank, world));
    GE_REQUIRE(plan->solver->symmetric(), "symmetric plan refused (graph too small, scratch too "
                                          "large, or GE_REP_SYM=0)");
    *out = plan.release();
  });
}
int32_t ge_flat_symmetric_share(int64_t ld, int32_t rank, int32_t world, int32_t capacity,
                                int32_t* blocks) {
  if (ld <= 0 || ld % 256 || world < 1 || rank < 0 || rank >= world) return -1;
  std::vector<int> v;
  sym_share(ld, rank, world, v);
  const int nb = (int)v.size() / 5;
  if (blocks)
    for (int i = 0; i < std::min(nb, (int)capacity) * 5; ++i) blocks[i] = v[i];
  return nb;
}
int32_t ge_flat_symmetric_pass_share(int64_t ld, int32_t rank, int32_t world, int32_t npass, int32_t pass,
                                     int32_t capacity, int32_t* blocks) {
  if (ld <= 0 || ld % 256 || world < 1 || rank < 0 || rank >= world || npass < 1 || pass < 0 || pass >= npass)
    return -1;
  std::vector<int> v;
  sym_pass_share(ld, rank, world, npass, pass, v);
  const int nb = (int)v.size() / 5;
  if (blocks)
    for (int i = 0; i < std::min(nb, (int)capacity) * 5; ++i) blocks[i] = v[i];
  return nb;
}
ge_status ge_embed_aggregate_ranges(const ge_csr* A, const ge_csr* P_T, int32_t ndev, int32_t* cuts,
                                    double* pairs_per_iteration) {
  return guarded([&] {
    check_csr(A, "A");
    check_csr(P_T, "P_T");
    GE_REQUIRE(ndev >= 1 && cuts != nullptr, "bad argument");
    GE_REQUIRE(P_T->cols == A->rows && P_T->indptr[P_T->rows] == A->rows, "P_T must list every vertex once");
    std::vector<int> c;
    const double pairs = aggregate_ranges(*A, *P_T, ndev, c);
    for (int d = 0; d <= ndev; ++d) cuts[d] = c[d];
    if (pairs_per_iteration) *pairs_per_iteration = pairs;
  });
}
ge_status ge_embed_aggregate_owners(const ge_csr* A, const ge_csr* P_T, int32_t ndev, int32_t* owner,
                                    double* pairs_per_iteration) {
  return guarded([&] {
    check_csr(A, "A");
    check_csr(P_T, "P_T");
    GE_REQUIRE(ndev >= 1 && owner != nullptr, "bad argument");
    GE_REQUIRE(P_T->cols == A->rows && P_T->indptr[P_T->rows] == A->rows, "P_T must list every vertex once");
    std::vector<std::vector<int>> sets;
    const double pairs = aggregate_assignment(*A, *P_T, ndev, sets);
    for (int a = 0; a < P_T->rows; ++a) owner[a] = -1;
    for (int d = 0; d < ndev; ++d)
      for (int a : sets[d]) owner[a] = d;
    if (pairs_per_iteration) *pairs_per_iteration = pairs;
  });
}
int32_t ge_flat_plan_is_symmetric(const ge_flat_plan* plan) { return plan->solver->symmetric() ? 1 : 0; }
void* ge_flat_plan_pair_sums(ge_flat_plan* plan) { return plan->solver->pair_sums(); }
ge_status ge_flat_plan_bind_pair_sums(ge_flat_plan* plan, void* dev_buf) {
  return guarded([&] {
    GE_REQUIRE(plan && dev_buf, "null argument");
    plan->solver->bind_pair_sums(dev_buf);
  });
}
ge_status ge_flat_plan_launch_repulsion(ge_flat_plan* plan) {
  return guarded([&] { plan->solver->launch_repulsion(); });
}
ge_status ge_flat_plan_launch_step(ge_flat_plan* plan) {
  return guarded([&] { plan->solver->launch_step(true); });
}
void ge_flat_plan_destroy(ge_flat_plan* plan) { delete plan; }
int64_t ge_flat_plan_ld(const ge_flat_plan* plan) { return plan->solver->ld(); }
int32_t ge_flat_plan_elem_size(const ge_flat_plan* plan) { return plan->solver->elem_size(); }
ge_status ge_flat_plan_bind_coords(ge_flat_plan* plan, void* b0, void* b1) {
  return guarded([&] {
    GE_REQUIRE(plan && b0 && b1, "null argument");
    plan->solver->bind_coords(b0, b1);
  });
}
ge_status ge_flat_plan_upload_coords(ge_flat_plan* plan, const double* coords) {
  return guarded([&] { plan->solver->upload_coords(coords); });
}
ge_status ge_flat_plan_download_coords(ge_flat_plan* plan, double* coords) {
  return guarded([&] { plan->solver->download_coords(coords); });
}
ge_status ge_flat_plan_download_forces(ge_flat_plan* plan, double* forces) {
  return guarded([&] { plan->solver->download_forces(forces); });
}
void* ge_flat_plan_cur_coords(ge_flat_plan* plan) { return plan->solver->cur_coords(); }
void* ge_flat_plan_next_coords(ge_flat_plan* plan) { return plan->solver->next_coords(); }
ge_status ge_flat_plan_launch_iteration(ge_flat_plan* plan) {
  return guarded([&] { plan->solver->launch_iteration(true); });
}
void ge_flat_plan_swap(ge_flat_plan* plan) { plan->solver->swap(); }
ge_status ge_flat_plan_iterate(ge_flat_plan* plan, int iters) {
  return guarded([&] {
    for (int it = 0; it < iters; ++it) {
      plan->solver->launch_iteration(true);
      plan->solver->swap();
    }
  });
}
ge_status ge_flat_plan_sync(ge_flat_plan* plan) {
  return guarded([&] { GE_CUDA(cudaStreamSynchronize(plan->solver->ctx->stream)); });
}
void ge_flat_plan_select_kernels(ge_flat_plan* plan, int mask) { plan->solver->select_kernels(mask); }
void ge_flat_plan_profile(ge_flat_plan* plan, int enable) { plan->solver->profile(enable != 0); }
ge_status ge_flat_plan_profile_get(ge_flat_plan* plan, double* repulsion_ms, int64_t* repulsion_launches,
                                   double* attract_step_ms, int64_t* attract_step_launches) {
  return guarded([&] {
    plan->solver->profile_get(repulsion_ms, repulsion_launches, attract_step_ms, attract_step_launches);
  });
}

}  // extern "C"

// graph-embed_b200 :: CSR from an edge list on the device (sm_100a).
//
// The result is what linalgcpp's CooMatrix (host/compat/sparsematrix.hpp) returns from ToSparse()
// after, for every edge e in order: skip it if it is a self-loop that is not kept; Add(src, dst, w);
// then, when symmetrising and src != dst, Add(dst, src, w).  Contribution `mirror` of edge e is its
// slot 2e + mirror.  Here:
//   check    a thread per edge: ids in [0, n), finite weight (device flag, as k_check_graph), and
//            the number of slots the edge keeps (0, 1 or 2)
//   emit     kept slots compacted by the scan of those counts (slot order preserved), each written
//            as the key (row << b) | col, b = bit width of n - 1, with its weight as value
//   sort     cub::DeviceRadixSort on bits [0, 2b): SortPairs in sum mode, SortKeys in unit mode.
//            The sort is stable, so equal keys stay in slot order: the reduction below adds the
//            duplicates in exactly the order CooMatrix's `+=` does
//   reduce   run heads flagged and scanned into output positions; a thread per run head writes the
//            column and sums up to kShortRun values from +0.0; longer runs (raw R-MAT-20 has runs of
//            hundreds of duplicates) are queued for a warp that fetches 32 values at a time and adds
//            them in order through shuffles (the Galerkin run reducer's technique, ge_galerkin.cu)
//   rowptr   a thread per row: lower bound of the row in the rows of the unique entries (no atomics,
//            empty rows anywhere come out right)
#include <cub/cub.cuh>

#include <algorithm>
#include <climits>

#include "ge_context.h"

namespace ge {

namespace {

constexpr int kShortRun = 32;
using Key = unsigned long long;

unsigned grid_of(int64_t n, int threads) { return (unsigned)std::max<int64_t>(1, (n + threads - 1) / threads); }

// bad: 1 = id outside [0, n), 2 = non-finite weight
__global__ void __launch_bounds__(256) k_edges_check(const int* __restrict__ src, const int* __restrict__ dst,
                                                     const double* __restrict__ w, int64_t E, int n,
                                                     int symmetrize, int keep_loops, int* __restrict__ count,
                                                     int* __restrict__ bad) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  const int s = src[e], d = dst[e];
  if (s < 0 || s >= n || d < 0 || d >= n) atomicOr(bad, 1);
  if (w && !isfinite(w[e])) atomicOr(bad, 2);
  count[e] = s == d ? keep_loops : 1 + symmetrize;
}

__global__ void __launch_bounds__(256) k_edges_emit(const int* __restrict__ src, const int* __restrict__ dst,
                                                    const double* __restrict__ w, int64_t E, int b,
                                                    const int* __restrict__ pos, Key* __restrict__ keys,
                                                    double* __restrict__ vals) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  const int p = pos[e], cnt = pos[e + 1] - p;
  if (cnt == 0) return;
  const Key s = (unsigned)src[e], d = (unsigned)dst[e];
  keys[p] = (s << b) | d;
  if (cnt == 2) keys[p + 1] = (d << b) | s;
  if (vals) {
    const double v = w ? w[e] : 1.0;
    vals[p] = v;
    if (cnt == 2) vals[p + 1] = v;
  }
}

__global__ void __launch_bounds__(256) k_edges_heads(const Key* __restrict__ keys, int S, int* __restrict__ head) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < S) head[i] = i == 0 || keys[i] != keys[i - 1];
}

struct ReduceArgs {
  const Key* keys;
  const double* vals;  // nullptr: unit mode
  const int* upos;     // [S+1]: output position of each slot's run (exclusive scan of the heads)
  int S, b;
  int* row;            // [U] row of each unique entry
  int* col;            // [U]
  double* out;         // [U]
  int* long_head;      // slots that start a run longer than kShortRun
  int* long_n;
};

// a thread per slot; run heads write their entry
__global__ void __launch_bounds__(256) k_edges_reduce(ReduceArgs a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.S) return;
  const int u = a.upos[i];
  if (a.upos[i + 1] == u) return;  // not a run head
  const Key k = a.keys[i];
  a.row[u] = (int)(k >> a.b);
  a.col[u] = (int)(k & ((Key(1) << a.b) - 1));
  if (!a.vals) {
    a.out[u] = 1.0;
    return;
  }
  double sum = 0.0;
  int r = i;
  for (; r < a.S && r < i + kShortRun && a.keys[r] == k; ++r) sum += a.vals[r];
  if (r < a.S && r == i + kShortRun && a.keys[r] == k) a.long_head[atomicAdd(a.long_n, 1)] = i;
  else a.out[u] = sum;
}

// a warp per long run: the lanes load 32 consecutive values, every lane then adds them in run order
// (the same additions as one thread walking the run, with the loads taken out of the chain)
__global__ void __launch_bounds__(256) k_edges_reduce_long(ReduceArgs a) {
  const int lane = threadIdx.x & 31;
  const int nq = *a.long_n;
  const int stride = gridDim.x * (blockDim.x >> 5);
  for (int q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); q < nq; q += stride) {
    const int r0 = a.long_head[q];
    const Key k = a.keys[r0];
    double sum = 0.0;
    for (int c = r0;; c += 32) {
      const int r = c + lane;
      const bool ok = r < a.S && a.keys[r] == k;
      const double v = ok ? a.vals[r] : 0.0;
      const int cnt = __popc(__ballot_sync(0xffffffffu, ok));  // the run is contiguous: lanes 0 .. cnt-1
      for (int l = 0; l < cnt; ++l) sum += __shfl_sync(0xffffffffu, v, l);
      if (cnt < 32) break;
    }
    if (lane == 0) a.out[a.upos[r0]] = sum;
  }
}

// indptr[r] = first unique entry of a row >= r (rows ascending)
__global__ void __launch_bounds__(256) k_edges_rowptr(const int* __restrict__ row, int U, int n,
                                                      int* __restrict__ indptr) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r > n) return;
  int lo = 0, hi = U;
  while (lo < hi) {
    const int mid = (int)(((unsigned)lo + (unsigned)hi) >> 1);
    if (row[mid] < r) lo = mid + 1;
    else hi = mid;
  }
  indptr[r] = lo;
}

int read_int(ge_context* ctx, const int* d) {
  int h = 0;
  GE_CUDA(cudaMemcpyAsync(&h, d, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  GE_CUDA(cudaStreamSynchronize(ctx->stream));
  return h;
}

}  // namespace

void check_edges_args(int64_t n, int64_t E, const int32_t* src, const int32_t* dst, const ge_edges_options& opt) {
  GE_REQUIRE(n >= 0 && n <= INT_MAX, "n must lie in [0, 2^31)");
  GE_REQUIRE(E >= 0, "E must be >= 0");
  GE_REQUIRE(E == 0 || (src && dst), "src / dst are null");
  // every slot, and so every output entry, must be addressable by int32 row pointers
  GE_REQUIRE(E <= (int64_t)INT_MAX / (opt.symmetrize ? 2 : 1), "too many edges for int32 row pointers");
}

void edges_to_graph_device(ge_context* ctx, int n, int64_t E, const int32_t* src, const int32_t* dst,
                           const double* w, const ge_edges_options& opt, DevGraph& out, ge_edges_stats* stats) {
  check_edges_args(n, E, src, dst, opt);
  cudaStream_t s = ctx->stream;
  const int64_t launches0 = ctx->launches;
  const bool sum_mode = !opt.unit_weights;
  int b = 1;  // bit width of n - 1 (at least 1)
  while (b < 31 && (int64_t(1) << b) < n) ++b;

  DevBuf<int> d_src(ctx, E), d_dst(ctx, E);
  DevBuf<double> d_w;
  d_src.upload(ctx, src, E);
  d_dst.upload(ctx, dst, E);
  if (w) {
    d_w.alloc(ctx, E);
    d_w.upload(ctx, w, E);
  }
  cudaEvent_t ev[2];
  for (auto& e : ev) GE_CUDA(cudaEventCreate(&e));
  struct Events {
    cudaEvent_t* e;
    ~Events() {
      cudaEventDestroy(e[0]);
      cudaEventDestroy(e[1]);
    }
  } events{ev};
  GE_CUDA(cudaEventRecord(ev[0], s));

  // check, count and compact the kept slots
  DevBuf<int> count(ctx, std::max<int64_t>(E, 1)), pos(ctx, (size_t)E + 1), bad(ctx, 1);
  bad.zero(s);
  k_edges_check<<<grid_of(E, 256), 256, 0, s>>>(d_src.get(), d_dst.get(), d_w.get(), E, n, opt.symmetrize ? 1 : 0,
                                                opt.keep_self_loops ? 1 : 0, count.get(), bad.get());
  GE_CUDA(cudaGetLastError());
  ctx->launches++;
  exclusive_scan(ctx, count.get(), (int)E, pos.get());
  int info[2] = {0, 0};  // bad flag, slot count
  GE_CUDA(cudaMemcpyAsync(&info[0], bad.get(), sizeof(int), cudaMemcpyDeviceToHost, s));
  GE_CUDA(cudaMemcpyAsync(&info[1], pos.get() + E, sizeof(int), cudaMemcpyDeviceToHost, s));
  GE_CUDA(cudaStreamSynchronize(s));
  GE_REQUIRE(!(info[0] & 1), "an edge has a vertex id outside [0, n)");
  GE_REQUIRE(!(info[0] & 2), "an edge weight is not finite");
  const int S = info[1];
  count.release();

  DevBuf<Key> k0(ctx, std::max(S, 1)), k1(ctx, std::max(S, 1));
  DevBuf<double> v0, v1;
  if (sum_mode) {
    v0.alloc(ctx, std::max(S, 1));
    v1.alloc(ctx, std::max(S, 1));
  }
  k_edges_emit<<<grid_of(E, 256), 256, 0, s>>>(d_src.get(), d_dst.get(), d_w.get(), E, b, pos.get(), k0.get(),
                                               v0.get());
  GE_CUDA(cudaGetLastError());
  ctx->launches++;
  pos.release();
  d_src.release();
  d_dst.release();
  d_w.release();

  // stable radix sort on the 2b key bits: equal keys keep their slot order, which fixes the order of
  // the additions below
  cub::DoubleBuffer<Key> keys(k0.get(), k1.get());
  cub::DoubleBuffer<double> vals(v0.get(), v1.get());
  if (S > 1) {
    size_t bytes = 0;
    if (sum_mode) GE_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, bytes, keys, vals, S, 0, 2 * b, s));
    else GE_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, bytes, keys, S, 0, 2 * b, s));
    DevBuf<unsigned char> temp(ctx, std::max<size_t>(bytes, 1));
    if (sum_mode) GE_CUDA(cub::DeviceRadixSort::SortPairs(temp.get(), bytes, keys, vals, S, 0, 2 * b, s));
    else GE_CUDA(cub::DeviceRadixSort::SortKeys(temp.get(), bytes, keys, S, 0, 2 * b, s));
    ctx->launches++;
  }

  // runs of equal keys -> unique entries
  DevBuf<int> head(ctx, std::max(S, 1)), upos(ctx, (size_t)S + 1);
  k_edges_heads<<<grid_of(S, 256), 256, 0, s>>>(keys.Current(), S, head.get());
  GE_CUDA(cudaGetLastError());
  ctx->launches++;
  exclusive_scan(ctx, head.get(), S, upos.get());
  head.release();
  const int U = read_int(ctx, upos.get() + S);
  DevBuf<int> row(ctx, std::max(U, 1)), long_head(ctx, S / (kShortRun + 1) + 1), long_n(ctx, 1);
  out.n = n;
  out.nnz = U;
  out.I.alloc(ctx, (size_t)n + 1);
  out.J.alloc(ctx, std::max(U, 1));
  out.W.alloc(ctx, std::max(U, 1));
  long_n.zero(s);
  ReduceArgs a;
  a.keys = keys.Current();
  a.vals = sum_mode ? vals.Current() : nullptr;
  a.upos = upos.get();
  a.S = S;
  a.b = b;
  a.row = row.get();
  a.col = out.J.get();
  a.out = out.W.get();
  a.long_head = long_head.get();
  a.long_n = long_n.get();
  k_edges_reduce<<<grid_of(S, 256), 256, 0, s>>>(a);
  ctx->launches++;
  if (sum_mode) {
    k_edges_reduce_long<<<(unsigned)std::max(1, ctx->sm_count * 8), 256, 0, s>>>(a);
    ctx->launches++;
  }
  k_edges_rowptr<<<grid_of((int64_t)n + 1, 256), 256, 0, s>>>(row.get(), U, n, out.I.get());
  GE_CUDA(cudaGetLastError());
  ctx->launches++;
  GE_CUDA(cudaEventRecord(ev[1], s));
  if (stats) {
    GE_CUDA(cudaEventSynchronize(ev[1]));
    float ms = 0;
    GE_CUDA(cudaEventElapsedTime(&ms, ev[0], ev[1]));
    stats->device_ms = ms;
    stats->nnz = U;
    // S = (E - loops) * (1 + symmetrize) + loops * keep_self_loops
    const int64_t per = opt.symmetrize ? 2 : 1;
    stats->self_loops_dropped = opt.keep_self_loops ? 0 : E - S / per;
    stats->duplicates_merged = (int64_t)S - U;
    stats->kernel_launches = ctx->launches - launches0;
  }
}

}  // namespace ge

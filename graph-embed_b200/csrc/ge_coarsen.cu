// graph-embed_b200 :: multilevel hierarchy on the device (sm_100a): ge_coarsen.
//
// Random-mate matching, the algorithm of the stand-in generator graphs.coarsen, made a pure
// function of (A, options) by counter-based hashing; tests/coarsen_restatement.py restates it on
// the host and the device reproduces it bit for bit.  One round on the current graph S (m vertices):
//   degree   k_i = sum of row i in CSR order (self-loop included), 1 where k_i <= 0
//   coin     head[v] = top bit of H(0, v)
//   propose  tail i takes the head neighbour j != i with the largest w_ij / (k_i * k_j); ties to
//            the smaller H(2, i << 32 | j), then the smaller j (a total order: any reduction tree
//            gives the same winner)
//   truncate when more than M - target tails found a head, the M - target smallest (H(1, i), i)
//   relabel  the survivors (heads and unmatched tails) are renumbered in ascending id order and a
//            tail takes its head's new id; the level's map is the composition of its rounds' maps
//   contract S <- Q S Q^T with the Galerkin product of ge_galerkin.cu (same kernels, device inputs)
// with H(tag, v) = mix64(mix64(seed << 32 | level << 20 | round << 4 | tag) ^ v), mix64 = the
// splitmix64 finaliser.  Everything stays on the device between the upload of A and the download
// of the levels at the end; the host reads a handful of counters per round (candidate count,
// survivor count, segment offsets for the Galerkin size classes).
#include <cub/cub.cuh>

#include <algorithm>
#include <cmath>
#include <memory>
#include <vector>

#include "ge_context.h"

namespace ge {

namespace {

constexpr int kHubRow = 1024;     // rows longer than this take a whole CTA (R-MAT hubs: 10^4 entries)
constexpr int kHubThreads = 512;
constexpr int kWarpRows = 8;      // rows per 256-thread CTA in the warp-per-row kernels

__host__ __device__ __forceinline__ uint64_t mix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

uint64_t hash_base(uint32_t seed, int level, int round, int tag) {
  return mix64(((uint64_t)seed << 32) | ((uint64_t)level << 20) | ((uint64_t)round << 4) | (uint64_t)tag);
}

struct RoundArgs {
  int m;
  const int* I;
  const int* J;
  const double* W;  // nullptr: unit weights
  uint64_t base_coin, base_tie;
  double* k;
  unsigned char* head;
  int* choice;          // chosen head, -1 for heads and tails without a candidate
  unsigned char* cand;  // choice >= 0
  int* hubs;            // rows longer than kHubRow
  int* nhub;
};

// Integer weights whose magnitudes add up to at most 2^50 sum exactly in any order; anything else
// is added sequentially in CSR order (the definition).  Unit weights: the row length.
constexpr double kExactIntSum = 1125899906842624.0;  // 2^50

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}

// sum of W[e0 .. e0+len) in order, by one warp: lanes fetch 32 values, lane order adds them
__device__ double warp_sequential_sum(const double* W, int e0, int len, int lane) {
  double s = 0.0;
  for (int c = 0; c < len; c += 32) {
    const double v = c + lane < len ? W[e0 + c + lane] : 0.0;
    const int cnt = min(32, len - c);
    for (int l = 0; l < cnt; ++l) s += __shfl_sync(0xffffffffu, v, l);
  }
  return s;
}

__global__ void __launch_bounds__(256) k_classify(RoundArgs a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.m) return;
  a.head[i] = (unsigned char)(mix64(a.base_coin ^ (uint64_t)i) >> 63);
  if (a.I[i + 1] - a.I[i] > kHubRow) a.hubs[atomicAdd(a.nhub, 1)] = i;
}

__device__ __forceinline__ void store_degree(const RoundArgs& a, int i, double s) {
  a.k[i] = s > 0.0 ? s : 1.0;
}

__global__ void __launch_bounds__(256) k_degree_warp(RoundArgs a) {
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * kWarpRows + (threadIdx.x >> 5);
  if (i >= a.m) return;
  const int e0 = a.I[i], len = a.I[i + 1] - e0;
  if (len > kHubRow) return;
  if (a.W == nullptr) {
    if (lane == 0) store_degree(a, i, (double)len);
    return;
  }
  double part = 0.0, mag = 0.0;
  bool integral = true;
  for (int t = lane; t < len; t += 32) {
    const double v = a.W[e0 + t];
    part += v;
    mag += fabs(v);
    integral = integral && v == trunc(v);
  }
  part = warp_sum(part);
  mag = warp_sum(mag);
  double s = part;
  if (!__all_sync(0xffffffffu, integral) || !(mag <= kExactIntSum)) s = warp_sequential_sum(a.W, e0, len, lane);
  if (lane == 0) store_degree(a, i, s);
}

__global__ void __launch_bounds__(kHubThreads) k_degree_hub(RoundArgs a) {
  __shared__ double s_part[kHubThreads / 32], s_mag[kHubThreads / 32];
  __shared__ int s_int[kHubThreads / 32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int nhub = *a.nhub;
  for (int b = blockIdx.x; b < nhub; b += gridDim.x) {
    const int i = a.hubs[b];
    const int e0 = a.I[i], len = a.I[i + 1] - e0;
    if (a.W == nullptr) {
      if (threadIdx.x == 0) store_degree(a, i, (double)len);
      continue;
    }
    double part = 0.0, mag = 0.0;
    bool integral = true;
    for (int t = threadIdx.x; t < len; t += kHubThreads) {
      const double v = a.W[e0 + t];
      part += v;
      mag += fabs(v);
      integral = integral && v == trunc(v);
    }
    part = warp_sum(part);
    mag = warp_sum(mag);
    const bool wint = __all_sync(0xffffffffu, integral);
    if (lane == 0) {
      s_part[w] = part;
      s_mag[w] = mag;
      s_int[w] = wint;
    }
    __syncthreads();
    if (w == 0) {
      double p = 0.0, g = 0.0;
      bool all = true;
      for (int q = 0; q < kHubThreads / 32; ++q) {
        p += s_part[q];
        g += s_mag[q];
        all = all && s_int[q];
      }
      double s = p;
      if (!all || !(g <= kExactIntSum)) s = warp_sequential_sum(a.W, e0, len, lane);
      if (lane == 0) store_degree(a, i, s);
    }
    __syncthreads();
  }
}

struct Best {
  double s;
  uint64_t h;
  int j;  // -1: none
};

// the total order of the proposal: larger score, then smaller hash, then smaller id
__device__ __forceinline__ bool better(const Best& x, const Best& y) {
  if (x.j < 0) return false;
  if (y.j < 0) return true;
  if (x.s != y.s) return x.s > y.s;
  if (x.h != y.h) return x.h < y.h;
  return x.j < y.j;
}

__device__ __forceinline__ void scan_entries(const RoundArgs& a, int i, double ki, int e0, int len,
                                             int t0, int stride, Best& best) {
  for (int t = t0; t < len; t += stride) {
    const int e = e0 + t;
    const int j = a.J[e];
    if (j == i || !a.head[j]) continue;
    const double w = a.W ? a.W[e] : 1.0;
    Best c;
    c.s = __ddiv_rn(w, __dmul_rn(ki, a.k[j]));  // an IEEE multiply, then a divide: no FMA
    c.h = mix64(a.base_tie ^ (((uint64_t)(uint32_t)i << 32) | (uint64_t)(uint32_t)j));
    c.j = j;
    if (better(c, best)) best = c;
  }
}

__device__ __forceinline__ Best warp_best(Best b) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    Best o;
    o.s = __shfl_xor_sync(0xffffffffu, b.s, off);
    o.h = __shfl_xor_sync(0xffffffffu, b.h, off);
    o.j = __shfl_xor_sync(0xffffffffu, b.j, off);
    if (better(o, b)) b = o;
  }
  return b;
}

__device__ __forceinline__ void store_choice(const RoundArgs& a, int i, int j) {
  a.choice[i] = j;
  a.cand[i] = j >= 0;
}

__global__ void __launch_bounds__(256) k_propose_warp(RoundArgs a) {
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * kWarpRows + (threadIdx.x >> 5);
  if (i >= a.m) return;
  const int e0 = a.I[i], len = a.I[i + 1] - e0;
  if (len > kHubRow) return;
  if (a.head[i]) {
    if (lane == 0) store_choice(a, i, -1);
    return;
  }
  Best b;
  b.s = 0.0;
  b.h = 0;
  b.j = -1;
  scan_entries(a, i, a.k[i], e0, len, lane, 32, b);
  b = warp_best(b);
  if (lane == 0) store_choice(a, i, b.j);
}

__global__ void __launch_bounds__(kHubThreads, 1) k_propose_hub(RoundArgs a) {
  __shared__ double s_s[kHubThreads / 32];
  __shared__ unsigned long long s_h[kHubThreads / 32];
  __shared__ int s_j[kHubThreads / 32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int nhub = *a.nhub;
  for (int q = blockIdx.x; q < nhub; q += gridDim.x) {
    const int i = a.hubs[q];
    if (a.head[i]) {
      if (threadIdx.x == 0) store_choice(a, i, -1);
      continue;
    }
    const int e0 = a.I[i], len = a.I[i + 1] - e0;
    Best b;
    b.s = 0.0;
    b.h = 0;
    b.j = -1;
    scan_entries(a, i, a.k[i], e0, len, threadIdx.x, kHubThreads, b);
    b = warp_best(b);
    if (lane == 0) {
      s_s[w] = b.s;
      s_h[w] = b.h;
      s_j[w] = b.j;
    }
    __syncthreads();
    if (w == 0) {
      Best c;
      c.j = -1;
      c.s = 0.0;
      c.h = 0;
      if (lane < kHubThreads / 32) {
        c.s = s_s[lane];
        c.h = s_h[lane];
        c.j = s_j[lane];
      }
      c = warp_best(c);
      if (lane == 0) store_choice(a, i, c.j);
    }
    __syncthreads();
  }
}

__global__ void k_iota(int* x, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] = i;
}

__global__ void k_trunc_keys(const int* tails, int n, uint64_t base, unsigned long long* keys) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) keys[t] = mix64(base ^ (uint64_t)tails[t]);
}

// tails past the first `keep` of the sorted (H(1, i), i) order do not merge this round
__global__ void k_trunc_drop(const int* sorted_tails, int keep, int n, int* choice) {
  const int t = keep + blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) choice[sorted_tails[t]] = -1;
}

__global__ void k_survivors(const int* choice, int m, int* surv) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m) surv[i] = choice[i] < 0;
}

__global__ void k_relabel(const int* choice, const int* newid, int m, int* label) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m) label[i] = newid[choice[i] >= 0 ? choice[i] : i];
}

__global__ void k_compose(int* agg, const int* label, int n) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v < n) agg[v] = label[agg[v]];
}

// P_T row pointers from the vertex -> aggregate map sorted by aggregate (every aggregate non-empty)
__global__ void k_rowptr(const int* sorted_agg, int n, int m, int* Pptr) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  if (t == 0 || sorted_agg[t] != sorted_agg[t - 1]) Pptr[sorted_agg[t]] = t;
  if (t == 0) Pptr[m] = n;
}

__global__ void k_member_rowlen(const int* I, const int* Pidx, int n, int* len) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < n) len[c] = I[Pidx[c] + 1] - I[Pidx[c]];
}

// segment offsets of the Galerkin product from the scanned member row lengths pos [n+1]
__global__ void k_segments(const int* pos, const int* Pptr, const int* Pidx, const int* sorted_agg,
                           int n, int m, int* segoff, int* rowoff) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t <= m) segoff[t] = pos[Pptr[t]];
  if (t < n) rowoff[Pidx[t]] = pos[t] - pos[Pptr[sorted_agg[t]]];
}

__global__ void k_check_graph(const int* I, const int* J, int n, int* bad) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int e0 = I[i], e1 = I[i + 1];
  if (e1 < e0) {
    *bad = 1;
    return;
  }
  for (int e = e0; e < e1; ++e)
    if (J[e] < 0 || J[e] >= n) *bad = 1;
}

unsigned grid_of(int64_t n, int threads) { return (unsigned)std::max<int64_t>(1, (n + threads - 1) / threads); }

class Coarsener {
 public:
  explicit Coarsener(ge_context* ctx) : ctx_(ctx) {}

  // CUB temporary storage, grown as needed
  void* temp(size_t bytes) {
    if (bytes > temp_.size()) temp_.alloc(ctx_, bytes);
    return temp_.get();
  }

  // stable sort of (key, iota) pairs: the vertices grouped by key, ascending ids inside a group
  template <typename K>
  void sort_pairs(const K* keys, K* keys_out, const int* vals, int* vals_out, int n, int end_bit) {
    size_t bytes = 0;
    GE_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, bytes, keys, keys_out, vals, vals_out, n, 0, end_bit,
                                            ctx_->stream));
    GE_CUDA(cub::DeviceRadixSort::SortPairs(temp(bytes), bytes, keys, keys_out, vals, vals_out, n, 0,
                                            end_bit, ctx_->stream));
    ctx_->launches++;
  }

  // P_T of a vertex -> aggregate map (n vertices, m aggregates): members ascending per row
  void aggregation(const int* agg, int n, int m, DevBuf<int>& ptr, DevBuf<int>& idx, DevBuf<int>& sorted) {
    ptr.alloc(ctx_, (size_t)m + 1);
    idx.alloc(ctx_, std::max(n, 1));
    sorted.alloc(ctx_, std::max(n, 1));
    int bits = 1;
    while (bits < 31 && (1 << bits) < m) ++bits;
    sort_pairs(agg, sorted.get(), iota_.get(), idx.get(), n, bits);
    k_rowptr<<<grid_of(n, 256), 256, 0, ctx_->stream>>>(sorted.get(), n, m, ptr.get());
    GE_CUDA(cudaGetLastError());
    ctx_->launches++;
  }

  // S <- Q S Q^T for the round's map `label` (S.n -> m)
  DevGraph contract(const DevGraph& S, const int* label, int m) {
    const int n = S.n;
    DevBuf<int> Pptr, Pidx, sorted, len(ctx_, std::max(n, 1)), pos(ctx_, (size_t)n + 1),
        segoff(ctx_, (size_t)m + 1), rowoff(ctx_, std::max(n, 1));
    aggregation(label, n, m, Pptr, Pidx, sorted);
    k_member_rowlen<<<grid_of(n, 256), 256, 0, ctx_->stream>>>(S.I.get(), Pidx.get(), n, len.get());
    exclusive_scan(ctx_, len.get(), n, pos.get());
    k_segments<<<grid_of(std::max(n, m + 1), 256), 256, 0, ctx_->stream>>>(
        pos.get(), Pptr.get(), Pidx.get(), sorted.get(), n, m, segoff.get(), rowoff.get());
    GE_CUDA(cudaGetLastError());
    ctx_->launches += 2;
    std::vector<int> segoff_host((size_t)m + 1);
    segoff.download(ctx_, segoff_host.data(), (size_t)m + 1);
    GE_CUDA(cudaStreamSynchronize(ctx_->stream));
    GalerkinInput in;
    in.n = n;
    in.m = m;
    in.I = S.I.get();
    in.J = S.J.get();
    in.W = S.w();
    in.vA = label;
    in.Pptr = Pptr.get();
    in.Pidx = Pidx.get();
    in.rowoff = rowoff.get();
    in.segoff = segoff.get();
    DevGraph C;
    C.n = m;
    C.nnz = (int)galerkin_device(ctx_, in, segoff_host.data(), nullptr, C.I, C.J, C.W, S.nnz, nullptr);
    if (C.nnz == 0) {  // no entries: keep the arrays non-null
      C.J.alloc(ctx_, 1);
      C.W.alloc(ctx_, 1);
    }
    return C;
  }

  // One round on S (level `level`, round `round`): the map S.n -> *m_out, or false without candidates.
  bool round(const DevGraph& S, uint32_t seed, int level, int rnd, int max_merges, DevBuf<int>& label,
             int* m_out) {
    const int m = S.n;
    DevBuf<double> k(ctx_, std::max(m, 1));
    DevBuf<unsigned char> head(ctx_, std::max(m, 1)), cand(ctx_, std::max(m, 1));
    DevBuf<int> choice(ctx_, std::max(m, 1)), hubs(ctx_, std::max(m, 1)), counters(ctx_, 2),
        tails(ctx_, std::max(m, 1));
    counters.zero(ctx_->stream);
    RoundArgs a;
    a.m = m;
    a.I = S.I.get();
    a.J = S.J.get();
    a.W = S.w();
    a.base_coin = hash_base(seed, level, rnd, 0);
    a.base_tie = hash_base(seed, level, rnd, 2);
    a.k = k.get();
    a.head = head.get();
    a.choice = choice.get();
    a.cand = cand.get();
    a.hubs = hubs.get();
    a.nhub = counters.get();
    const unsigned hub_grid = (unsigned)std::max(1, ctx_->sm_count * 2);
    k_classify<<<grid_of(m, 256), 256, 0, ctx_->stream>>>(a);
    k_degree_warp<<<grid_of(m, kWarpRows), 256, 0, ctx_->stream>>>(a);
    k_degree_hub<<<hub_grid, kHubThreads, 0, ctx_->stream>>>(a);
    k_propose_warp<<<grid_of(m, kWarpRows), 256, 0, ctx_->stream>>>(a);
    k_propose_hub<<<hub_grid, kHubThreads, 0, ctx_->stream>>>(a);
    GE_CUDA(cudaGetLastError());
    ctx_->launches += 5;
    // the tails that found a head, ascending
    size_t bytes = 0;
    int* ncand_d = counters.get() + 1;
    GE_CUDA(cub::DeviceSelect::Flagged(nullptr, bytes, iota_.get(), cand.get(), tails.get(), ncand_d, m,
                                       ctx_->stream));
    GE_CUDA(cub::DeviceSelect::Flagged(temp(bytes), bytes, iota_.get(), cand.get(), tails.get(), ncand_d, m,
                                       ctx_->stream));
    ctx_->launches++;
    int ncand = 0;
    GE_CUDA(cudaMemcpyAsync(&ncand, ncand_d, sizeof(int), cudaMemcpyDeviceToHost, ctx_->stream));
    GE_CUDA(cudaStreamSynchronize(ctx_->stream));
    if (ncand == 0) return false;
    if (ncand > max_merges) {  // keep the max_merges smallest (H(1, i), i): a stable sort on H(1, i)
      DevBuf<unsigned long long> keys(ctx_, ncand), keys_out(ctx_, ncand);
      DevBuf<int> sorted(ctx_, ncand);
      k_trunc_keys<<<grid_of(ncand, 256), 256, 0, ctx_->stream>>>(tails.get(), ncand,
                                                                   hash_base(seed, level, rnd, 1), keys.get());
      sort_pairs<unsigned long long>(keys.get(), keys_out.get(), tails.get(), sorted.get(), ncand, 64);
      k_trunc_drop<<<grid_of(ncand - max_merges, 256), 256, 0, ctx_->stream>>>(sorted.get(), max_merges,
                                                                                ncand, choice.get());
      GE_CUDA(cudaGetLastError());
      ctx_->launches += 2;
    }
    DevBuf<int> surv(ctx_, std::max(m, 1)), newid(ctx_, (size_t)m + 1);
    k_survivors<<<grid_of(m, 256), 256, 0, ctx_->stream>>>(choice.get(), m, surv.get());
    exclusive_scan(ctx_, surv.get(), m, newid.get());
    label.alloc(ctx_, std::max(m, 1));
    k_relabel<<<grid_of(m, 256), 256, 0, ctx_->stream>>>(choice.get(), newid.get(), m, label.get());
    GE_CUDA(cudaGetLastError());
    ctx_->launches += 2;
    GE_CUDA(cudaMemcpyAsync(m_out, newid.get() + m, sizeof(int), cudaMemcpyDeviceToHost, ctx_->stream));
    GE_CUDA(cudaStreamSynchronize(ctx_->stream));
    return true;
  }

  // Levels of h.graphs[0] until min_coarse, max_levels or a level that merges nothing.
  void build(DeviceHierarchy& h, const ge_coarsen_options& opt, bool check, int64_t* rounds_out) {
    const DevGraph& S0 = *h.graphs[0];
    const int n0 = S0.n;
    iota_.alloc(ctx_, std::max(n0, 1));
    if (check) check_graph(ctx_, S0);
    k_iota<<<grid_of(n0, 256), 256, 0, ctx_->stream>>>(iota_.get(), n0);
    GE_CUDA(cudaGetLastError());
    ctx_->launches++;
    int64_t rounds = 0;
    const DevGraph* level_graph = &S0;
    while (level_graph->n > opt.min_coarse && h.levels() < opt.max_levels) {
      const int level = h.levels();
      const int N = level_graph->n;
      const int target = std::max((int)std::floor(opt.coarsening_factor * (double)N), opt.min_coarse);
      DevBuf<int> agg(ctx_, std::max(N, 1));
      GE_CUDA(cudaMemcpyAsync(agg.get(), iota_.get(), sizeof(int) * (size_t)N, cudaMemcpyDeviceToDevice,
                              ctx_->stream));
      int M = N;
      DevGraph S;  // the level's graph after its latest round
      const DevGraph* cur = level_graph;
      for (int rnd = 0; M > target; ++rnd) {
        DevBuf<int> label;
        int M2 = 0;
        ++rounds;
        if (!round(*cur, opt.seed, level, rnd, M - target, label, &M2)) break;
        k_compose<<<grid_of(N, 256), 256, 0, ctx_->stream>>>(agg.get(), label.get(), N);
        GE_CUDA(cudaGetLastError());
        ctx_->launches++;
        DevGraph C = contract(*cur, label.get(), M2);
        S = std::move(C);
        cur = &S;
        M = M2;
      }
      if (M == N) break;
      auto P = std::make_unique<DevAgg>();
      P->m = M;
      P->n = N;
      DevBuf<int> sorted;
      aggregation(agg.get(), N, M, P->ptr, P->idx, sorted);
      h.aggs.push_back(std::move(P));
      h.graphs.push_back(std::make_unique<DevGraph>(std::move(S)));
      level_graph = h.graphs.back().get();
    }
    if (rounds_out) *rounds_out = rounds;
  }

  void run(const ge_csr& A, const ge_coarsen_options& opt, HostHierarchy& out, ge_coarsen_stats* stats) {
    const double t_begin = now_ms();
    const int64_t launches0 = ctx_->launches;
    DeviceHierarchy h;
    h.graphs.push_back(std::make_unique<DevGraph>());
    upload_graph(ctx_, A, *h.graphs[0]);
    cudaEvent_t ev0, ev1;
    GE_CUDA(cudaEventCreate(&ev0));
    GE_CUDA(cudaEventCreate(&ev1));
    struct Events {
      cudaEvent_t a, b;
      ~Events() {
        cudaEventDestroy(a);
        cudaEventDestroy(b);
      }
    } events{ev0, ev1};
    GE_CUDA(cudaEventRecord(ev0, ctx_->stream));
    int64_t rounds = 0;
    build(h, opt, true, &rounds);
    // one download of every level
    const int L = h.levels();
    out.graphs.assign(L, HostHierarchy::Csr());
    out.aggs.assign(L, HostHierarchy::Csr());
    for (int l = 0; l < L; ++l) {
      const DevGraph& G = *h.graphs[l + 1];
      HostHierarchy::Csr& g = out.graphs[l];
      g.rows = g.cols = G.n;
      g.indptr.resize((size_t)G.n + 1);
      g.indices.resize(G.nnz);
      g.data.resize(G.nnz);
      G.I.download(ctx_, g.indptr.data(), (size_t)G.n + 1);
      G.J.download(ctx_, g.indices.data(), G.nnz);
      G.W.download(ctx_, g.data.data(), G.nnz);
      const DevAgg& P = *h.aggs[l];
      HostHierarchy::Csr& p = out.aggs[l];
      p.rows = P.m;
      p.cols = P.n;
      p.indptr.resize((size_t)P.m + 1);
      p.indices.resize(P.n);
      p.data.assign(P.n, 1.0);
      P.ptr.download(ctx_, p.indptr.data(), (size_t)P.m + 1);
      P.idx.download(ctx_, p.indices.data(), P.n);
    }
    GE_CUDA(cudaEventRecord(ev1, ctx_->stream));
    GE_CUDA(cudaStreamSynchronize(ctx_->stream));
    if (stats) {
      float ms = 0;
      GE_CUDA(cudaEventElapsedTime(&ms, ev0, ev1));
      stats->device_ms = ms;
      stats->total_ms = now_ms() - t_begin;
      stats->rounds = rounds;
      stats->kernel_launches = ctx_->launches - launches0;
    }
  }

 private:
  ge_context* ctx_;
  DevBuf<unsigned char> temp_;
  DevBuf<int> iota_;  // 0, 1, ..., n0-1
};

}  // namespace

void upload_graph(ge_context* ctx, const ge_csr& A, DevGraph& G) {
  GE_REQUIRE(A.rows == A.cols, "A must be square");
  const int n = A.rows;
  const int nnz = A.indptr[n];
  G.n = n;
  G.nnz = nnz;
  G.I.alloc(ctx, (size_t)n + 1);
  G.J.alloc(ctx, std::max(nnz, 1));
  G.I.upload(ctx, A.indptr, (size_t)n + 1);
  G.J.upload(ctx, A.indices, nnz);
  if (A.data != nullptr) {
    G.W.alloc(ctx, std::max(nnz, 1));
    G.W.upload(ctx, A.data, nnz);
  }
}

void check_graph(ge_context* ctx, const DevGraph& G) {
  DevBuf<int> bad(ctx, 1);
  bad.zero(ctx->stream);
  k_check_graph<<<grid_of(G.n, 256), 256, 0, ctx->stream>>>(G.I.get(), G.J.get(), G.n, bad.get());
  GE_CUDA(cudaGetLastError());
  ctx->launches++;
  int bad_h = 0;
  GE_CUDA(cudaMemcpyAsync(&bad_h, bad.get(), sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  GE_CUDA(cudaStreamSynchronize(ctx->stream));
  GE_REQUIRE(!bad_h, "A.indptr is not ascending or A.indices has an entry outside [0, rows)");
}

void check_coarsen_options(const ge_coarsen_options& opt) {
  GE_REQUIRE(opt.coarsening_factor > 0.0 && opt.coarsening_factor <= 1.0,
             "coarsening_factor must lie in (0, 1]");
  GE_REQUIRE(opt.min_coarse >= 1, "min_coarse must be >= 1");
  GE_REQUIRE(opt.max_levels >= 0, "max_levels must be >= 0");
}

void coarsen_device(ge_context* ctx, DeviceHierarchy& h, const ge_coarsen_options& opt, bool check,
                    int64_t* rounds) {
  check_coarsen_options(opt);
  Coarsener c(ctx);
  c.build(h, opt, check, rounds);
}

void coarsen(ge_context* ctx, const ge_csr& A, const ge_coarsen_options& opt, HostHierarchy& out,
             ge_coarsen_stats* stats) {
  GE_REQUIRE(A.rows == A.cols, "A must be square");
  check_coarsen_options(opt);
  Coarsener c(ctx);
  c.run(A, opt, out, stats);
}

}  // namespace ge

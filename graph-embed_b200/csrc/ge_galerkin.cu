// graph-embed_b200 :: Galerkin coarse graph  A_c = P_T * A * P_T^T  on the device (sm_100a).
//
// Replaces the step every caller of partition::embed runs before it,
// /root/reference/examples/embedder.cpp:213-216 and examples/embed.cpp:95-98
//     As.push_back(P.Mult(As.back()).Mult(P.Transpose()))
// for an aggregation matrix P_T (m x n, 0/1, one entry per column; row a lists the members of
// aggregate a).  With such a P_T the product is a relabel-and-merge:
//     A_c[a][b] = sum of A[i][j] over i in a, j in b            (diagonal entries included, quirk Q5)
// HBM-bound integer/byte work -- no GEMM, no tensor cores.
//
// One CTA per coarse row a ("segment" = the E_a entries of its members' rows, members in P_T
// order, entries in CSR order):
//   expand   key = (v_A[j] << 32 | position in the segment), value = A[i][j]
//   sort     bitonic on the 64-bit keys (shared memory up to 4096 entries, global scratch above)
//            -> entries ordered by coarse column, ties in member / entry order
//   reduce   every run of equal coarse columns is summed sequentially in that order (one thread
//            per run): deterministic, and exactly the order of a row-by-row Gustavson
//            accumulation; run heads are ranked with a block scan and written to the segment's
//            slot of a staging buffer, the number of runs is the row length of A_c
// then the row lengths are scanned on the device and k_gal_compact moves the staged rows to their
// final offsets.  Segments of up to 128 entries -- the bulk of every hierarchy -- take one warp
// each (k_gal_warp), larger ones a CTA (k_gal_segment); segments beyond 4096 entries (hub aggregates) are sorted
// together by a grid-wide segmented bitonic network over global scratch.  Columns come out
// ascending within each row.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <thread>
#include <vector>

#include "ge_context.h"

namespace ge {

namespace {

constexpr int kGalSmemMax = 4096;  // largest segment (padded to a power of two) sorted in shared memory
constexpr unsigned long long kPadKey = ~0ull;

struct GalArgs {
  const int* I;        // A.indptr  [n+1]
  const int* J;        // A.indices [nnz]
  const double* W;     // A.data    [nnz] or nullptr (unit weights)
  const int* vA;       // vertex -> aggregate [n]
  const int* Pptr;     // P_T.indptr [m+1]
  const int* Pidx;     // P_T.indices [n]
  const int* rowoff;   // offset of fine row i inside its segment [n]
  const int* segoff;   // first staging slot of segment a [m+1]
  const int* list;     // segments handled by this launch
  int* count;          // out: row length of A_c [m]
  int* tmpcol;         // staging [nnz]
  double* tmpval;      // staging [nnz]
  unsigned long long* gkeys;  // big segments: keys scratch (padded sizes, see bigoff)
  double* gvals;              // big segments: values scratch
  const long long* bigoff;    // big segments: offset of segment list[b] in gkeys / gvals
};

__device__ __forceinline__ int block_exclusive_scan(int v, int* scratch, int& total) {
  // blockDim.x <= 1024, multiple of 32
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int x = v;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, x, off);
    if (lane >= off) x += y;
  }
  if (lane == 31) scratch[w] = x;
  __syncthreads();
  if (w == 0) {
    int s = lane < nw ? scratch[lane] : 0;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, s, off);
      if (lane >= off) s += y;
    }
    scratch[32 + lane] = s;  // inclusive warp totals
  }
  __syncthreads();
  const int base = w > 0 ? scratch[32 + w - 1] : 0;
  total = scratch[32 + nw - 1];
  __syncthreads();
  return base + x - v;
}

// Normalised bitonic network (every compare-exchange ascending; the first step of a merge pairs
// i with i ^ (2k-1)), so padding keys at the end stay at the end.  N = power of two.
__device__ __forceinline__ void bitonic_sort(unsigned long long* keys, int N) {
  for (int k = 2; k <= N; k <<= 1) {
    for (int t = threadIdx.x; t < N / 2; t += blockDim.x) {
      const int hk = k >> 1;
      const int lo = (t / hk) * k + (t % hk);
      const int hi = lo ^ (k - 1);
      const unsigned long long a = keys[lo], b = keys[hi];
      if (a > b) {
        keys[lo] = b;
        keys[hi] = a;
      }
    }
    __syncthreads();
    for (int j = k >> 2; j > 0; j >>= 1) {
      for (int t = threadIdx.x; t < N / 2; t += blockDim.x) {
        const int lo = (t / j) * 2 * j + (t % j);
        const int hi = lo + j;
        const unsigned long long a = keys[lo], b = keys[hi];
        if (a > b) {
          keys[lo] = b;
          keys[hi] = a;
        }
      }
      __syncthreads();
    }
  }
}

// N: padded segment size of this launch's class (small: shared memory, N <= kGalSmemMax;
// big: N is read per segment and the arrays live in global scratch).
// phase bits (BIG only; the shared-memory classes always run all three): 1 expand, 2 sort, 4 reduce.
// Big segments are expanded by their CTA, sorted by the grid-wide network below, then reduced.
template <bool BIG>
__global__ void __launch_bounds__(512) k_gal_segment(const GalArgs g, int Nclass, int phase) {
  extern __shared__ __align__(16) unsigned char gal_smem[];
  __shared__ int scan_scratch[64];
  const int a = g.list[blockIdx.x];
  const int p0 = g.Pptr[a], p1 = g.Pptr[a + 1];
  const int s0 = g.segoff[a];
  const int E = g.segoff[a + 1] - s0;
  int N = Nclass;
  unsigned long long* keys;
  double* vals;
  if (BIG) {
    N = 2 * kGalSmemMax;
    while (N < E) N <<= 1;
    keys = g.gkeys + g.bigoff[blockIdx.x];
    vals = g.gvals + g.bigoff[blockIdx.x];
  } else {
    keys = reinterpret_cast<unsigned long long*>(gal_smem);
    vals = reinterpret_cast<double*>(gal_smem + (size_t)N * sizeof(unsigned long long));
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;

  if (phase & 1) {  // expand: members in P_T order, entries in CSR order
    for (int mi = p0 + w; mi < p1; mi += nw) {
      const int i = g.Pidx[mi];
      const int e0 = g.I[i], len = g.I[i + 1] - e0;
      const int base = g.rowoff[i];
      for (int t = lane; t < len; t += 32) {
        const int e = e0 + t;
        keys[base + t] = ((unsigned long long)(unsigned)g.vA[g.J[e]] << 32) | (unsigned)(base + t);
        vals[base + t] = g.W ? g.W[e] : 1.0;
      }
    }
    for (int t = E + threadIdx.x; t < N; t += blockDim.x) keys[t] = kPadKey;
    __syncthreads();
  }
  if (phase & 2) bitonic_sort(keys, N);
  if (!(phase & 4)) return;

  // runs of equal coarse column: rank the heads, sum each run in order.  A head thread sums runs
  // of up to kShortRun entries itself; longer runs (a hub aggregate's own column can collect 10^5
  // entries) are queued and summed by a whole warp: the lanes fetch 32 values at a time, then
  // every lane adds them in run order through shuffles -- the same sequence of additions, with
  // the memory latency taken out of the chain.
  constexpr int kShortRun = 32;
  __shared__ int q_idx[512], q_rank[512];
  __shared__ int q_n;
  int carry = 0;
  for (int c0 = 0; c0 < E; c0 += blockDim.x) {
    if (threadIdx.x == 0) q_n = 0;
    const int idx = c0 + threadIdx.x;
    const bool in = idx < E;
    const unsigned col = in ? (unsigned)(keys[idx] >> 32) : 0u;
    const bool head = in && (idx == 0 || (unsigned)(keys[idx - 1] >> 32) != col);
    int total;
    const int rank = carry + block_exclusive_scan(head ? 1 : 0, scan_scratch, total);  // (barriers)
    if (head) {
      double sum = 0.0;
      int r = idx;
      for (; r < E && r < idx + kShortRun && (unsigned)(keys[r] >> 32) == col; ++r)
        sum += vals[(unsigned)(keys[r] & 0xffffffffu)];
      g.tmpcol[s0 + rank] = (int)col;
      if (r < E && r == idx + kShortRun && (unsigned)(keys[r] >> 32) == col) {
        const int slot = atomicAdd(&q_n, 1);
        q_idx[slot] = idx;
        q_rank[slot] = rank;
      } else {
        g.tmpval[s0 + rank] = sum;
      }
    }
    __syncthreads();
    for (int q = w; q < q_n; q += nw) {  // one warp per long run
      const int r0 = q_idx[q];
      const unsigned qcol = (unsigned)(keys[r0] >> 32);
      double sum = 0.0;
      for (int c = r0;; c += 32) {
        const int r = c + lane;
        const bool ok = r < E && (unsigned)(keys[r] >> 32) == qcol;
        const double v = ok ? vals[(unsigned)(keys[r] & 0xffffffffu)] : 0.0;
        const unsigned okmask = __ballot_sync(0xffffffffu, ok);
        const int cnt = __popc(okmask);  // the run is contiguous: ok lanes are 0 .. cnt-1
        for (int l = 0; l < cnt; ++l) sum += __shfl_sync(0xffffffffu, v, l);
        if (cnt < 32) break;
      }
      if (lane == 0) g.tmpval[s0 + q_rank[q]] = sum;
    }
    __syncthreads();
    carry += total;
  }
  if (threadIdx.x == 0) g.count[a] = carry;
}

// ---- grid-wide segmented bitonic sort for the big segments ------------------------------------
// Every big segment is padded to a power of two >= 8192, so it consists of whole 1024-key tiles;
// tileseg[tile] names its segment, segN / segtile0 / segbase the segment's padded size, first tile
// and first key.  Distances below 1024 are handled inside a tile in shared memory, larger ones by
// one launch per step over all segments at once (segments shorter than the current merge size
// sit the step out).
constexpr int kTileKeys = 1024;
struct BigSort {
  unsigned long long* keys;
  const int* tileseg;
  const int* segN;
  const int* segtile0;
  const long long* segbase;
};
__device__ __forceinline__ void cmpx(unsigned long long* k, long long lo, long long hi) {
  const unsigned long long a = k[lo], b = k[hi];
  if (a > b) {
    k[lo] = b;
    k[hi] = a;
  }
}
// full sort of every 1024-key tile (merge sizes 2 .. 1024)
__global__ void __launch_bounds__(512) k_bitonic_tile_sort(const BigSort b) {
  __shared__ unsigned long long t[kTileKeys];
  unsigned long long* src = b.keys + (long long)blockIdx.x * kTileKeys;
  for (int i = threadIdx.x; i < kTileKeys; i += 512) t[i] = src[i];
  __syncthreads();
  bitonic_sort(t, kTileKeys);
  for (int i = threadIdx.x; i < kTileKeys; i += 512) src[i] = t[i];
}
// one global step of merge size k: flip (j == 0) or half-cleaner at distance j >= 1024
__global__ void __launch_bounds__(256) k_bitonic_global(const BigSort b, int k, int j) {
  const long long gp = (long long)blockIdx.x * 256 + threadIdx.x;  // pair index over all tiles
  const int tile = (int)(gp / (kTileKeys / 2));
  const int seg = b.tileseg[tile];
  if (k > b.segN[seg]) return;
  const long long q = (long long)(tile - b.segtile0[seg]) * (kTileKeys / 2) + gp % (kTileKeys / 2);
  unsigned long long* keys = b.keys + b.segbase[seg];
  if (j == 0) {
    const long long hk = k >> 1;
    const long long lo = (q / hk) * k + (q % hk);
    cmpx(keys, lo, lo ^ (long long)(k - 1));
  } else {
    const long long lo = (q / j) * 2 * j + (q % j);
    cmpx(keys, lo, lo + j);
  }
}
// the half-cleaners at distances 512 .. 1 of merge size k, inside each tile
__global__ void __launch_bounds__(512) k_bitonic_tile_merge(const BigSort b, int k) {
  __shared__ unsigned long long t[kTileKeys];
  const int seg = b.tileseg[blockIdx.x];
  if (k > b.segN[seg]) return;
  unsigned long long* src = b.keys + (long long)blockIdx.x * kTileKeys;
  for (int i = threadIdx.x; i < kTileKeys; i += 512) t[i] = src[i];
  __syncthreads();
  for (int j = kTileKeys / 2; j > 0; j >>= 1) {
    const int lo = (threadIdx.x / j) * 2 * j + (threadIdx.x % j);
    const unsigned long long a = t[lo], c = t[lo + j];
    if (a > c) {
      t[lo] = c;
      t[lo + j] = a;
    }
    __syncthreads();
  }
  for (int i = threadIdx.x; i < kTileKeys; i += 512) src[i] = t[i];
}

// Segments of up to 128 entries (the bulk of every hierarchy: a handful of members with ~10
// entries each): one WARP per segment, eight segments per CTA, warp-synchronous throughout, and no
// sort.  The first version sorted (coarse column, position) keys with a bitonic network in shared
// memory and was issue-bound at ~2000 warp instructions per 40-entry segment (ncu,
// profiles/r02_gal_warp.txt).  A segment has only a handful of distinct coarse columns, so: the
// entries are staged by position (lane l keeps positions l, l + 32, ...), then the warp repeatedly
// takes the smallest column still present (__reduce_min_sync) and hands it to the next lane; every
// lane then adds the entries of its column in position order -- the member-then-CSR order of the
// oracle, bit for bit.  Columns come out ascending.  K = padded size / 32 (1, 2 or 4).
template <int K>
__global__ void __launch_bounds__(256) k_gal_warp(const GalArgs g, int nseg) {
  constexpr int N = 32 * K;
  constexpr unsigned kFull = 0xffffffffu, kNone = 0xffffffffu;
  __shared__ unsigned scol[8][N];
  __shared__ double sval[8][N];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int sid = blockIdx.x * 8 + w;
  if (sid >= nseg) return;
  const int a = g.list[sid];
  const int p0 = g.Pptr[a], p1 = g.Pptr[a + 1];
  const int s0 = g.segoff[a];
  const int E = g.segoff[a + 1] - s0;

  // expand: 32 members at a time fetch their row descriptors together, then the rows are copied
  // one after the other with the descriptor broadcast by shuffle
  for (int m0 = p0; m0 < p1; m0 += 32) {
    const int cnt = min(32, p1 - m0);
    int i = 0, e0 = 0, len = 0, base = 0;
    if (lane < cnt) {
      i = g.Pidx[m0 + lane];
      e0 = g.I[i];
      len = g.I[i + 1] - e0;
      base = g.rowoff[i];
    }
    for (int q = 0; q < cnt; ++q) {
      const int qe0 = __shfl_sync(kFull, e0, q), qlen = __shfl_sync(kFull, len, q);
      const int qbase = __shfl_sync(kFull, base, q);
      for (int t = lane; t < qlen; t += 32) {
        const int e = qe0 + t;
        scol[w][qbase + t] = (unsigned)g.vA[g.J[e]];
        sval[w][qbase + t] = g.W ? g.W[e] : 1.0;
      }
    }
  }
  __syncwarp();
  unsigned col[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const int pidx = k * 32 + lane;
    col[k] = pidx < E ? scol[w][pidx] : kNone;
  }
  // Up to 32 distinct columns at a time, ascending: lane j keeps the j-th smallest still present.
  // Then every lane adds the entries of ITS column in position order (all lanes read the same
  // staged entry: shared-memory broadcasts), so a segment costs ~4 instructions per entry instead
  // of a sort.
  int nout = 0;
  for (;;) {
    unsigned my_col = kNone;
    int found = 0;
    for (; found < 32; ++found) {
      unsigned mine = col[0];
#pragma unroll
      for (int k = 1; k < K; ++k) mine = min(mine, col[k]);
      const unsigned cmin = __reduce_min_sync(kFull, mine);
      if (cmin == kNone) break;
      if (lane == found) my_col = cmin;
#pragma unroll
      for (int k = 0; k < K; ++k)
        if (col[k] == cmin) col[k] = kNone;
    }
    if (found == 0) break;
    double sum = 0.0;
#pragma unroll 4
    for (int pidx = 0; pidx < E; ++pidx) {
      const unsigned c = scol[w][pidx];
      const double v = sval[w][pidx];
      if (c == my_col) sum += v;  // member order, then CSR order: the oracle's sequence of additions
    }
    if (lane < found) {
      g.tmpcol[s0 + nout + lane] = (int)my_col;
      g.tmpval[s0 + nout + lane] = sum;
    }
    nout += found;
    if (found < 32) break;
  }
  if (lane == 0) g.count[a] = nout;
}

// Exclusive scan of the row lengths on the device (three small kernels; m is at most a few million).
constexpr int kScanBlock = 1024;
__global__ void __launch_bounds__(kScanBlock) k_scan_blocks(const int* __restrict__ in, int n,
                                                           int* __restrict__ out, int* __restrict__ sums) {
  __shared__ int scratch[64];
  const int i = blockIdx.x * kScanBlock + threadIdx.x;
  const int v = i < n ? in[i] : 0;
  int total;
  const int ex = block_exclusive_scan(v, scratch, total);
  if (i < n) out[i] = ex;
  if (threadIdx.x == 0) sums[blockIdx.x] = total;
}
__global__ void __launch_bounds__(kScanBlock) k_scan_sums(int* sums, int nb) {  // one CTA
  __shared__ int scratch[64];
  int carry = 0;
  for (int c0 = 0; c0 < nb; c0 += kScanBlock) {
    const int i = c0 + threadIdx.x;
    const int v = i < nb ? sums[i] : 0;
    int total;
    const int ex = block_exclusive_scan(v, scratch, total);
    if (i < nb) sums[i] = carry + ex;
    carry += total;
  }
  if (threadIdx.x == 0) sums[nb] = carry;  // grand total
}
__global__ void __launch_bounds__(kScanBlock) k_scan_add(int* __restrict__ out, int n,
                                                        const int* __restrict__ sums, int nb) {
  const int i = blockIdx.x * kScanBlock + threadIdx.x;
  if (i < n) out[i] += sums[blockIdx.x];
  if (i == 0) out[n] = sums[nb];
}

// One warp per coarse row: staged row -> final offsets.
__global__ void __launch_bounds__(256) k_gal_compact(const int* __restrict__ segoff,
                                                     const int* __restrict__ outptr, int m,
                                                     const int* __restrict__ tmpcol,
                                                     const double* __restrict__ tmpval,
                                                     int* __restrict__ outcol, double* __restrict__ outval) {
  const int a = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (a >= m) return;
  const int lane = threadIdx.x & 31;
  const int s0 = segoff[a], o0 = outptr[a], len = outptr[a + 1] - o0;
  for (int t = lane; t < len; t += 32) {
    outcol[o0 + t] = tmpcol[s0 + t];
    outval[o0 + t] = tmpval[s0 + t];
  }
}

}  // namespace

void exclusive_scan(ge_context* ctx, const int* d_in, int n, int* d_out) {
  const int nb = (n + kScanBlock - 1) / kScanBlock;
  DevBuf<int> d_sums(ctx, nb + 1);
  if (n == 0) {
    GE_CUDA(cudaMemsetAsync(d_out, 0, sizeof(int), ctx->stream));
    return;
  }
  k_scan_blocks<<<nb, kScanBlock, 0, ctx->stream>>>(d_in, n, d_out, d_sums.get());
  k_scan_sums<<<1, kScanBlock, 0, ctx->stream>>>(d_sums.get(), nb);
  k_scan_add<<<nb, kScanBlock, 0, ctx->stream>>>(d_out, n, d_sums.get(), nb);
  GE_CUDA(cudaGetLastError());
  ctx->launches += 3;
}

int64_t galerkin_device(ge_context* ctx, const GalerkinInput& in, const int* segoff_host,
                        int32_t* c_indptr, DevBuf<int>& outptr, DevBuf<int>& outcol,
                        DevBuf<double>& outval, int64_t capacity, ge_galerkin_stats* stats,
                        cudaEvent_t start) {
  const int m = in.m;
  const int nnz = segoff_host[m];
  // size classes: padded power-of-two size 32 .. 4096 in shared memory, larger in global scratch
  constexpr int kClasses = 8;  // 32, 64, ..., 4096
  std::vector<int> lists[kClasses], big;
  std::vector<long long> bigoff;
  std::vector<int> bigN;
  long long big_elems = 0;
  for (int a = 0; a < m; ++a) {
    const int E = segoff_host[a + 1] - segoff_host[a];
    if (E == 0) continue;  // count stays 0
    int N = 32, k = 0;
    while (N < E && N < kGalSmemMax) {
      N <<= 1;
      ++k;
    }
    if (E <= kGalSmemMax) {
      lists[k].push_back(a);
    } else {
      long long Np = 2 * kGalSmemMax;  // whole 1024-key tiles for the grid-wide sort
      while (Np < E) Np <<= 1;
      big.push_back(a);
      bigoff.push_back(big_elems);
      bigN.push_back((int)Np);
      big_elems += Np;
    }
  }
  std::vector<int> all_list;
  int class_begin[kClasses + 1];
  for (int k = 0; k < kClasses; ++k) {
    class_begin[k] = (int)all_list.size();
    all_list.insert(all_list.end(), lists[k].begin(), lists[k].end());
  }
  class_begin[kClasses] = (int)all_list.size();
  const int big_begin = (int)all_list.size();
  all_list.insert(all_list.end(), big.begin(), big.end());

  DevBuf<int> d_list(ctx, std::max<size_t>(all_list.size(), 1)), d_count(ctx, std::max(m, 1)),
      d_tmpcol(ctx, std::max(nnz, 1));
  DevBuf<double> d_tmpval(ctx, std::max(nnz, 1)), d_gvals(ctx, (size_t)std::max<long long>(big_elems, 1));
  DevBuf<unsigned long long> d_gkeys(ctx, (size_t)std::max<long long>(big_elems, 1));
  DevBuf<long long> d_bigoff(ctx, std::max<size_t>(bigoff.size(), 1));
  d_list.upload(ctx, all_list.data(), all_list.size());
  if (!bigoff.empty()) d_bigoff.upload(ctx, bigoff.data(), bigoff.size());
  d_count.zero(ctx->stream);

  const bool verbose = std::getenv("GE_VERBOSE") != nullptr;
  double t_mark = now_ms();
  auto lap = [&](const char* what) {
    if (!verbose) return;
    GE_CUDA(cudaStreamSynchronize(ctx->stream));
    const double t = now_ms();
    std::fprintf(stderr, "[ge] galerkin n=%d %-22s %9.3f ms\n", in.n, what, t - t_mark);
    t_mark = t;
  };
  lap("layout + upload");
  if (start) GE_CUDA(cudaEventRecord(start, ctx->stream));
  GalArgs g;
  g.I = in.I;
  g.J = in.J;
  g.W = in.W;
  g.vA = in.vA;
  g.Pptr = in.Pptr;
  g.Pidx = in.Pidx;
  g.rowoff = in.rowoff;
  g.segoff = in.segoff;
  g.count = d_count.get();
  g.tmpcol = d_tmpcol.get();
  g.tmpval = d_tmpval.get();
  g.gkeys = d_gkeys.get();
  g.gvals = d_gvals.get();
  g.bigoff = d_bigoff.get();
  // (function attributes are per device: set on every call, it costs microseconds)
  GE_CUDA(cudaFuncSetAttribute(k_gal_segment<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               kGalSmemMax * 16));
  for (int k = 0; k < kClasses; ++k) {
    const int cnt = class_begin[k + 1] - class_begin[k];
    if (cnt == 0) continue;
    const int N = 32 << k;
    const int threads = std::max(32, std::min(512, N / 2));
    g.list = d_list.get() + class_begin[k];
    if (N == 32)
      k_gal_warp<1><<<(cnt + 7) / 8, 256, 0, ctx->stream>>>(g, cnt);
    else if (N == 64)
      k_gal_warp<2><<<(cnt + 7) / 8, 256, 0, ctx->stream>>>(g, cnt);
    else if (N == 128)
      k_gal_warp<4><<<(cnt + 7) / 8, 256, 0, ctx->stream>>>(g, cnt);
    else
      k_gal_segment<false><<<cnt, threads, (size_t)N * 16, ctx->stream>>>(g, N, 7);
    GE_CUDA(cudaGetLastError());
    ctx->launches++;
  }
  lap("shared-memory segments");
  DevBuf<int> d_tileseg, d_segN, d_segtile0;
  if (!big.empty()) {
    g.list = d_list.get() + big_begin;
    const int ntiles = (int)(big_elems / kTileKeys);
    std::vector<int> tileseg((size_t)ntiles), segtile0(big.size());
    int maxN = 0;
    for (size_t b = 0; b < big.size(); ++b) {
      segtile0[b] = (int)(bigoff[b] / kTileKeys);
      for (int t = 0; t < bigN[b] / kTileKeys; ++t) tileseg[(size_t)segtile0[b] + t] = (int)b;
      maxN = std::max(maxN, bigN[b]);
    }
    d_tileseg.alloc(ctx, tileseg.size());
    d_segN.alloc(ctx, big.size());
    d_segtile0.alloc(ctx, big.size());
    d_tileseg.upload(ctx, tileseg.data(), tileseg.size());
    d_segN.upload(ctx, bigN.data(), big.size());
    d_segtile0.upload(ctx, segtile0.data(), big.size());
    BigSort bs;
    bs.keys = d_gkeys.get();
    bs.tileseg = d_tileseg.get();
    bs.segN = d_segN.get();
    bs.segtile0 = d_segtile0.get();
    bs.segbase = d_bigoff.get();
    lap("big: tables");
    k_gal_segment<true><<<(unsigned)big.size(), 512, 0, ctx->stream>>>(g, 0, 1);  // expand + pad
    lap("big: expand");
    k_bitonic_tile_sort<<<ntiles, 512, 0, ctx->stream>>>(bs);
    ctx->launches += 2;
    const unsigned pair_grid = (unsigned)((long long)ntiles * (kTileKeys / 2) / 256);
    for (int k = 2 * kTileKeys; k <= maxN; k <<= 1) {
      k_bitonic_global<<<pair_grid, 256, 0, ctx->stream>>>(bs, k, 0);
      ctx->launches++;
      for (int j = k >> 2; j >= kTileKeys; j >>= 1) {
        k_bitonic_global<<<pair_grid, 256, 0, ctx->stream>>>(bs, k, j);
        ctx->launches++;
      }
      k_bitonic_tile_merge<<<ntiles, 512, 0, ctx->stream>>>(bs, k);
      ctx->launches++;
    }
    lap("big: sort");
    k_gal_segment<true><<<(unsigned)big.size(), 512, 0, ctx->stream>>>(g, 0, 4);  // reduce the runs
    GE_CUDA(cudaGetLastError());
    ctx->launches++;
    lap("big: reduce");
  }
  // row lengths -> exclusive scan on the device -> final offsets (nnz(A_c) <= nnz(A) < 2^31)
  outptr.alloc(ctx, (size_t)m + 1);
  int total32 = 0;
  if (m > 0) {
    exclusive_scan(ctx, d_count.get(), m, outptr.get());
    if (c_indptr) {
      outptr.download(ctx, c_indptr, (size_t)m + 1);
      GE_CUDA(cudaStreamSynchronize(ctx->stream));
      total32 = c_indptr[m];
    } else {
      GE_CUDA(cudaMemcpyAsync(&total32, outptr.get() + m, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
      GE_CUDA(cudaStreamSynchronize(ctx->stream));
    }
  } else {
    outptr.zero(ctx->stream);
    if (c_indptr) c_indptr[0] = 0;
  }
  lap("scan + row pointers");
  const int64_t total = total32;
  if (total <= capacity && total > 0) {
    outcol.alloc(ctx, (size_t)total);
    outval.alloc(ctx, (size_t)total);
    const unsigned grid = (unsigned)(((int64_t)m * 32 + 255) / 256);
    k_gal_compact<<<grid, 256, 0, ctx->stream>>>(in.segoff, outptr.get(), m, d_tmpcol.get(),
                                                 d_tmpval.get(), outcol.get(), outval.get());
    GE_CUDA(cudaGetLastError());
    ctx->launches++;
  }
  if (stats) {
    stats->segments_shared = big_begin;
    stats->segments_global = (int64_t)big.size();
    stats->nnz_out = total;
  }
  return total;
}

// Returns nnz(A_c); fills c_indptr always, c_indices / c_data when capacity suffices.
int64_t galerkin(ge_context* ctx, const ge_csr& A, const ge_csr& P, int32_t* c_indptr,
                 int32_t* c_indices, double* c_data, int64_t capacity, ge_galerkin_stats* stats) {
  const int n = A.rows, m = P.rows;
  GE_REQUIRE(A.rows == A.cols, "A must be square");
  GE_REQUIRE(P.cols == n, "P_T.cols != A.rows");
  GE_REQUIRE(P.indptr[m] == n, "P_T must have exactly one entry per column");
  const int nnz = A.indptr[n];
  const double t_begin = now_ms();

  // The fine graph does not depend on the layout: a helper thread uploads it (through the pinned
  // staging ring when the caller's arrays are pageable) while this thread computes the layout.
  const int64_t launches0 = ctx->launches;
  DevBuf<int> d_I(ctx, n + 1), d_J(ctx, std::max(nnz, 1));
  DevBuf<double> d_W;
  if (A.data != nullptr) d_W.alloc(ctx, std::max(nnz, 1));
  ge_status up_status = GE_OK;
  std::string up_error;
  std::thread uploader([&] {
    try {
      GE_CUDA(cudaSetDevice(ctx->device));
      d_I.upload(ctx, A.indptr, n + 1);
      d_J.upload(ctx, A.indices, nnz);
      if (A.data != nullptr) d_W.upload(ctx, A.data, nnz);
    } catch (const Fail& f) {
      up_status = f.st;
      up_error = ge_last_error();
    }
  });
  struct Joiner {
    std::thread& t;
    ~Joiner() {
      if (t.joinable()) t.join();
    }
  } joiner{uploader};

  // host: vertex -> aggregate, segment offsets, row offsets inside the segments (O(n)); the
  // aggregates are independent, so a few threads share them out and a prefix sum follows
  std::vector<int> vA(std::max(n, 1), -1), rowoff(std::max(n, 1), 0), segoff((size_t)m + 1, 0);
  {
    const int nt = m > (1 << 16) ? 8 : 1;
    std::vector<int> bad(nt, 0);
    auto part = [&](int t) {
      const int a0 = (int)((int64_t)m * t / nt), a1 = (int)((int64_t)m * (t + 1) / nt);
      for (int a = a0; a < a1; ++a) {
        int run = 0;
        for (int c = P.indptr[a]; c < P.indptr[a + 1]; ++c) {
          const int i = P.indices[c];
          if (i < 0 || i >= n) {
            bad[t] = 1;
            continue;
          }
          vA[i] = a;
          rowoff[i] = run;
          run += A.indptr[i + 1] - A.indptr[i];
        }
        segoff[a + 1] = run;  // length for now; prefix-summed below
      }
    };
    if (nt == 1) {
      part(0);
    } else {
      std::vector<std::thread> pool;
      for (int t = 0; t < nt; ++t) pool.emplace_back(part, t);
      for (auto& th : pool) th.join();
    }
    bool ok = true;
    for (int t = 0; t < nt; ++t) ok = ok && !bad[t];
    // n entries in P_T, every one in range: all n vertices covered <=> none listed twice
    for (int i = 0; ok && i < n; ++i) ok = vA[i] >= 0;
    GE_REQUIRE(ok, "P_T is not a partition of the vertices");
    for (int a = 0; a < m; ++a) segoff[a + 1] += segoff[a];
  }

  uploader.join();  // (this thread issues CUDA calls from here on)
  if (up_status != GE_OK) {
    set_error("graph upload: " + up_error);
    throw Fail{up_status};
  }
  DevBuf<int> d_vA(ctx, std::max(n, 1)), d_Pptr(ctx, m + 1), d_Pidx(ctx, std::max(n, 1)),
      d_rowoff(ctx, std::max(n, 1)), d_segoff(ctx, m + 1);
  d_vA.upload(ctx, vA.data(), n);
  d_Pptr.upload(ctx, P.indptr, m + 1);
  d_Pidx.upload(ctx, P.indices, n);
  d_rowoff.upload(ctx, rowoff.data(), n);
  d_segoff.upload(ctx, segoff.data(), m + 1);

  cudaEvent_t ev0, ev1;
  GE_CUDA(cudaEventCreate(&ev0));
  GE_CUDA(cudaEventCreate(&ev1));
  GalerkinInput in;
  in.n = n;
  in.m = m;
  in.I = d_I.get();
  in.J = d_J.get();
  in.W = A.data != nullptr ? d_W.get() : nullptr;
  in.vA = d_vA.get();
  in.Pptr = d_Pptr.get();
  in.Pidx = d_Pidx.get();
  in.rowoff = d_rowoff.get();
  in.segoff = d_segoff.get();
  DevBuf<int> d_outptr, d_outcol;
  DevBuf<double> d_outval;
  const int64_t total = galerkin_device(ctx, in, segoff.data(), c_indptr, d_outptr, d_outcol, d_outval,
                                        capacity, stats, ev0);
  GE_CUDA(cudaEventRecord(ev1, ctx->stream));
  if (total <= capacity && total > 0) {
    GE_REQUIRE(c_indices && c_data, "null output arrays");
    d_outcol.download(ctx, c_indices, (size_t)total);
    d_outval.download(ctx, c_data, (size_t)total);
  }
  GE_CUDA(cudaStreamSynchronize(ctx->stream));
  if (stats) {
    float ms = 0;
    GE_CUDA(cudaEventElapsedTime(&ms, ev0, ev1));
    stats->device_ms = ms;  // kernels + the row-length round trip
    stats->total_ms = now_ms() - t_begin;
    stats->kernel_launches = ctx->launches - launches0;
  }
  cudaEventDestroy(ev0);
  cudaEventDestroy(ev1);
  return total;
}

}  // namespace ge

// graph-embed_b200 :: largest connected component on the device (sm_100a).
//
// examples/embedder.cpp:156 (largestComponent, :35-93) keeps the largest connected component of the
// input before it partitions.  Here:
//   components  weak components (every CSR entry (i, j) links i and j) by a lock-free union-find in
//               the style of ECL-CC: a root is only ever hooked under a smaller root (atomicCAS on
//               its parent), find halves the path it walks, and a last pass points every vertex at
//               its root.  Parents only decrease, so the root of a component is its smallest vertex:
//               the labels are canonical, whatever order the atomics ran in.
//   choice      vertices per label (integer atomics); the largest component, ties to the smaller label
//               (np.argmax(np.bincount(label))); components = vertices that are their own label
//   extraction  kept vertices renumbered in ascending order (scan of the flags), their rows copied
//               with the columns renumbered.  Every neighbour of a kept vertex is kept and the
//               renumbering is monotone: entry order and ascending columns survive, weights are
//               copied bit for bit.
// Rows are hooked in the three tiers of ge_coarsen.cu: a thread per short row, a warp per row and a
// CTA per row longer than kHubRow (raw R-MAT-20 has rows of 64 772 entries).
#include <cub/cub.cuh>

#include <algorithm>

#include "ge_context.h"

namespace ge {

namespace {

constexpr int kThreadRow = 16;    // rows up to this length: one thread
constexpr int kHubRow = 1024;     // rows longer than this: a whole CTA (as in ge_coarsen.cu)
constexpr int kHubThreads = 512;

unsigned grid_of(int64_t n, int threads) { return (unsigned)std::max<int64_t>(1, (n + threads - 1) / threads); }

// The root of v, halving the path on the way (every vertex on it then points two steps up).  Other
// threads hook roots concurrently: the parents are read through a volatile pointer.
__device__ __forceinline__ int find_root(int* parent, int v) {
  volatile int* p = parent;
  int cur = p[v];
  if (cur != v) {
    int prev = v, next;
    while (cur > (next = p[cur])) {
      p[prev] = next;
      prev = cur;
      cur = next;
    }
  }
  return cur;
}

// Joins the components of a and b: the larger root goes under the smaller one.
__device__ __forceinline__ void hook(int* parent, int a, int b) {
  int ra = find_root(parent, a), rb = find_root(parent, b);
  while (ra != rb) {
    const int hi = max(ra, rb), lo = min(ra, rb);
    const int old = atomicCAS(&parent[hi], hi, lo);
    if (old == hi) return;
    // hi was hooked by someone else meanwhile: continue from its new root
    if (hi == ra) {
      ra = find_root(parent, old);
      rb = lo;
    } else {
      rb = find_root(parent, old);
      ra = lo;
    }
  }
}

struct CcArgs {
  int n;
  const int* I;
  const int* J;
  int* parent;
  int* warp_rows;  // rows of kThreadRow < len <= kHubRow
  int* hub_rows;   // rows longer than kHubRow
  int* counts;     // [0]: warp rows, [1]: hub rows, [2]: components
};

__global__ void __launch_bounds__(256) k_cc_init(CcArgs a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  a.parent[i] = i;
  const int len = a.I[i + 1] - a.I[i];
  if (len > kHubRow) a.hub_rows[atomicAdd(&a.counts[1], 1)] = i;
  else if (len > kThreadRow) a.warp_rows[atomicAdd(&a.counts[0], 1)] = i;
}

__global__ void __launch_bounds__(256) k_cc_hook_thread(CcArgs a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  const int e0 = a.I[i], e1 = a.I[i + 1];
  if (e1 - e0 > kThreadRow) return;
  for (int e = e0; e < e1; ++e) {
    const int j = a.J[e];
    if (j != i) hook(a.parent, i, j);
  }
}

__global__ void __launch_bounds__(256) k_cc_hook_warp(CcArgs a) {
  const int lane = threadIdx.x & 31;
  const int nw = a.counts[0];
  const int stride = gridDim.x * (blockDim.x >> 5);
  for (int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); w < nw; w += stride) {
    const int i = a.warp_rows[w];
    const int e0 = a.I[i], e1 = a.I[i + 1];
    for (int e = e0 + lane; e < e1; e += 32) {
      const int j = a.J[e];
      if (j != i) hook(a.parent, i, j);
    }
  }
}

__global__ void __launch_bounds__(kHubThreads) k_cc_hook_hub(CcArgs a) {
  const int nh = a.counts[1];
  for (int b = blockIdx.x; b < nh; b += gridDim.x) {
    const int i = a.hub_rows[b];
    const int e0 = a.I[i], e1 = a.I[i + 1];
    for (int e = e0 + threadIdx.x; e < e1; e += kHubThreads) {
      const int j = a.J[e];
      if (j != i) hook(a.parent, i, j);
    }
  }
}

// label[v] = root of v (in place: the roots never move again), size per label, component count
__global__ void __launch_bounds__(256) k_cc_label(CcArgs a, int* size) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= a.n) return;
  const int r = find_root(a.parent, v);
  a.parent[v] = r;
  atomicAdd(&size[r], 1);
  if (r == v) atomicAdd(&a.counts[2], 1);
}

// the largest component, ties to the smaller label: the largest (size, n - 1 - label)
__global__ void __launch_bounds__(256) k_cc_choose(const int* label, const int* size, int n,
                                                   unsigned long long* best) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n || label[v] != v) return;
  atomicMax(best, ((unsigned long long)(unsigned)size[v] << 32) | (unsigned)(n - 1 - v));
}

__global__ void __launch_bounds__(256) k_cc_flags(const int* label, int n, int keep, int* flag, int* iota) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n) return;
  flag[v] = label[v] == keep;
  iota[v] = v;
}

__global__ void __launch_bounds__(256) k_cc_rowlen(const int* I, const int* vert, int nk, int* len) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < nk) len[k] = I[vert[k] + 1] - I[vert[k]];
}

// row k of the subgraph = row vert[k] of A, columns renumbered (a warp per row)
__global__ void __launch_bounds__(256) k_cc_copy_rows(const int* I, const int* J, const double* W,
                                                      const int* vert, const int* newid, const int* CI,
                                                      int nk, int* CJ, double* CW) {
  const int lane = threadIdx.x & 31;
  const int k = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (k >= nk) return;
  const int e0 = I[vert[k]], len = CI[k + 1] - CI[k], c0 = CI[k];
  for (int t = lane; t < len; t += 32) {
    CJ[c0 + t] = newid[J[e0 + t]];
    CW[c0 + t] = W ? W[e0 + t] : 1.0;
  }
}

__global__ void k_cc_fill(double* x, int64_t n, double v) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] = v;
}

}  // namespace

int64_t largest_component_device(ge_context* ctx, const DevGraph& A, DevGraph& out, DevBuf<int>& vertices) {
  const int n = A.n;
  if (n == 0) return 0;
  cudaStream_t s = ctx->stream;
  DevBuf<int> parent(ctx, n), warp_rows(ctx, n), hub_rows(ctx, n), counts(ctx, 3), size(ctx, n);
  DevBuf<unsigned long long> best(ctx, 1);
  counts.zero(s);
  size.zero(s);
  best.zero(s);
  CcArgs a;
  a.n = n;
  a.I = A.I.get();
  a.J = A.J.get();
  a.parent = parent.get();
  a.warp_rows = warp_rows.get();
  a.hub_rows = hub_rows.get();
  a.counts = counts.get();
  k_cc_init<<<grid_of(n, 256), 256, 0, s>>>(a);
  k_cc_hook_thread<<<grid_of(n, 256), 256, 0, s>>>(a);
  k_cc_hook_warp<<<(unsigned)std::max(1, ctx->sm_count * 8), 256, 0, s>>>(a);
  k_cc_hook_hub<<<(unsigned)std::max(1, ctx->sm_count * 2), kHubThreads, 0, s>>>(a);
  k_cc_label<<<grid_of(n, 256), 256, 0, s>>>(a, size.get());
  k_cc_choose<<<grid_of(n, 256), 256, 0, s>>>(parent.get(), size.get(), n, best.get());
  GE_CUDA(cudaGetLastError());
  ctx->launches += 6;
  int ncomp = 0;
  unsigned long long best_h = 0;
  GE_CUDA(cudaMemcpyAsync(&ncomp, counts.get() + 2, sizeof(int), cudaMemcpyDeviceToHost, s));
  GE_CUDA(cudaMemcpyAsync(&best_h, best.get(), sizeof(best_h), cudaMemcpyDeviceToHost, s));
  GE_CUDA(cudaStreamSynchronize(s));
  if (ncomp == 1) return 1;
  const int keep = n - 1 - (int)(best_h & 0xffffffffu);
  const int nk = (int)(best_h >> 32);
  // kept vertices, ascending, and their new ids
  DevBuf<int> flag(ctx, n), newid(ctx, (size_t)n + 1), iota(ctx, n), nsel(ctx, 1);
  vertices.alloc(ctx, nk);
  k_cc_flags<<<grid_of(n, 256), 256, 0, s>>>(parent.get(), n, keep, flag.get(), iota.get());
  GE_CUDA(cudaGetLastError());
  ctx->launches++;
  exclusive_scan(ctx, flag.get(), n, newid.get());
  {
    size_t bytes = 0;
    GE_CUDA(cub::DeviceSelect::Flagged(nullptr, bytes, iota.get(), flag.get(), vertices.get(), nsel.get(), n, s));
    DevBuf<unsigned char> temp(ctx, std::max<size_t>(bytes, 1));
    GE_CUDA(cub::DeviceSelect::Flagged(temp.get(), bytes, iota.get(), flag.get(), vertices.get(), nsel.get(), n,
                                       s));
    ctx->launches++;
  }
  // the kept rows
  DevBuf<int> len(ctx, std::max(nk, 1));
  out.n = nk;
  out.I.alloc(ctx, (size_t)nk + 1);
  k_cc_rowlen<<<grid_of(nk, 256), 256, 0, s>>>(A.I.get(), vertices.get(), nk, len.get());
  GE_CUDA(cudaGetLastError());
  ctx->launches++;
  exclusive_scan(ctx, len.get(), nk, out.I.get());
  int nnz = 0;
  GE_CUDA(cudaMemcpyAsync(&nnz, out.I.get() + nk, sizeof(int), cudaMemcpyDeviceToHost, s));
  GE_CUDA(cudaStreamSynchronize(s));
  out.nnz = nnz;
  out.J.alloc(ctx, std::max(nnz, 1));
  out.W.alloc(ctx, std::max(nnz, 1));
  k_cc_copy_rows<<<grid_of(nk, 8), 256, 0, s>>>(A.I.get(), A.J.get(), A.w(), vertices.get(), newid.get(),
                                                  out.I.get(), nk, out.J.get(), out.W.get());
  GE_CUDA(cudaGetLastError());
  ctx->launches++;
  return ncomp;
}

void unit_weights(ge_context* ctx, DevGraph& G) {
  if (G.W.size()) return;
  G.W.alloc(ctx, std::max(G.nnz, 1));
  k_cc_fill<<<grid_of(G.nnz, 256), 256, 0, ctx->stream>>>(G.W.get(), G.nnz, 1.0);
  GE_CUDA(cudaGetLastError());
  ctx->launches++;
}

}  // namespace ge

// graph-embed_b200 :: per-aggregate ForceAtlas + prolongation (kernel family K2), sm_100a.
//
// Replaces partition::forceAtlasMultilevel, /root/reference/include/forceatlas.hpp:314-574.
// Aggregates are independent (they read only their own members and the parent level's
// coords_A / r_A), so one level is a batch of small all-pairs problems with no global
// synchronisation.  Work is binned by aggregate size:
//   1 member      k_ml_singletons : closed form (centre - mean = 0  =>  x = coords_A[a]).
//   2..32         k_onchip_warp   : one lane per member, packs of equal-size aggregates per warp.
//   33..512       k_onchip_cta    : one CTA per aggregate, positions in shared memory.
//   larger        k_repulsion / k_attract_step over 256-aligned segments, one launch pair per
//                 iteration, then k_ml_segment_epilogue (R-MAT hierarchies: up to ~3800 members).
// Vertices are renumbered into SLOTS so that each aggregate is contiguous (member order of the
// P_T row preserved, which quirk Q1 at :417 depends on).  k_ml_prep walks every CSR row once and
// emits, per slot: the intra-aggregate degree (:362-383), the compacted intra-aggregate edge list
// (in place, at the row's own CSR offsets) and the constant external-pull numerator
// sum_e 100 * (cA[b]-cA[a]) / max(|cA[b]-cA[a]|, eps)  (:451-466), so that the 100 iterations touch
// only on-chip data plus the compact edge list.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <numeric>
#include <memory>
#include <vector>

#include "ge_flat.cuh"
#include "ge_onchip.cuh"

namespace ge {

namespace {

int env_int(const char* name, int dflt) {
  const char* v = std::getenv(name);
  return v ? std::atoi(v) : dflt;
}

template <typename T>
struct PrepArgs {
  const int* I;
  const int* J;
  const double* Dw;        // nullptr: ones
  const int* v_A;          // vertex -> aggregate
  const int* vtx;          // slot -> vertex (-1: padding)
  const int* slot_of;      // vertex -> slot
  const int* agg_base;     // aggregate -> first slot
  const double* cA;        // [m][D]
  T* mass;                 // [NM][ld]
  T* Eext;                 // [D][ld]
  int* e_begin;
  int* e_end;
  int* e_idx;              // compact neighbour slots, written at the row's CSR offsets
  T* e_w;                  // compact weights (nullptr when unweighted)
  int64_t ld;
  int nslots;
  int use_weights;
  // rows of the large-aggregate tier (slots [0, grid_slots)) with more than long_len internal
  // entries are listed for the CTA-per-row attraction kernel (power-law hierarchies: a hub keeps
  // hundreds of neighbours inside its aggregate)
  int grid_slots;
  int long_len;
  int* long_rows;
  int* long_count;
};

// One warp per slot.
template <typename T, int D>
__global__ void __launch_bounds__(256) k_ml_prep(const PrepArgs<T> a) {
  constexpr int NM = Real<T>::kMassArrays;
  const int slot = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (slot >= a.nslots) return;
  const int v = a.vtx[slot];
  if (v < 0) {  // padding slot inside a 256-aligned segment: massless, edgeless, at the origin
    if (lane == 0) {
      for (int k = 0; k < NM; ++k) a.mass[(int64_t)k * a.ld + slot] = (T)0;
      for (int k = 0; k < D; ++k) a.Eext[(int64_t)k * a.ld + slot] = (T)0;
      a.e_begin[slot] = 0;
      a.e_end[slot] = 0;
    }
    return;
  }
  const int agg = a.v_A[v];
  const int li = slot - a.agg_base[agg];  // local member index i of :391
  const int rb = a.I[v], re = a.I[v + 1];
  double ca[D];
#pragma unroll
  for (int k = 0; k < D; ++k) ca[k] = a.cA[(int64_t)agg * D + k];
  double deg = 0.0, E[D];
#pragma unroll
  for (int k = 0; k < D; ++k) E[k] = 0.0;
  int cnt = 0;
  // four 32-entry trips per pass: their index -> aggregate -> centre load chains are in flight
  // together (a hub row of a power-law level has 1e5 entries and one warp)
  constexpr int kTrips = 4;
  for (int e00 = rb; e00 < re; e00 += 32 * kTrips) {
    int jn[kTrips], bn[kTrips];
    double wn[kTrips];
#pragma unroll
    for (int u = 0; u < kTrips; ++u) {
      const int e = e00 + 32 * u + lane;
      jn[u] = e < re ? a.J[e] : -1;
      wn[u] = (e < re && a.Dw != nullptr) ? a.Dw[e] : 1.0;
    }
#pragma unroll
    for (int u = 0; u < kTrips; ++u) bn[u] = jn[u] >= 0 ? a.v_A[jn[u]] : -1;
#pragma unroll
    for (int u = 0; u < kTrips; ++u) {
    if (e00 + 32 * u >= re) break;  // warp-uniform
    const bool valid = jn[u] >= 0;
    const int j = valid ? jn[u] : 0;
    const double w = wn[u];
    const int b = bn[u];
    const bool same = valid && b == agg;
    if (same) deg += a.use_weights ? w : 1.0;  // :366-369 / :376-379, self-loops included (Q5)
    // :417 compares the GLOBAL id j with the LOCAL index i (Q1): such an edge, and a self-loop,
    // falls through to a term that is exactly zero, so neither enters the compact list.
    const bool internal = same && j != li && j != v;
    if (valid && !same) {  // :451-466
      double dir[D], d2 = 0.0;
#pragma unroll
      for (int k = 0; k < D; ++k) {
        dir[k] = a.cA[(int64_t)b * D + k] - ca[k];
        d2 += dir[k] * dir[k];
      }
      double dis = sqrt(d2);
      if (dis < kEpsilon) dis = kEpsilon;
#pragma unroll
      for (int k = 0; k < D; ++k) E[k] += dir[k] / dis * 100.0;
    }
    const unsigned mask = __ballot_sync(0xffffffffu, internal);
    if (internal) {
      const int dst = rb + cnt + __popc(mask & ((1u << lane) - 1u));
      a.e_idx[dst] = a.slot_of[j];
      if (a.e_w) a.e_w[dst] = (T)w;
    }
    cnt += __popc(mask);
    }
  }
  for (int off = 16; off > 0; off >>= 1) {
    deg += __shfl_xor_sync(0xffffffffu, deg, off);
#pragma unroll
    for (int k = 0; k < D; ++k) E[k] += __shfl_xor_sync(0xffffffffu, E[k], off);
  }
  if (lane == 0) {
    const double c = deg + 1.0;
    a.mass[slot] = (T)c;
    if (NM > 1) a.mass[a.ld + slot] = (T)(1.5 * c);
    if (NM > 2) a.mass[2 * a.ld + slot] = (T)(1.875 * c);
#pragma unroll
    for (int k = 0; k < D; ++k) a.Eext[(int64_t)k * a.ld + slot] = (T)E[k];
    a.e_begin[slot] = rb;
    a.e_end[slot] = rb + cnt;
    if (slot < a.grid_slots && cnt > a.long_len) a.long_rows[atomicAdd(a.long_count, 1)] = slot;
  }
}

// :539-569 for an aggregate with one member: coords - avg == 0 exactly, max -> eps, so the
// member lands on its parent centre (r_A * 0 kept literal so a non-finite radius propagates).
template <int D>
__global__ void k_ml_singletons(const int* __restrict__ vtx, const int* __restrict__ v_A,
                                const double* __restrict__ cA, const double* __restrict__ rA,
                                int slot_begin, int count, double* __restrict__ out) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= count) return;
  const int v = vtx[slot_begin + t];
  const int a = v_A[v];
  const double c = 0.0 / kEpsilon;
#pragma unroll
  for (int k = 0; k < D; ++k) out[(int64_t)v * D + k] = cA[(int64_t)a * D + k] + rA[a] * c;
}

// Initial local coordinates U(-1,1) drawn on the device (seed 0 = the reference's
// std::random_device mode): a counter-based splitmix64 hash of (seed, element index).
__global__ void k_random_init(double* __restrict__ out, int64_t count, uint64_t seed) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  uint64_t z = seed + 0x9E3779B97F4A7C15ull * (uint64_t)(i + 1);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  out[i] = (double)(z >> 11) * (2.0 / 9007199254740992.0) - 1.0;
}

template <typename T, int D>
__global__ void k_ml_gather_pos(const double* __restrict__ init, const int* __restrict__ vtx,
                                int nslots, int64_t ld, T* __restrict__ pos) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= nslots) return;
  const int v = vtx[s];
#pragma unroll
  for (int k = 0; k < D; ++k) pos[(int64_t)k * ld + s] = v >= 0 ? (T)init[(int64_t)v * D + k] : (T)0;
}

template <typename T, int D>
__global__ void k_ml_scatter_forces(const T* __restrict__ F, const int* __restrict__ vtx,
                                    int nslots, int64_t ld, double* __restrict__ out) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= nslots) return;
  const int v = vtx[s];
  if (v < 0) return;
#pragma unroll
  for (int k = 0; k < D; ++k) out[(int64_t)v * D + k] = (double)F[(int64_t)k * ld + s];
}

// :539-570 for one large aggregate whose positions live in global memory: one CTA per segment.
template <typename T, int D>
__global__ void __launch_bounds__(1024) k_ml_segment_epilogue(const T* __restrict__ pos, int64_t ld,
                                                             const int4* __restrict__ segs,
                                                             const int* __restrict__ vtx,
                                                             const double* __restrict__ cA,
                                                             const double* __restrict__ rA,
                                                             double* __restrict__ out) {
  __shared__ double red[32];
  __shared__ double bc[D + 1];
  const int4 seg = segs[blockIdx.x];
  const int slot0 = seg.x, s = seg.y, agg = seg.z;
  const int tid = threadIdx.x;
  auto block_reduce = [&](double val, bool is_max) -> double {
    for (int off = 16; off > 0; off >>= 1) {
      const double o = __shfl_xor_sync(0xffffffffu, val, off);
      val = is_max ? fmax(val, o) : val + o;
    }
    if ((tid & 31) == 0) red[tid >> 5] = val;
    __syncthreads();
    if (tid < 32) {
      double w = (tid < (int)(blockDim.x >> 5)) ? red[tid] : 0.0;
      for (int off = 16; off > 0; off >>= 1) {
        const double o = __shfl_xor_sync(0xffffffffu, w, off);
        w = is_max ? fmax(w, o) : w + o;
      }
      if (tid == 0) red[0] = w;
    }
    __syncthreads();
    const double r = red[0];
    __syncthreads();
    return r;
  };
  for (int k = 0; k < D; ++k) {
    double part = 0.0;
    for (int i = tid; i < s; i += blockDim.x) part += (double)pos[(int64_t)k * ld + slot0 + i];
    const double tot = block_reduce(part, false);
    if (tid == 0) bc[k] = tot / s;
  }
  __syncthreads();
  double mx = 0.0;
  for (int i = tid; i < s; i += blockDim.x) {
    double m2 = 0.0;
    for (int k = 0; k < D; ++k) {
      const double c = (double)pos[(int64_t)k * ld + slot0 + i] - bc[k];
      m2 += c * c;
    }
    mx = fmax(mx, sqrt(m2));
  }
  double maxlen = block_reduce(mx, true);
  if (maxlen < kEpsilon) maxlen = kEpsilon;
  for (int i = tid; i < s; i += blockDim.x) {
    const int v = vtx[slot0 + i];
    for (int k = 0; k < D; ++k) {
      const double c = ((double)pos[(int64_t)k * ld + slot0 + i] - bc[k]) / maxlen;
      out[(int64_t)v * D + k] = cA[(int64_t)agg * D + k] + rA[agg] * c;
    }
  }
}


// ---------------------------------------------------------------------------------------------
// Slot layout of one level: depends only on the aggregation P_T (and on the on-chip tier limits),
// not on any coordinates -- ge_embed builds it ahead of time, on the copy stream, while the
// coarsest-level solve runs.
// ---------------------------------------------------------------------------------------------
struct CtaClass {  // CTA tier: one launch per lanes-per-vertex class (the kernel is specialised on it)
  std::vector<int4> tasks;
  int threads = 32, size_max = 1;
};
}  // namespace

struct LevelLayout {
  std::vector<int4> segs, packs;
  CtaClass cta_class[4];  // L = 1, 2, 4, 8
  int grid_slots = 0, single_begin = 0, n_single = 0, nslots = 0;
  int64_t ld = 0;
  double pairs = 0.0;
  DevBuf<int> d_vA, d_vtx, d_slot_of, d_agg_base, d_agg_of_slot;
  DevBuf<int> d_PI, d_PJ;  // the aggregation's CSR (member lists): the families of the radii step
  int n = 0, m = 0, agg_begin = 0, agg_end = 0, n_owned = -1;  // n_owned >= 0: an explicit aggregate set
};

namespace {
void build_level_layout(ge_context* ctx, const ge_csr& P, int n, const int32_t* v_A, bool forces_only,
                        int agg_begin, int agg_end, LevelLayout& L_, bool members = false,
                        const std::vector<int>* owned = nullptr) {
  // the aggregates this layout solves: a contiguous range, or (multi-device embed) an explicit set
  auto for_each_aggregate = [&](auto&& body) {
    if (owned != nullptr) {
      for (int a : *owned) body(a);
    } else {
      for (int a = agg_begin; a < agg_end; ++a) body(a);
    }
  };
  const int m = P.rows;
  int cta_max = std::min(env_int("GE_CTA_MAX", 512), kOnchipMaxVertices);
  if (std::getenv("GE_CTA_MAX") == nullptr) {
    // A SMALL multi-CTA tier is all launch overhead and pipeline fill: below the size where the
    // tier runs on the symmetric sweep (8e6 pairs per iteration) its aggregates of up to 1024
    // members are better off with one persistent CTA each.  Above, the captured sweep + long-row
    // attraction wins (R-MAT-20 level 2, 28 aggregates of 653 members, 1.9e7 pairs: 14.4 vs
    // 16.3 ms), and large tiers keep the measured 512 limit anyway (level 0 of the same hierarchy:
    // 14.7 vs 21.2 ms).
    double big_pairs = 0.0;
    for_each_aggregate([&](int a) {
      const double sz = P.indptr[a + 1] - P.indptr[a];
      if (sz > cta_max) big_pairs += sz * (sz - 1);
    });
    if (big_pairs > 0.0 && big_pairs < 1e6 * env_int("GE_ML_SYM_MIN_MPAIRS", 8)) cta_max = kOnchipMaxVertices;
  }
  std::vector<int4>& segs = L_.segs;
  std::vector<int4>& packs = L_.packs;
  CtaClass* cta_class = L_.cta_class;
  // ---- host: bin aggregates by size and lay out the slots -------------------------------------
  std::vector<int> by_size[33];
  std::vector<int> cta_aggs, grid_aggs;
  double pairs = 0.0;
  for_each_aggregate([&](int a) {
    const int s = P.indptr[a + 1] - P.indptr[a];
    pairs += double(s) * double(s - 1);
    if (s <= 0) return;
    if (s <= 32) by_size[s].push_back(a);
    else if (s <= cta_max) cta_aggs.push_back(a);
    else grid_aggs.push_back(a);
  });
  L_.pairs = pairs;
  auto size_of = [&](int a) { return P.indptr[a + 1] - P.indptr[a]; };
  std::sort(cta_aggs.begin(), cta_aggs.end(), [&](int x, int y) { return size_of(x) > size_of(y); });

  std::vector<int> agg_base(std::max(m, 1), 0);
  int64_t cursor = 0;
  for (int a : grid_aggs) {
    const int s = size_of(a);
    agg_base[a] = (int)cursor;
    segs.push_back(make_int4((int)cursor, s, a, 0));
    cursor = round_up(cursor + s, kTileJ);
  }
  L_.grid_slots = (int)cursor;
  for (int a : cta_aggs) {
    const int s = size_of(a);
    agg_base[a] = (int)cursor;
    int L = 1, li = 0;
    while (L < 8 && (int64_t)s * (L * 2) <= kOnchipMaxThreads) {
      L *= 2;
      ++li;
    }
    CtaClass& cc = cta_class[li];
    cc.tasks.push_back(make_int4((int)cursor, s, a, L));
    cc.threads = std::max<int>(cc.threads, (int)round_up((int64_t)s * L, 32));
    cc.size_max = std::max(cc.size_max, s);
    cursor += s;
  }
  const int single_lo = forces_only ? 1 : 2;  // forces hook: singletons go through the warp tier
  for (int s = 32; s >= single_lo; --s) {
    const int per = 32 / s;
    const auto& list = by_size[s];
    for (size_t i0 = 0; i0 < list.size(); i0 += per) {
      const int cnt = (int)std::min<size_t>(per, list.size() - i0);
      packs.push_back(make_int4((int)cursor, s, cnt, 0));
      for (int q = 0; q < cnt; ++q) {
        agg_base[list[i0 + q]] = (int)cursor;
        cursor += s;
      }
    }
  }
  L_.single_begin = (int)cursor;
  if (!forces_only) {
    for (int a : by_size[1]) agg_base[a] = (int)cursor++;
    L_.n_single = (int)by_size[1].size();
  }
  L_.nslots = (int)cursor;
  const int64_t ld = round_up(std::max(L_.nslots, 1), kTileJ);
  L_.ld = ld;
  std::vector<int> vtx((size_t)ld, -1), slot_of(std::max(n, 1), -1), agg_of_slot((size_t)ld, -1);
  for_each_aggregate([&](int a) {
    const int s = size_of(a);
    for (int i = 0; i < s; ++i) {
      const int v = P.indices[P.indptr[a] + i];
      vtx[agg_base[a] + i] = v;
      slot_of[v] = agg_base[a] + i;
      agg_of_slot[agg_base[a] + i] = a;
    }
  });

  // the vertex -> aggregate map: the caller's, or derived from P_T
  std::vector<int32_t> vA_local;
  if (v_A == nullptr) {
    vA_local.assign(std::max(n, 1), 0);
    for (int a = 0; a < m; ++a)
      for (int c = P.indptr[a]; c < P.indptr[a + 1]; ++c) vA_local[P.indices[c]] = a;
    v_A = vA_local.data();
  }
  L_.d_vA.alloc(ctx, std::max(n, 1));
  L_.d_vtx.alloc(ctx, (size_t)ld);
  L_.d_slot_of.alloc(ctx, std::max(n, 1));
  L_.d_agg_base.alloc(ctx, std::max(m, 1));
  L_.d_agg_of_slot.alloc(ctx, (size_t)ld);
  L_.d_vA.upload(ctx, v_A, n);
  L_.d_vtx.upload(ctx, vtx.data(), (size_t)ld);
  L_.d_slot_of.upload(ctx, slot_of.data(), n);
  L_.d_agg_base.upload(ctx, agg_base.data(), m);
  L_.d_agg_of_slot.upload(ctx, agg_of_slot.data(), (size_t)ld);
  if (members) {
    L_.d_PI.alloc(ctx, (size_t)m + 1);
    L_.d_PJ.alloc(ctx, (size_t)std::max(n, 1));
    L_.d_PI.upload(ctx, P.indptr, (size_t)m + 1);
    L_.d_PJ.upload(ctx, P.indices, (size_t)n);
  }
  L_.n = n;
  L_.m = m;
  L_.agg_begin = agg_begin;
  L_.agg_end = agg_end;
  L_.n_owned = owned ? (int)owned->size() : -1;
  // (copies from pageable memory have left the host arrays when cudaMemcpyAsync returns)
}

template <typename T>
void multilevel_t(ge_context* ctx, const ge_csr& A, const ge_csr& P, const int32_t* v_A,
                  const double* coords_A, const double* r_A, const double* init,
                  double* coords_out, int dim, const ge_params& p, bool forces_only,
                  double* pairs_out, int agg_begin, int agg_end, const PrefetchedGraph* pre,
                  const LevelIO* io) {
  constexpr int NM = Real<T>::kMassArrays;
  const int n = A.rows, m = P.rows;
  const int nnz = A.indptr[n];
  // a prepared graph carries its own weights (ge_layout_graph's levels are on the device only)
  const bool has_weights = pre != nullptr ? pre->Dw.size() != 0 : A.data != nullptr;
  const bool weighted = p.use_weights && has_weights;

  const bool verbose = std::getenv("GE_VERBOSE") != nullptr;
  double t_mark = now_ms();
  auto lap = [&](const char* what) {
    if (!verbose) return;
    GE_CUDA(cudaStreamSynchronize(ctx->stream));
    const double t = now_ms();
    std::fprintf(stderr, "[ge] level n=%d %-18s %8.3f ms\n", n, what, t - t_mark);
    t_mark = t;
  };
  // ---- slot layout (host + its device copies): prepared ahead of time or built here ----------
  LevelLayout own_layout;
  const LevelLayout* lay = (pre != nullptr && pre->layout != nullptr) ? pre->layout : nullptr;
  const std::vector<int>* owned = io ? io->owned : nullptr;
  if (lay != nullptr)
    GE_REQUIRE(owned ? lay->n_owned == (int)owned->size()
                     : (lay->n_owned < 0 && lay->agg_begin == agg_begin && lay->agg_end == agg_end),
               "prepared layout covers another set of aggregates");
  if (lay == nullptr) {
    build_level_layout(ctx, P, n, v_A, forces_only, agg_begin, agg_end, own_layout, false, owned);
    lay = &own_layout;
  }
  if (pairs_out) *pairs_out = lay->pairs;
  const std::vector<int4>& segs = lay->segs;
  const std::vector<int4>& packs = lay->packs;
  const CtaClass* cta_class = lay->cta_class;
  const int grid_slots = lay->grid_slots, single_begin = lay->single_begin, n_single = lay->n_single;
  const int nslots = lay->nslots;
  const int64_t ld = lay->ld;
  const DevBuf<int>&d_vA = lay->d_vA, &d_vtx = lay->d_vtx, &d_slot_of = lay->d_slot_of,
                   &d_agg_base = lay->d_agg_base, &d_agg_of_slot = lay->d_agg_of_slot;
  lap("host layout");
  // ---- upload ------------------------------------------------------------------------------
  DevBuf<int> d_I, d_J, d_eb(ctx, (size_t)ld), d_ee(ctx, (size_t)ld), d_eidx(ctx, std::max(nnz, 1));
  const bool dev_in = io != nullptr && io->d_coords_A != nullptr;
  DevBuf<double> d_Dw, d_cA, d_rA, d_init(ctx, (size_t)std::max(n, 1) * dim), d_out(ctx, (size_t)std::max(n, 1) * dim);
  if (!dev_in) {
    d_cA.alloc(ctx, (size_t)std::max(m, 1) * dim);
    d_rA.alloc(ctx, std::max(m, 1));
  }
  DevBuf<T> d_mass(ctx, (size_t)NM * ld), d_E(ctx, (size_t)dim * ld), d_ew;
  const int* dI;
  const int* dJ;
  const double* dDw = nullptr;
  if (pre != nullptr) {  // the graph was uploaded ahead of time on the copy stream
    GE_CUDA(cudaStreamWaitEvent(ctx->stream, pre->ready, 0));
    dI = pre->I.get();
    dJ = pre->J.get();
    if (has_weights) dDw = pre->Dw.get();
  } else {
    d_I.alloc(ctx, n + 1);
    d_J.alloc(ctx, std::max(nnz, 1));
    d_I.upload(ctx, A.indptr, n + 1);
    d_J.upload(ctx, A.indices, nnz);
    if (A.data != nullptr) {
      d_Dw.alloc(ctx, std::max(nnz, 1));
      d_Dw.upload(ctx, A.data, nnz);
      dDw = d_Dw.get();
    }
    dI = d_I.get();
    dJ = d_J.get();
  }
  if (weighted) d_ew.alloc(ctx, std::max(nnz, 1));
  if (!dev_in) {
    d_cA.upload(ctx, coords_A, (size_t)m * dim);
    d_rA.upload(ctx, r_A, m);
  }
  const double* dcA = dev_in ? io->d_coords_A : d_cA.get();
  const double* drA = dev_in ? io->d_r_A : d_rA.get();
  if (init != nullptr) {
    d_init.upload(ctx, init, (size_t)n * dim);
  } else {
    const int64_t count = (int64_t)n * dim;
    const uint64_t seed64 = ((uint64_t)resolve_seed(0) << 32) | resolve_seed(0);
    if (count > 0)
      k_random_init<<<(unsigned)((count + 255) / 256), 256, 0, ctx->stream>>>(d_init.get(), count, seed64);
    ctx->launches++;
  }
  d_eb.zero(ctx->stream);
  d_ee.zero(ctx->stream);
  if (agg_begin > 0 || agg_end < m || owned != nullptr) d_out.zero(ctx->stream);  // rows of other ranks' aggregates

  lap("upload");
  // ---- prep --------------------------------------------------------------------------------
  PrepArgs<T> pa;
  pa.I = dI;
  pa.J = dJ;
  pa.Dw = dDw;
  pa.v_A = d_vA.get();
  pa.vtx = d_vtx.get();
  pa.slot_of = d_slot_of.get();
  pa.agg_base = d_agg_base.get();
  pa.cA = dcA;
  pa.mass = d_mass.get();
  pa.Eext = d_E.get();
  pa.e_begin = d_eb.get();
  pa.e_end = d_ee.get();
  pa.e_idx = d_eidx.get();
  pa.e_w = weighted ? d_ew.get() : nullptr;
  pa.ld = ld;
  pa.nslots = nslots;
  pa.use_weights = p.use_weights;
  const int long_len = env_int("GE_ML_LONG_ROW", 128);
  DevBuf<int> d_long_rows, d_long_count(ctx, 1);
  d_long_count.zero(ctx->stream);
  if (grid_slots > 0) d_long_rows.alloc(ctx, (size_t)grid_slots);
  pa.grid_slots = long_len > 0 ? grid_slots : 0;
  pa.long_len = long_len;
  pa.long_rows = d_long_rows.get();
  pa.long_count = d_long_count.get();
  d_mass.zero(ctx->stream);
  d_E.zero(ctx->stream);
  if (nslots > 0) {
    const unsigned grid = (unsigned)(((int64_t)nslots * 32 + 255) / 256);
    if (dim == 2) k_ml_prep<T, 2><<<grid, 256, 0, ctx->stream>>>(pa);
    else k_ml_prep<T, 3><<<grid, 256, 0, ctx->stream>>>(pa);
    GE_CUDA(cudaGetLastError());
    ctx->launches++;
  }

  lap("prep kernel");
  OnchipArgs<T> oa;
  oa.init_aos = d_init.get();
  oa.vtx = d_vtx.get();
  oa.agg_of_slot = d_agg_of_slot.get();
  oa.mass = d_mass.get();
  oa.e_begin = d_eb.get();
  oa.e_end = d_ee.get();
  oa.e_idx = d_eidx.get();
  oa.e_w = weighted ? d_ew.get() : nullptr;
  oa.Eext = d_E.get();
  oa.ld = ld;
  oa.cA_aos = dcA;
  oa.rA = drA;
  oa.out_aos = d_out.get();
  oa.iters = p.iterations;
  oa.forces_only = forces_only ? 1 : 0;
  oa.normalize = 0;
  oa.ph = make_physics<T>(p);

  // ---- singletons --------------------------------------------------------------------------
  if (n_single > 0) {
    const unsigned grid = (unsigned)((n_single + 255) / 256);
    if (dim == 2)
      k_ml_singletons<2><<<grid, 256, 0, ctx->stream>>>(d_vtx.get(), d_vA.get(), dcA,
                                                        drA, single_begin, n_single, d_out.get());
    else
      k_ml_singletons<3><<<grid, 256, 0, ctx->stream>>>(d_vtx.get(), d_vA.get(), dcA,
                                                        drA, single_begin, n_single, d_out.get());
    GE_CUDA(cudaGetLastError());
    ctx->launches++;
  }

  // ---- warp tier ---------------------------------------------------------------------------
  DevBuf<int4> d_packs(ctx, std::max<size_t>(packs.size(), 1)), d_segs(ctx, std::max<size_t>(segs.size(), 1));
  if (!packs.empty()) {
    d_packs.upload(ctx, packs.data(), packs.size());
    OnchipArgs<T> wa = oa;
    wa.tasks = d_packs.get();
    launch_onchip_warp<T>(ctx, wa, (int)packs.size(), dim);
  }
  // ---- CTA tier ----------------------------------------------------------------------------
  std::vector<DevBuf<int4>> d_cta_tasks(4);
  for (int li = 0; li < 4; ++li) {
    const CtaClass& cc = cta_class[li];
    if (cc.tasks.empty()) continue;
    d_cta_tasks[li].alloc(ctx, cc.tasks.size());
    d_cta_tasks[li].upload(ctx, cc.tasks.data(), cc.tasks.size());
    OnchipArgs<T> ca = oa;
    ca.tasks = d_cta_tasks[li].get();
    launch_onchip_cta<T>(ctx, ca, (int)cc.tasks.size(), dim, true, 1 << li, cc.threads, cc.size_max);
  }
  // ---- grid tier ---------------------------------------------------------------------------
  DevBuf<T> d_pos0, d_pos1, d_Frep, d_Fprev;
  cudaEvent_t tier_ev[2] = {nullptr, nullptr};
  if (!segs.empty()) {
    GE_CUDA(cudaEventCreate(&tier_ev[0]));
    GE_CUDA(cudaEventCreate(&tier_ev[1]));
    GE_CUDA(cudaEventRecord(tier_ev[0], ctx->stream));
    d_segs.upload(ctx, segs.data(), segs.size());
    d_pos0.alloc(ctx, (size_t)dim * ld);
    d_pos1.alloc(ctx, (size_t)dim * ld);
    d_Frep.alloc(ctx, (size_t)dim * ld);
    d_Fprev.alloc(ctx, (size_t)dim * ld);
    d_pos0.zero(ctx->stream);
    d_pos1.zero(ctx->stream);
    d_Frep.zero(ctx->stream);
    d_Fprev.zero(ctx->stream);
    const unsigned ggrid = (unsigned)((grid_slots + 255) / 256);
    if (dim == 2) k_ml_gather_pos<T, 2><<<ggrid, 256, 0, ctx->stream>>>(d_init.get(), d_vtx.get(), grid_slots, ld, d_pos0.get());
    else k_ml_gather_pos<T, 3><<<ggrid, 256, 0, ctx->stream>>>(d_init.get(), d_vtx.get(), grid_slots, ld, d_pos0.get());
    GE_CUDA(cudaGetLastError());
    ctx->launches++;
    // Repulsion plan of the tier: from a few million pairs per iteration on, every unordered pair
    // inside an aggregate is evaluated once (k_repulsion_sym over one segment per aggregate);
    // small tiers keep the ordered sweep with its fine-grained units.
    double tier_pairs = 0.0;
    for (auto& sg : segs) tier_pairs += double(sg.y) * double(sg.y - 1);
    const bool use_sym = tier_pairs >= 1e6 * env_int("GE_ML_SYM_MIN_MPAIRS", 8) && env_int("GE_ML_SYM", 1) != 0;
    std::unique_ptr<RepulsionPlan<T>> rep;
    std::unique_ptr<RepulsionSymPlan<T>> sym;
    if (use_sym) {
      std::vector<SymSegment> ssegs;
      for (auto& sg : segs) ssegs.push_back(SymSegment{sg.x, sg.x + sg.y});
      sym.reset(new RepulsionSymPlan<T>(ctx, dim, ld, ssegs));
    } else {
      std::vector<RowSegment> rsegs;
      for (auto& sg : segs)
        rsegs.push_back(RowSegment{sg.x, sg.x + sg.y, sg.x, (int)round_up((int64_t)sg.x + sg.y, kTileJ)});
      rep.reset(new RepulsionPlan<T>(ctx, dim, rsegs));
    }
    int nlong = 0;  // rows the prep kernel listed for the CTA-per-row attraction kernel
    d_long_count.download(ctx, &nlong, 1);
    GE_CUDA(cudaStreamSynchronize(ctx->stream));
    T* pos[2] = {d_pos0.get(), d_pos1.get()};
    int cur = 0;
    const int iters = forces_only ? 1 : p.iterations;
    const double avg_deg = grid_slots > 0 ? double(nnz) / std::max(n, 1) : 0.0;
    const int group = group_for_degree(avg_deg);
    auto one_iteration = [&]() {
      if (sym) sym->launch(pos[cur], d_mass.get(), d_Frep.get(), oa.ph.eps2, oa.ph.repel);
      else rep->launch(pos[cur], d_mass.get(), ld, d_Frep.get(), ld, 0, oa.ph.repel, oa.ph.eps2);
      StepArgs<T> sa;
      sa.e_begin = d_eb.get();
      sa.e_end = d_ee.get();
      sa.J = d_eidx.get();
      sa.W = weighted ? d_ew.get() : nullptr;
      sa.pos_cur = pos[cur];
      sa.pos_next = pos[cur ^ 1];
      sa.Frep = d_Frep.get();
      sa.Fprev = d_Fprev.get();
      sa.mass = d_mass.get();
      sa.Eext = d_E.get();
      sa.ld = ld;
      sa.ldf = ld;
      sa.row0 = 0;
      sa.nrows = grid_slots;
      sa.update = forces_only ? 0 : 1;
      sa.ph = oa.ph;
      sa.long_threshold = nlong > 0 ? long_len : 0;
      launch_attract_step<T>(ctx, sa, dim, group, true);
      launch_attract_step_long<T>(ctx, sa, dim, d_long_rows.get(), nlong, 128, true);
      if (!forces_only) cur ^= 1;
    };
    int it = 0;
    // The iterations of a tier are 3-4 short launches each: the steady-state pair of iterations
    // (the position buffers ping-pong) is captured once and replayed.
    if (iters >= 8 && std::getenv("GE_NO_GRAPH") == nullptr) {
      for (; it < 2; ++it) one_iteration();
      cudaGraph_t graph = nullptr;
      cudaGraphExec_t exec = nullptr;
      const int64_t launches_before = ctx->launches;
      GE_CUDA(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
      one_iteration();
      one_iteration();
      GE_CUDA(cudaStreamEndCapture(ctx->stream, &graph));
      const int64_t per_replay = ctx->launches - launches_before;
      ctx->launches = launches_before;
      GE_CUDA(cudaGraphInstantiate(&exec, graph, 0));
      for (; it + 2 <= iters; it += 2) {
        GE_CUDA(cudaGraphLaunch(exec, ctx->stream));
        ctx->launches += per_replay;
      }
      GE_CUDA(cudaStreamSynchronize(ctx->stream));
      cudaGraphExecDestroy(exec);
      cudaGraphDestroy(graph);
    }
    for (; it < iters; ++it) one_iteration();
    if (forces_only) {
      if (dim == 2) k_ml_scatter_forces<T, 2><<<ggrid, 256, 0, ctx->stream>>>(d_Fprev.get(), d_vtx.get(), grid_slots, ld, d_out.get());
      else k_ml_scatter_forces<T, 3><<<ggrid, 256, 0, ctx->stream>>>(d_Fprev.get(), d_vtx.get(), grid_slots, ld, d_out.get());
    } else {
      if (dim == 2) k_ml_segment_epilogue<T, 2><<<(unsigned)segs.size(), 1024, 0, ctx->stream>>>(pos[cur], ld, d_segs.get(), d_vtx.get(), dcA, drA, d_out.get());
      else k_ml_segment_epilogue<T, 3><<<(unsigned)segs.size(), 1024, 0, ctx->stream>>>(pos[cur], ld, d_segs.get(), d_vtx.get(), dcA, drA, d_out.get());
    }
    GE_CUDA(cudaGetLastError());
    ctx->launches++;
    GE_CUDA(cudaEventRecord(tier_ev[1], ctx->stream));
  }

  lap("solve kernels");
  if (io == nullptr || io->download) d_out.download(ctx, coords_out, (size_t)n * dim);
  GE_CUDA(cudaStreamSynchronize(ctx->stream));
  if (io != nullptr && io->keep_out != nullptr) *io->keep_out = std::move(d_out);
  if (tier_ev[0] != nullptr) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, tier_ev[0], tier_ev[1]) == cudaSuccess) ctx->grid_tier_ms += ms;
    cudaEventDestroy(tier_ev[0]);
    cudaEventDestroy(tier_ev[1]);
  }
  lap("download");
}

}  // namespace

LevelLayout* make_level_layout(ge_context* ctx, const ge_csr& P_T, int n, int agg_begin, int agg_end,
                               bool members, const std::vector<int>* owned) {
  if (agg_end < 0) agg_end = P_T.rows;
  std::unique_ptr<LevelLayout> L(new LevelLayout);
  build_level_layout(ctx, P_T, n, nullptr, false, agg_begin, agg_end, *L, members, owned);
  return L.release();
}
void free_level_layout(LevelLayout* layout) { delete layout; }

RadiiLevel radii_level_of(const PrefetchedGraph& g, int mc) {
  GE_REQUIRE(g.layout != nullptr && g.layout->d_PI.size() > 0, "level layout without member lists");
  RadiiLevel lv;
  lv.I = g.I.get();
  lv.J = g.J.get();
  lv.parent = g.layout->d_vA.get();
  lv.PI = g.layout->d_PI.get();
  lv.PJ = g.layout->d_PJ.get();
  lv.mc = mc;
  return lv;
}

void multilevel_solve(ge_context* ctx, const ge_csr& A, const ge_csr& P_T, const int32_t* v_A,
                      const double* coords_A, const double* r_A, const double* init,
                      double* coords_out, int dim, const ge_params& p, bool forces_only,
                      double* pairs_out, int agg_begin, int agg_end, const PrefetchedGraph* pre,
                      const LevelIO* io) {
  if (agg_end < 0) agg_end = P_T.rows;
  GE_REQUIRE(0 <= agg_begin && agg_begin <= agg_end && agg_end <= P_T.rows, "bad aggregate range");
  GE_REQUIRE(dim == 2 || dim == 3, "dim must be 2 or 3");
  GE_REQUIRE(A.rows == A.cols, "A must be square");
  GE_REQUIRE(P_T.cols == A.rows, "P_T.cols must equal A.rows");
  GE_REQUIRE(P_T.indptr[P_T.rows] == A.rows, "P_T must list every vertex exactly once");
  if (p.precision == GE_F32)
    multilevel_t<float>(ctx, A, P_T, v_A, coords_A, r_A, init, coords_out, dim, p, forces_only, pairs_out, agg_begin, agg_end, pre, io);
  else
    multilevel_t<double>(ctx, A, P_T, v_A, coords_A, r_A, init, coords_out, dim, p, forces_only, pairs_out, agg_begin, agg_end, pre, io);
}

}  // namespace ge

/*
 * graph_embed_b200.h -- C ABI of the B200-native ForceAtlas hot path of LLNL/graph-embed.
 *
 * This is the drop-in boundary.  Everything below is `extern "C"`, plain pointers and sizes;
 * no C++ or torch types cross it.  All host buffers are caller-owned and not retained after a
 * call returns (same ownership as the reference's `const&` inputs, SURVEY.md section 8b); device
 * buffers live inside the opaque handles.  Coordinates cross the ABI as row-major n x dim
 * doubles, the flat image of the reference's `std::vector<std::vector<double>>`.
 *
 * The reference interface each entry point replaces is cited as file:line relative to the
 * reference tree (/root/reference).  The C++ header-only shim that keeps the reference's own
 * signatures (`partition::embed`, `partition::forceAtlas`, ...) on top of this ABI is
 * graph-embed_b200/host/include/embed.hpp; INTEGRATION.md shows the binding a maintainer of the
 * reference would add.
 *
 * There is no CPU fallback: every compute entry point returns GE_ERR_NO_DEVICE when no CUDA
 * device is usable.
 */
#ifndef GRAPH_EMBED_B200_H
#define GRAPH_EMBED_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum ge_status {
  GE_OK = 0,
  GE_ERR_INVALID = 1,     /* bad argument (shape mismatch, null pointer, unsupported dim) */
  GE_ERR_NO_DEVICE = 2,   /* no usable CUDA device / driver */
  GE_ERR_CUDA = 3,        /* a CUDA runtime call or kernel failed; see ge_last_error() */
  GE_ERR_OOM = 4,         /* device or host allocation failed */
  GE_ERR_UNSUPPORTED = 5  /* valid request this build does not implement */
} ge_status;

typedef enum ge_precision { GE_F64 = 0, GE_F32 = 1 } ge_precision;

/* CSR view of a linalgcpp::SparseMatrix<double> (GetIndptr/GetIndices/GetData/Rows/Cols,
 * used at include/forceatlas.hpp:112-116, 342-346).  data may be NULL = all ones. */
typedef struct ge_csr {
  int32_t rows, cols;
  int64_t nnz;
  const int32_t* indptr;  /* rows + 1 */
  const int32_t* indices; /* nnz */
  const double* data;     /* nnz or NULL */
} ge_csr;

/* The default arguments of forceAtlas (include/forceatlas.hpp:92-103) and
 * forceAtlasMultilevel (:320-331), plus the knobs the reference does not have. */
typedef struct ge_params {
  int32_t iterations; /* flat default 100000 (:92); multilevel declared 10 (:321), embed passes 100 */
  double ks;          /* 0.1 */
  double ksmax;       /* 1.0 */
  double repel;       /* 1.0 */
  double attract;     /* 1.0 */
  double gravity;     /* 1.0 */
  double delta;       /* 1.0 */
  double tolerate;    /* 1.0 */
  int32_t use_weights; /* 1 */
  int32_t linlog;      /* 0 */
  int32_t nohubs;      /* 0 */
  int32_t normalize;   /* 0; flat only (:272-303) */
  int32_t precision;   /* ge_precision; arithmetic type of the device path (reference: FP64) */
  uint32_t seed;       /* 0 = std::random_device like the reference; else std::mt19937(seed) */
} ge_params;

/* Options of ge_embed; zero-initialise then call ge_embed_options_default. */
typedef struct ge_embed_options {
  int32_t coarse_iterations; /* 100000: forceAtlas defaults at the coarsest level (src/embed.cpp:586) */
  int32_t level_iterations;  /* 100:    src/embed.cpp:793 */
  int32_t precision;         /* ge_precision */
  uint32_t seed;             /* 0 = std::random_device; else every stream = std::mt19937(seed) */
  int32_t verbose;           /* 1 = print the reference's "embedding layer N" lines (src/embed.cpp:583,613) */
  int32_t first_layer;       /* layer number printed for As[0] (1; embedMultilevel from level k passes k+1) */
} ge_embed_options;

/* Per-call statistics filled by ge_embed (all optional to read). */
typedef struct ge_embed_stats {
  double total_ms;        /* wall time of the whole call */
  double coarse_ms;       /* device time of the coarsest-level flat solve */
  double levels_ms;       /* device time of all multilevel levels */
  double host_radii_ms;   /* host time in the ball-radius / rescale step */
  double h2d_bytes, d2h_bytes;
  double pair_interactions; /* ordered pairs x iterations, all levels */
  double edge_visits;       /* CSR entries x iterations, all levels */
  int64_t kernel_launches;
  double grid_tier_ms;    /* device time of the multi-CTA tier (aggregates > 512 members), all levels */
  double device_radii_ms; /* device time of the ball-radius / rescale kernels, all levels */
} ge_embed_stats;

typedef struct ge_context ge_context;     /* device, stream, scratch */
typedef struct ge_flat_plan ge_flat_plan; /* device-resident flat solver (one row block) */

/* ---- library ---------------------------------------------------------------------------- */
const char* ge_version(void);
/* Message of the last failing call on this thread ("" if none). */
const char* ge_last_error(void);
void ge_params_default_flat(ge_params* p);       /* include/forceatlas.hpp:92-103 */
void ge_params_default_multilevel(ge_params* p); /* include/forceatlas.hpp:320-331, iterations = 100 */
void ge_embed_options_default(ge_embed_options* o);

/* ---- context ---------------------------------------------------------------------------- */
/* device < 0 selects the current device.  stream == NULL: the context creates its own. */
ge_status ge_context_create(int device, void* cuda_stream, ge_context** out);
/* One process, `ndev` GPUs of one box (device ordinals devices[0..ndev), or 0..ndev-1 when devices
 * is NULL): the context owns a stream and memory pool per device and an NCCL communicator over
 * them (NCCL is bound at run time; GE_ERR_UNSUPPORTED if libnccl.so.2 cannot be loaded).  On such a
 * context ge_flat_forceatlas -- hence partition::forceAtlas through the C++ shim -- shards the
 * iteration: every device evaluates 1/ndev of the unordered pairs, the pair sums are
 * reduce-scattered, each device steps its row block and the new positions are all-gathered
 * (include/forceatlas.hpp:146-270; no all-reduce, the global swing sums are dead code).  Graphs
 * below 32768 vertices and the other entry points run on devices[0].  ndev must divide the row
 * count padded to 256 (1, 2, 4, 8 always do). */
ge_status ge_context_create_multi(int ndev, const int* devices, ge_context** out);
int32_t ge_context_device_count(const ge_context* ctx);
void ge_context_destroy(ge_context* ctx);
/* Kernels launched by this context since creation (the library counts its own launches). */
int64_t ge_context_launch_count(const ge_context* ctx);
/* Bytes this context copied host->device / device->host since creation. */
void ge_context_bytes(const ge_context* ctx, double* h2d, double* d2h);
/* Roofline denominator for the repulsion kernels: sustained FMA rate (TFLOP/s, 2 flops per FMA)
 * of the FP64 or FP32 pipe, measured with a register-resident independent-FMA kernel over all
 * SMs and timed with CUDA events. */
ge_status ge_measure_fma_peak(ge_context* ctx, int precision, double* tflops);

/* ---- the reference's kernels, host buffers in and out ------------------------------------ */

/* partition::forceAtlas(A, dim, coords, iterations, ks, ksmax, repel, attract, gravity,
 * useWeights, linlog, nohubs, delta, tolerate, normalize)      include/forceatlas.hpp:89-305.
 * coords: n x dim, in (initial positions) / out.  The random initialisation of :118-125 is done
 * by the caller-side shim (or ge_embed) so that this entry point is deterministic. */
ge_status ge_flat_forceatlas(ge_context* ctx, const ge_csr* A, int dim, double* coords,
                             const ge_params* p);

/* partition::forceAtlasMultilevel(A, P, v_A, coords_A, r_A, coords, dim, iterations, ...)
 *                                                              include/forceatlas.hpp:314-574.
 * P_T: m x n aggregation matrix; v_A: n (vertex -> aggregate); coords_A: m x dim; r_A: m.
 * init: n x dim initial LOCAL coordinates by global vertex id, or NULL to draw them from
 * std::mt19937 in the reference's order (:341, :356-358) using p->seed.  coords: n x dim out. */
ge_status ge_multilevel_forceatlas(ge_context* ctx, const ge_csr* A, const ge_csr* P_T,
                                   const int32_t* v_A, const double* coords_A, const double* r_A,
                                   const double* init, double* coords, int dim,
                                   const ge_params* p);

/* The same for the aggregates [agg_begin, agg_end) only (multi-GPU: aggregates are independent,
 * include/forceatlas.hpp:340-341, so ranks take disjoint ranges and exchange the level's output
 * once).  Rows of `coords` that belong to other aggregates are set to 0, so the exchange can be a
 * sum (x + 0 is exact). */
ge_status ge_multilevel_forceatlas_shard(ge_context* ctx, const ge_csr* A, const ge_csr* P_T,
                                         const int32_t* v_A, const double* coords_A,
                                         const double* r_A, const double* init, double* coords,
                                         int dim, const ge_params* p, int32_t agg_begin,
                                         int32_t agg_end);

/* partition::embed(As, P_Ts, d)  src/embed.cpp:561-574, i.e. the embedMultilevel recursion of
 * :576-796: coarsest level flat solve, then per level radii + rescale (:615-777, host) and the
 * per-aggregate solve + prolongation.  As: n_levels + 1 matrices, P_Ts: n_levels.
 * coords_out: As[0].rows x dim.  r_A_out (As[1].rows) / coords_A_out (As[1].rows x dim), when not
 * NULL and n_levels > 0, receive what embedMultilevel leaves in its r_A / coords_A out-parameters:
 * the radii and rescaled coordinates of level 1.  opt / stats may be NULL. */
ge_status ge_embed(ge_context* ctx, int n_levels, const ge_csr* As, const ge_csr* P_Ts, int dim,
                   const ge_embed_options* opt, double* coords_out, double* r_A_out,
                   double* coords_A_out, ge_embed_stats* stats);

/* ---- parity hooks: forces of ONE iteration from given positions --------------------------- */
/* include/forceatlas.hpp:148-212 -> forces (n x dim).  `path`: 0 = auto, 1 = tiled multi-CTA
 * kernels (large-n path), 2 = on-chip persistent kernel (small-n path). */
ge_status ge_flat_forces(ge_context* ctx, const ge_csr* A, int dim, const double* coords,
                         const ge_params* p, int path, double* forces);
/* include/forceatlas.hpp:391-475 for every aggregate, positions n x dim by global vertex id. */
ge_status ge_multilevel_forces(ge_context* ctx, const ge_csr* A, const ge_csr* P_T,
                               const int32_t* v_A, const double* coords_A,
                               const double* positions, int dim, const ge_params* p,
                               double* forces);

/* ---- host-side level-driver step (no device needed) -------------------------------------- */
/* src/embed.cpp:615-778: ball radii r_A (m) of the level whose coordinates coords_A (m x dim,
 * rescaled in place) were just computed.  Base case (:616-679): A_c = P_T_c = NULL.  General
 * case (:680-777): A_c = graph of that level (m rows), P_T_c = its aggregation (mc x m),
 * coords_Ac (mc x dim) / r_Ac (mc) = the next-coarser level's rescaled centres and radii. */
ge_status ge_level_radii(int m, int dim, double* coords_A, double* r_A, const ge_csr* A_c,
                         const ge_csr* P_T_c, const double* coords_Ac, const double* r_Ac);
/* The same step on the device (SURVEY.md section 8 row f1): one CTA per family pops the events in
 * the reference's order; bit-identical to ge_level_radii.  ge_embed runs this between the levels
 * on coordinates that never leave the device; this entry point (host buffers in and out) exists
 * for callers that drive the levels themselves (embedVia) and for the parity tests. */
ge_status ge_level_radii_device(ge_context* ctx, int m, int dim, double* coords_A, double* r_A,
                                const ge_csr* A_c, const ge_csr* P_T_c, const double* coords_Ac,
                                const double* r_Ac);
/* ---- Galerkin coarse graph (SURVEY.md section 8 row f3) -------------------------------------- */
typedef struct ge_galerkin_stats {
  double device_ms;        /* kernels + the row-length round trip (CUDA events) */
  double total_ms;         /* whole call, host layout and copies included */
  int64_t kernel_launches;
  int64_t segments_shared; /* coarse rows sorted in shared memory */
  int64_t segments_global; /* coarse rows with more than 4096 fine entries (global scratch) */
  int64_t nnz_out;
} ge_galerkin_stats;
/* A_c = P_T * A * P_T^T, the step examples/embedder.cpp:213-216 (and examples/embed.cpp:95-98)
 * runs before partition::embed: `As.push_back(P.Mult(As.back()).Mult(P.Transpose()))`.
 * A: n x n CSR (data may be NULL: unit weights); P_T: m x n aggregation, one entry per column,
 * row a lists the members of aggregate a (its data is ignored).  Output: m x m CSR with ascending
 * columns per row, diagonal entries included (the reference keeps them and counts them in the
 * degree).  c_indptr (m+1) is always filled and *nnz_out set; c_indices / c_data are filled when
 * capacity >= *nnz_out -- capacity = A->nnz always suffices -- otherwise GE_ERR_INVALID is
 * returned with *nnz_out set so the caller can retry.  Sums are accumulated in member order, then
 * CSR entry order (bit-reproducible; unit-weight graphs give integer sums in any order). */
ge_status ge_galerkin(ge_context* ctx, const ge_csr* A, const ge_csr* P_T, int32_t* c_indptr,
                      int32_t* c_indices, double* c_data, int64_t capacity, int64_t* nnz_out,
                      ge_galerkin_stats* stats /* may be NULL */);

/* ---- multilevel hierarchy on the device ------------------------------------------------------ */
/* Random-mate matching, level by level: the stand-in hierarchy generator of the project
 * (graphs.coarsen) made deterministic.  This is NOT the reference's partitioner
 * (src/partitioner.cpp:1550-1893); it is an additional way to go from a graph to the input of
 * ge_embed.  Each round, a counter-based hash H(tag, v) of (seed, level, round) splits the vertices
 * into heads and tails; every tail picks the head neighbour with the largest w_ij / (k_i k_j)
 * (k = weighted degree, self-loop included), ties to the smaller hash then the smaller id; when
 * more tails found a head than the level still needs, the ones with the smallest H(1, i) merge.
 * The round's graph is contracted with the Galerkin product of ge_galerkin.  A level ends at
 * max(floor(coarsening_factor * n), min_coarse) vertices or when no tail finds a head; the
 * hierarchy ends after max_levels levels, at min_coarse vertices, or at a level that merged nothing.
 * The result is a pure function of (A, options); tests/coarsen_restatement.py restates it on
 * the host. */
typedef struct ge_coarsen_options {
  double coarsening_factor; /* 0.25; in (0, 1] */
  int32_t min_coarse;       /* 64; >= 1 */
  int32_t max_levels;       /* 32; >= 0 */
  uint32_t seed;            /* 0; every value, 0 included, is an ordinary seed */
} ge_coarsen_options;

typedef struct ge_coarsen_stats {
  double total_ms;         /* whole call: upload, every round, download of the levels */
  double device_ms;        /* CUDA events from the first kernel to the end of the download */
  int64_t rounds;          /* matching rounds, all levels */
  int64_t kernel_launches; /* one CUB sort / select call counts as one launch */
} ge_coarsen_stats;

typedef struct ge_hierarchy ge_hierarchy; /* host copy of the levels, owned by the handle */

void ge_coarsen_options_default(ge_coarsen_options* opt);
/* A: n x n CSR (data NULL = unit weights), finite weights.  On a multi-device context the call runs
 * on the first device.  *out receives a new handle (free it with ge_hierarchy_destroy); stats may
 * be NULL. */
ge_status ge_coarsen(ge_context* ctx, const ge_csr* A, const ge_coarsen_options* opt,
                     ge_hierarchy** out, ge_coarsen_stats* stats);
/* Number of levels L: the hierarchy has graphs As[0..L] (As[0] = A) and aggregations P_T[0..L-1]. */
int32_t ge_hierarchy_levels(const ge_hierarchy* h);
/* View of As[l], l = 1..L: columns ascending per row, diagonal entries included. */
ge_status ge_hierarchy_graph(const ge_hierarchy* h, int32_t l, ge_csr* out);
/* View of P_T[l], l = 0..L-1 (As[l+1].rows x As[l].rows, members ascending per row, unit data). */
ge_status ge_hierarchy_aggregation(const ge_hierarchy* h, int32_t l, ge_csr* out);
void ge_hierarchy_destroy(ge_hierarchy* h);

/* ---- raw graph -> coordinates on the device ----------------------------------------------------- */
/* examples/embedder.cpp:156 (largestComponent, :35-93) on the device: the largest weakly connected
 * component of A (every entry (i, j) links i and j), ties to the component with the smallest vertex.
 * vertices: A->rows capacity, original ids of the kept vertices, ascending; the subgraph is
 * A[vertices][:, vertices] with A's entry order (columns renumbered, so still ascending when A's
 * were).  c_indptr: A->rows + 1 capacity.  Capacity rule as ge_galerkin (A->nnz suffices).
 * c_data receives ones when A->data is NULL.  components (may be NULL): the number of components.
 * On a multi-device context the call runs on the first device. */
ge_status ge_largest_component(ge_context* ctx, const ge_csr* A, int32_t* vertices, int32_t* n_out,
                               int32_t* c_indptr, int32_t* c_indices, double* c_data,
                               int64_t capacity, int64_t* nnz_out, int64_t* components);

typedef struct ge_layout_stats {
  double total_ms;      /* whole call */
  double components_ms; /* CUDA events around the component step; 0 when skipped */
  double coarsen_ms;    /* CUDA events around the hierarchy build */
  double embed_ms;      /* host clock: download of the O(n) arrays and the embed */
  int64_t components;   /* components of A; 0 when the step is skipped */
  int32_t levels;       /* L of the hierarchy */
  double h2d_bytes, d2h_bytes;
  int64_t kernel_launches;
} ge_layout_stats;

/* Graph -> coordinates: [largest component] -> ge_coarsen's hierarchy -> ge_embed, on the device.
 * A is uploaded once and the coordinates come down once; of the hierarchy only every P_T, the row
 * pointers of every level and the coarsest graph cross PCIe.  With eopt->seed != 0 the result equals
 * ge_largest_component, then ge_coarsen, then ge_embed with the same options, bit for bit
 * (largest_component = 0 skips the first step); so do the error statuses.
 * copt / eopt NULL: defaults.  coords_out: A->rows x dim capacity, first *n_out rows written;
 * vertices_out (A->rows capacity, may be NULL): original id of each written row.  stats may be NULL.
 * On a multi-device context the component step and the coarsening run on the first device and the
 * embed behaves as ge_embed does on that context. */
ge_status ge_layout_graph(ge_context* ctx, const ge_csr* A, int dim, int32_t largest_component,
                          const ge_coarsen_options* copt, const ge_embed_options* eopt,
                          double* coords_out, int32_t* vertices_out, int32_t* n_out,
                          ge_layout_stats* stats);

/* ---- edge list -> graph on the device ------------------------------------------------------------ */
/* The CSR that linalgcpp's CooMatrix (host/compat/sparsematrix.hpp) returns from ToSparse() after,
 * for every edge e in order: skip it if src == dst and keep_self_loops == 0; Add(src, dst, w);
 * then, if symmetrize and src != dst, Add(dst, src, w) (a kept self-loop is added once).  So the
 * columns of each row are strictly ascending, duplicates are summed in that order starting from
 * +0.0, and entries whose sum is zero are kept.  unit_weights = 1: every stored entry is 1.0 (with
 * symmetrize = 1 and self-loops dropped, the canonical graph of graphs._finish). */
typedef struct ge_edges_options {
  int32_t symmetrize;      /* 1 */
  int32_t keep_self_loops; /* 0 */
  int32_t unit_weights;    /* 0 */
} ge_edges_options;

typedef struct ge_edges_stats {
  double total_ms;            /* whole call */
  double device_ms;           /* CUDA events from the first kernel to the end of the build */
  int64_t nnz;                /* entries of the graph */
  int64_t self_loops_dropped; /* edges skipped as self-loops */
  int64_t duplicates_merged;  /* contributions added into an earlier one of the same entry */
  int64_t kernel_launches;    /* one CUB sort counts as one launch */
} ge_edges_stats;

void ge_edges_options_default(ge_edges_options* opt);
/* n vertices, E edges src[e] -> dst[e] (int32 ids in [0, n)) with weights w[e] (NULL: 1.0; when
 * given, every weight must be finite, also with unit_weights).  opt NULL: defaults.  c_indptr:
 * n + 1 entries, always filled, and *nnz_out always set; c_indices / c_data are filled when
 * capacity >= *nnz_out -- capacity = 2E always suffices -- otherwise GE_ERR_INVALID is returned with
 * *nnz_out set so the caller can retry.  GE_ERR_INVALID for an id outside [0, n), a non-finite
 * weight, n < 0, E < 0, or more contributions than int32 row pointers can address (E > 2^30 - 1 when
 * symmetrising, E > 2^31 - 1 otherwise).  On a multi-device context the call runs on the first
 * device.  stats may be NULL. */
ge_status ge_graph_from_edges(ge_context* ctx, int32_t n, int64_t E, const int32_t* src, const int32_t* dst,
                              const double* w, const ge_edges_options* opt, int32_t* c_indptr,
                              int32_t* c_indices, double* c_data, int64_t capacity, int64_t* nnz_out,
                              ge_edges_stats* stats);
/* Edge list -> coordinates: ge_graph_from_edges, then the body of ge_layout_graph on the graph it
 * built, which stays on the device.  Only the edge arrays go up.  With eopt->seed != 0 the result
 * (coordinates, vertices_out, n_out, status) equals ge_graph_from_edges followed by ge_layout_graph
 * with the same options, bit for bit.  coords_out: n x dim capacity; vertices_out: n capacity (may
 * be NULL).  edges_stats covers the graph build; layout_stats covers the whole call, the edge upload
 * included.  Either may be NULL. */
ge_status ge_layout_edges(ge_context* ctx, int32_t n, int64_t E, const int32_t* src, const int32_t* dst,
                          const double* w, const ge_edges_options* edges_opt, int dim,
                          int32_t largest_component, const ge_coarsen_options* copt,
                          const ge_embed_options* eopt, double* coords_out, int32_t* vertices_out,
                          int32_t* n_out, ge_edges_stats* edges_stats, ge_layout_stats* layout_stats);

/* The reference's random stream: count draws of uniform_real_distribution<double>(-1,1) over
 * std::mt19937(seed) (include/forceatlas.hpp:104-108). */
void ge_reference_uniform(uint32_t seed, int64_t count, double* out);

/* ---- device-resident flat solver (bench / multi-GPU row-block sharding) ------------------ */
/* Owns rows [row_begin,row_end) of A; holds full coordinates (two buffers, SoA [dim][ld]) and
 * the full vertex masses.  One iteration = repulsion + (attraction, gravity, step) for the
 * owned rows, written into the NEXT coordinate buffer; with more than one rank the caller
 * all-gathers that buffer (see ge_flat_plan_next_coords) before calling ge_flat_plan_swap. */
ge_status ge_flat_plan_create(ge_context* ctx, const ge_csr* A, int dim, const ge_params* p,
                              int32_t row_begin, int32_t row_end, ge_flat_plan** out);
void ge_flat_plan_destroy(ge_flat_plan* plan);
/* Rank `rank` of a `world`-rank SYMMETRIC solve of the same loop (include/forceatlas.hpp:151-167
 * adds an exactly antisymmetric term for (i,j) and (j,i), so each unordered pair is evaluated
 * once, on one rank).  The rank owns the row block [rank*ld/world, (rank+1)*ld/world) (clipped to
 * n) for attraction + step, and an equal share of the unordered pairs for repulsion, whose sums it
 * accumulates over the FULL length [dim][ld].  Per iteration:
 *     ge_flat_plan_launch_repulsion            (pair sums of this rank's share)
 *     reduce-scatter (sum) of the pair sums    (caller: NCCL, per dimension, in place; the buffer
 *                                               is ge_flat_plan_pair_sums or the caller's own,
 *                                               bound with ge_flat_plan_bind_pair_sums)
 *     ge_flat_plan_launch_step                 (attraction, gravity, step for the owned rows)
 *     all-gather of the next coordinates, ge_flat_plan_swap   (as for row-block plans)
 * world == 1 is the plan ge_flat_plan_create makes for all rows.  GE_ERR_INVALID if the graph is
 * too small for the symmetric sweep (n < 32768) or its scratch would not fit. */
ge_status ge_flat_plan_create_symmetric(ge_context* ctx, const ge_csr* A, int dim, const ge_params* p,
                                        int32_t rank, int32_t world, ge_flat_plan** out);
/* Host-only: the units of rank `rank`'s share of the symmetric sweep over a padded length ld (a
 * multiple of 256) as quintuples (row0, row1, first column tile, tile count, first symmetric
 * tile); returns the number of quintuples (at most `capacity` are written), -1 on bad arguments. */
int32_t ge_flat_symmetric_share(int64_t ld, int32_t rank, int32_t world, int32_t capacity,
                                int32_t* blocks);
/* Host-only: the same for pass `pass` of `npass` column-panel passes of that share (large graphs cut
 * the sweep into passes that reuse one column-side scratch buffer). */
int32_t ge_flat_symmetric_pass_share(int64_t ld, int32_t rank, int32_t world, int32_t npass, int32_t pass,
                                     int32_t capacity, int32_t* blocks);
/* Host-only: how ge_embed on an ndev-device context cuts one level into contiguous aggregate ranges
 * of (nearly) equal cost (s^2 ordered pairs + the members' CSR entries): cuts[0..ndev], cuts[0] = 0,
 * cuts[ndev] = P_T->rows. */
ge_status ge_embed_aggregate_ranges(const ge_csr* A, const ge_csr* P_T, int32_t ndev, int32_t* cuts,
                                    double* pairs_per_iteration);
/* Host-only: the device (0 .. ndev-1) that solves each aggregate of a level in ge_embed on an
 * ndev-device context: heavy aggregates largest-first on the least loaded device, light ones filled
 * in index order.  owner: P_T->rows entries. */
ge_status ge_embed_aggregate_owners(const ge_csr* A, const ge_csr* P_T, int32_t ndev, int32_t* owner,
                                    double* pairs_per_iteration);
/* 1 if the plan evaluates unordered pairs (ge_flat_plan_create chooses this for whole-graph plans
 * on large graphs), 0 for the ordered row-block sweep. */
int32_t ge_flat_plan_is_symmetric(const ge_flat_plan* plan);
/* Symmetric plans: the [dim][ld] device buffer of raw pair sums (force = sum * c_i * repel). */
void* ge_flat_plan_pair_sums(ge_flat_plan* plan);
ge_status ge_flat_plan_bind_pair_sums(ge_flat_plan* plan, void* dev_buf);
/* The two halves of ge_flat_plan_launch_iteration. */
ge_status ge_flat_plan_launch_repulsion(ge_flat_plan* plan);
ge_status ge_flat_plan_launch_step(ge_flat_plan* plan);
/* Leading dimension (elements) of the SoA coordinate buffers and element size in bytes. */
int64_t ge_flat_plan_ld(const ge_flat_plan* plan);
int32_t ge_flat_plan_elem_size(const ge_flat_plan* plan);
/* Use caller-provided device memory (2 buffers of dim*ld elements) for the coordinates. */
ge_status ge_flat_plan_bind_coords(ge_flat_plan* plan, void* dev_buf0, void* dev_buf1);
ge_status ge_flat_plan_upload_coords(ge_flat_plan* plan, const double* coords);   /* n x dim */
ge_status ge_flat_plan_download_coords(ge_flat_plan* plan, double* coords);       /* n x dim */
ge_status ge_flat_plan_download_forces(ge_flat_plan* plan, double* forces);       /* owned rows x dim */
/* Device pointers of the current / next coordinate buffer (SoA [dim][ld]).  Row order is the
 * caller's for plans that own a row block of a multi-rank run; a plan that owns every row of a
 * large graph may renumber the vertices internally (breadth-first, for gather locality) and
 * restores the caller's order only in upload / download. */
void* ge_flat_plan_cur_coords(ge_flat_plan* plan);
void* ge_flat_plan_next_coords(ge_flat_plan* plan);
/* Launch the kernels of one iteration for the owned rows (asynchronous on the context stream). */
ge_status ge_flat_plan_launch_iteration(ge_flat_plan* plan);
/* Make the next buffer current (call after the all-gather, if any, was enqueued). */
void ge_flat_plan_swap(ge_flat_plan* plan);
/* Convenience: `iters` x (launch_iteration + swap), single rank. */
ge_status ge_flat_plan_iterate(ge_flat_plan* plan, int iters);
ge_status ge_flat_plan_sync(ge_flat_plan* plan);
/* Measurement hook: which kernels launch_iteration runs (bit 0 = repulsion, bit 1 = attraction +
 * step; default 3).  Lets the HBM-bound attraction kernel be timed alone on graphs whose
 * all-pairs repulsion would take seconds. */
void ge_flat_plan_select_kernels(ge_flat_plan* plan, int mask);
/* Per-kernel device time.  enable != 0 brackets each launch with CUDA events on the launching
 * stream; get returns the accumulated milliseconds and launch counts since the last reset. */
void ge_flat_plan_profile(ge_flat_plan* plan, int enable);
ge_status ge_flat_plan_profile_get(ge_flat_plan* plan, double* repulsion_ms, int64_t* repulsion_launches,
                                   double* attract_step_ms, int64_t* attract_step_launches);

#ifdef __cplusplus
}
#endif
#endif /* GRAPH_EMBED_B200_H */

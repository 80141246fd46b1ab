"""Synthetic inputs for the ForceAtlas hot path: graphs of the shapes BASELINE.json names and
the multilevel hierarchies (P_T per level + Galerkin coarse graphs) that `partition::embed`
consumes.

The reference builds its hierarchies with `partition::partition` (src/partitioner.cpp:1550-1893)
and the Galerkin products at examples/embedder.cpp:213-216; both are host-side INPUT to the hot
path and out of scope (SURVEY.md section 8).  `coarsen` below is a stand-in input generator
(random-mate star contraction), not a re-implementation of that partitioner; fixtures in
tests/golden/ carry hierarchies produced by the reference's own partitioner where index-for-index
agreement with it matters.
"""
import numpy as np
import scipy.sparse as sp
from scipy.sparse.csgraph import connected_components


def _finish(rows, cols, n, weights=None):
    """Symmetrise, de-duplicate, drop self-loops, unit weights; canonical int32/float64 CSR."""
    keep = rows != cols
    rows, cols = rows[keep], cols[keep]
    r = np.concatenate([rows, cols])
    c = np.concatenate([cols, rows])
    A = sp.csr_matrix((np.ones(r.shape[0]), (r, c)), shape=(n, n))
    A.sum_duplicates()
    A.data[:] = 1.0
    return canonical(A)


def canonical(A):
    A = sp.csr_matrix(A)
    A.sort_indices()
    return sp.csr_matrix((A.data.astype(np.float64), A.indices.astype(np.int32),
                          A.indptr.astype(np.int32)), shape=A.shape)


def largest_component(A):
    """What examples/embedder.cpp:156 (largestComponent, :35-93) does before partitioning."""
    ncomp, label = connected_components(A, directed=False)
    if ncomp == 1:
        return A
    big = np.argmax(np.bincount(label))
    idx = np.flatnonzero(label == big)
    return canonical(A[idx][:, idx])


def grid2d(nx, ny):
    """nx x ny 4-neighbour grid, unit weights, no diagonal (BASELINE config 1: 100 x 100)."""
    ids = np.arange(nx * ny).reshape(nx, ny)
    rows = np.concatenate([ids[:-1, :].ravel(), ids[:, :-1].ravel()])
    cols = np.concatenate([ids[1:, :].ravel(), ids[:, 1:].ravel()])
    return _finish(rows, cols, nx * ny)


def _largest(A, largest):
    return largest_component(A) if largest else A


def rgg_edges(n, avg_degree=10.0, dim=2, seed=12345):
    """The pairs (rows, cols, n) of a random geometric graph on U[0,1]^dim, each unordered pair once,
    radius chosen for the requested average degree."""
    from scipy.spatial import cKDTree
    rng = np.random.default_rng(seed)
    pts = rng.random((n, dim))
    if dim == 2:
        r = np.sqrt(avg_degree / (np.pi * n))
    else:
        r = (avg_degree / (4.0 / 3.0 * np.pi * n)) ** (1.0 / 3.0)
    pairs = cKDTree(pts).query_pairs(r, output_type="ndarray")
    return pairs[:, 0], pairs[:, 1], n


def rgg(n, avg_degree=10.0, dim=2, seed=12345, largest=True):
    """Random geometric graph on U[0,1]^dim, radius chosen for the requested average degree
    (BASELINE config 2: n = 100 000, avg degree 10, d = 2); largest component (largest=False: the
    raw graph, every component)."""
    return _largest(_finish(*rgg_edges(n, avg_degree, dim, seed)), largest)


def rmat_edges(scale, edge_factor=16, abc=(0.57, 0.19, 0.19), seed=12345):
    """The raw R-MAT edges (rows, cols, n): edge_factor * 2^scale pairs, duplicates and self-loops
    included."""
    rng = np.random.default_rng(seed)
    n = 1 << scale
    ne = edge_factor * n
    a, b, c = abc
    rows = np.zeros(ne, dtype=np.int64)
    cols = np.zeros(ne, dtype=np.int64)
    for _ in range(scale):
        u = rng.random(ne)
        rbit = u >= a + b
        cbit = ((u >= a) & (u < a + b)) | (u >= a + b + c)
        rows = (rows << 1) | rbit
        cols = (cols << 1) | cbit
    return rows, cols, n


def rmat(scale, edge_factor=16, abc=(0.57, 0.19, 0.19), seed=12345, largest=True):
    """R-MAT (BASELINE config 3: scale 20, edge factor 16); symmetrised, de-duplicated,
    self-loops dropped, unit weights, largest component (largest=False: the raw graph)."""
    return _largest(_finish(*rmat_edges(scale, edge_factor, abc, seed)), largest)


def delaunay3d_edges(n, seed=12345):
    """The edges (rows, cols, n) of the Delaunay tetrahedralisation of n points in U[0,1]^3: six per
    tetrahedron, so an edge shared by k tetrahedra appears k times."""
    from scipy.spatial import Delaunay
    rng = np.random.default_rng(seed)
    tets = Delaunay(rng.random((n, 3))).simplices
    pr = [(0, 1), (0, 2), (0, 3), (1, 2), (1, 3), (2, 3)]
    rows = np.concatenate([tets[:, i] for i, _ in pr])
    cols = np.concatenate([tets[:, j] for _, j in pr])
    return rows, cols, n


def delaunay3d(n, seed=12345, largest=True):
    """Edges of the Delaunay tetrahedralisation of n points in U[0,1]^3 (BASELINE config 5);
    largest component (largest=False: the raw graph)."""
    return _largest(_finish(*delaunay3d_edges(n, seed)), largest)


def aggregation_matrix(agg, m):
    """P_T (m x n, unit entries, members ascending per row) from a vertex->aggregate map; the
    shape `interpolationMatrix` emits (src/partitioner.cpp:29-65)."""
    n = agg.shape[0]
    order = np.argsort(agg, kind="stable").astype(np.int32)
    indptr = np.zeros(m + 1, dtype=np.int32)
    np.cumsum(np.bincount(agg, minlength=m), out=indptr[1:])
    return sp.csr_matrix((np.ones(n), order, indptr), shape=(m, n))


def galerkin(A, P_T):
    """A_{l+1} = P_T A P_T^T (examples/embedder.cpp:213-216).  Keeps the diagonal (intra-aggregate
    weight), which the kernels see as self-loops (SURVEY quirk Q5)."""
    return canonical(P_T @ A @ P_T.T)


def _matching_round(S, rng, max_merges=None):
    """One random-mate contraction round on the coarse graph S: vertices are split at random into
    heads and tails; every tail merges into the head neighbour with the best affinity
    w_ij / (k_i k_j) (several tails may pick the same head, so hubs grow stars, as the reference's
    hierarchies on power-law graphs do).  O(nnz); about 45 % of the vertices disappear per round."""
    m = S.shape[0]
    k = np.asarray(S.sum(axis=1)).ravel()
    k = np.where(k > 0, k, 1.0)
    rows = np.repeat(np.arange(m), np.diff(S.indptr))
    cols = S.indices
    head = rng.random(m) < 0.5
    ok = (rows != cols) & ~head[rows] & head[cols]
    rows, cols = rows[ok], cols[ok]
    if rows.size == 0:
        return None
    score = S.data[ok] / (k[rows] * k[cols]) * (1.0 + 1e-6 * rng.random(rows.size))
    starts = np.flatnonzero(np.r_[True, rows[1:] != rows[:-1]])       # CSR order: rows are sorted
    best = np.maximum.reduceat(score, starts)
    is_best = score == np.repeat(best, np.diff(np.r_[starts, rows.size]))
    sel = np.flatnonzero(is_best)
    tails, first = np.unique(rows[sel], return_index=True)
    if max_merges is not None and tails.size > max_merges:   # stop exactly at the level's target size
        keep = np.sort(rng.choice(tails.size, size=max_merges, replace=False))
        tails, first = tails[keep], first[keep]
    label = np.arange(m)
    label[tails] = cols[sel[first]]
    uniq, new = np.unique(label, return_inverse=True)
    return new.astype(np.int64), uniq.size


def coarsen(A, coarsening_factor=0.25, min_coarse=64, max_levels=32, seed=0):
    """Hierarchy generator: returns (As, P_Ts) with As[l+1] = P_Ts[l] As[l] P_Ts[l]^T and
    len(As) == len(P_Ts) + 1, each level reducing the vertex count to coarsening_factor x the
    previous one (a ratio M/N, like src/partitioner.cpp:1797) but never below min_coarse, which
    is the size of the coarsest level (the reference's hierarchies end at ~30-100 vertices)."""
    rng = np.random.default_rng(seed)
    As, P_Ts = [canonical(A)], []
    while As[-1].shape[0] > min_coarse and len(P_Ts) < max_levels:
        N = As[-1].shape[0]
        agg, M, S = np.arange(N), N, As[-1]
        target = max(int(np.floor(coarsening_factor * N)), min_coarse)
        while M > target:
            res = _matching_round(S, rng, max_merges=M - target)
            if res is None:
                break
            new, M2 = res
            agg, M = new[agg], M2
            Q = aggregation_matrix(new, M2)
            S = canonical(Q @ S @ Q.T)
        if M == N:
            break
        P_T = aggregation_matrix(agg, M)
        P_Ts.append(sp.csr_matrix((P_T.data, P_T.indices.astype(np.int32),
                                   P_T.indptr.astype(np.int32)), shape=P_T.shape))
        As.append(galerkin(As[-1], P_Ts[-1]))
    return As, P_Ts


def hierarchy_from(A, P_Ts):
    """As for a given list of P_T (e.g. one produced by the reference partitioner)."""
    As = [canonical(A)]
    for P in P_Ts:
        As.append(galerkin(As[-1], P))
    return As


def level_stats(As, P_Ts):
    """Per-level n, nnz, aggregate count / max size and ordered intra-aggregate pairs."""
    out = []
    for l, P in enumerate(P_Ts):
        s = np.diff(P.indptr).astype(np.int64)
        out.append(dict(level=l, n=As[l].shape[0], nnz=As[l].nnz, aggregates=P.shape[0],
                        max_size=int(s.max()), pairs=int((s * (s - 1)).sum())))
    n = As[-1].shape[0]
    out.append(dict(level=len(P_Ts), n=n, nnz=As[-1].nnz, aggregates=0, max_size=0,
                    pairs=n * (n - 1)))
    return out

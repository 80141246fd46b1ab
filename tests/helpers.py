"""Shared test helpers: golden loaders and tolerance metrics."""
import lzma
import os

import numpy as np
import scipy.sparse as sp

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# Tolerances stated by BASELINE.json's north_star for per-iteration force vectors.
TOL_F64 = 1e-10
TOL_F32 = 1e-4


def load_flat_golden():
    z = np.load(os.path.join(GOLDEN, "flat_grid12.npz"))
    n = len(z["indptr"]) - 1
    A = sp.csr_matrix((z["data"], z["indices"], z["indptr"]), shape=(n, n))
    return A, z


def load_hier_golden():
    z = np.load(os.path.join(GOLDEN, "hier_grid30.npz"))
    L = int(z["L"])
    As, Ps = [], []
    for l in range(L + 1):
        n = len(z["A%d_indptr" % l]) - 1
        As.append(sp.csr_matrix((z["A%d_data" % l], z["A%d_indices" % l], z["A%d_indptr" % l]), shape=(n, n)))
    for l in range(L):
        m = len(z["P%d_indptr" % l]) - 1
        idx = z["P%d_indices" % l]
        Ps.append(sp.csr_matrix((np.ones(len(idx)), idx, z["P%d_indptr" % l]), shape=(m, As[l].shape[0])))
    return As, Ps, z


def load_config1_golden(graphs):
    """BASELINE config 1 (grid 100x100, coarsening 0.25): hierarchy from the reference's own
    partitioner + the compiled reference's embed() output for seed 3."""
    z = np.load(os.path.join(GOLDEN, "config1_grid100.npz"))
    A = graphs.grid2d(100, 100)
    Ps, n = [], A.shape[0]
    for l in range(int(z["L"])):
        ptr, idx = z["P%d_indptr" % l], z["P%d_indices" % l]
        Ps.append(sp.csr_matrix((np.ones(len(idx)), idx, ptr), shape=(len(ptr) - 1, n)))
        n = len(ptr) - 1
    return graphs.hierarchy_from(A, Ps), Ps, z


def force_error(F, F_ref, scale):
    """Per-vertex |F - F_ref|_2 divided by the conditioning scale the oracle reports (the sum of
    the norms of the individual terms that were added into that vertex's force)."""
    return np.linalg.norm(F - F_ref, axis=1) / np.maximum(scale, 1e-300)


def layout_stats(A, x):
    """Edge-length mean / coefficient of variation and a sampled normalised stress."""
    coo = A.tocoo()
    keep = coo.row < coo.col
    el = np.linalg.norm(x[coo.row[keep]] - x[coo.col[keep]], axis=1)
    rng = np.random.default_rng(0)
    n = A.shape[0]
    i, j = rng.integers(0, n, 4000), rng.integers(0, n, 4000)
    dist = np.linalg.norm(x[i] - x[j], axis=1)
    extent = np.linalg.norm(x - x.mean(0), axis=1).max()
    return dict(edge_mean=el.mean() / extent, edge_cv=el.std() / el.mean(),
                pair_mean=dist.mean() / extent)


def load_galerkin_golden(graphs):
    """Galerkin products of the grid-30 hierarchy minted from the compiled reference driver."""
    z = np.load(os.path.join(GOLDEN, "galerkin_grid30.npz"))
    A = graphs.canonical(graphs.grid2d(30, 30))
    Ps, Cs, n = [], [], A.shape[0]
    for l in range(int(z["L"])):
        ptr, idx = z["P%d_indptr" % l], z["P%d_indices" % l]
        m = len(ptr) - 1
        Ps.append(sp.csr_matrix((np.ones(len(idx)), idx, ptr), shape=(m, n)))
        Cs.append(sp.csr_matrix((z["C%d_data" % l], z["C%d_indices" % l], z["C%d_indptr" % l]), shape=(m, m)))
        n = m
    return A, Ps, Cs, z


_REFHIER_CACHE = {}


def pack_i32(a):
    """An int32 array as an xz-compressed byte array (one npz member)."""
    raw = np.ascontiguousarray(a, dtype=np.int32).tobytes()
    return np.frombuffer(lzma.compress(raw, preset=9 | lzma.PRESET_EXTREME), dtype=np.uint8)


def unpack_i32(b):
    return np.frombuffer(lzma.decompress(b.tobytes()), dtype=np.int32)


def encode_aggregates(A, P_T):
    """The vertex->aggregate map of P_T (members ascending per row), stated relative to the graph A
    it partitions, which stores in a fraction of the map's size.  Every aggregate of the reference
    partitioner is connected in A; its smallest member is its root.  Each other vertex links to a
    neighbour in the same aggregate one step closer to the root (breadth-first depth), named by
    its 1-based position in the vertex's row of A; a root links to 0.  root_ids lists the aggregate
    ids of the roots in ascending vertex order.  -> (link, root_ids), both int32"""
    n, m = A.shape[0], P_T.shape[0]
    agg = np.empty(n, dtype=np.int64)
    agg[P_T.indices] = np.repeat(np.arange(m), np.diff(P_T.indptr))
    root = P_T.indices[P_T.indptr[:-1]]
    coo = A.tocoo()
    same = (agg[coo.row] == agg[coo.col]) & (coo.row != coo.col)
    r, c = coo.row[same], coo.col[same]
    pos = np.flatnonzero(same) - A.indptr[r] + 1
    depth = np.full(n, -1, dtype=np.int64)
    depth[root] = 0
    d = 0
    while True:
        f = (depth[c] == d) & (depth[r] < 0)
        if not f.any():
            break
        depth[r[f]] = d + 1
        d += 1
    assert (depth >= 0).all(), "an aggregate is not connected in its graph"
    ok = depth[c] == depth[r] - 1
    r, pos = r[ok], pos[ok]
    o = np.lexsort((pos, r))
    r, pos = r[o], pos[o]
    first = np.unique(r, return_index=True)[1]
    link = np.zeros(n, dtype=np.int32)
    link[r[first]] = pos[first]
    return link, np.argsort(root).astype(np.int32)


def decode_aggregates(A, link, root_ids):
    """Inverse of encode_aggregates -> the vertex->aggregate map (int32)."""
    n = A.shape[0]
    parent = np.arange(n)
    up = link > 0
    parent[up] = A.indices[A.indptr[:-1][up] + link[up] - 1]
    while True:  # pointer jumping: every vertex ends on its root
        nxt = parent[parent]
        if np.array_equal(nxt, parent):
            break
        parent = nxt
    roots = np.flatnonzero(link == 0)
    assert roots.shape == root_ids.shape
    agg = np.empty(n, dtype=np.int32)
    agg[roots] = root_ids
    return agg[parent]


def load_ref_hierarchy(graphs, name):
    """A hierarchy produced by the REFERENCE's own partitioner (src/partitioner.cpp:1550-1893, call
    shape of examples/embedder.cpp:187) on a synthetic graph of a BASELINE config, cached by
    tests/golden/make_ref_hierarchy.py as the vertex->aggregate map of every level, stored relative
    to that level's graph (encode_aggregates).  The graph is regenerated from its seed and checked
    against the stored digest; the coarse graphs are the Galerkin products
    examples/embedder.cpp:213-216 forms.  -> (As, P_Ts, meta)"""
    import hashlib
    if name in _REFHIER_CACHE:
        return _REFHIER_CACHE[name]
    z = np.load(os.path.join(GOLDEN, "refhier_%s.npz" % name))
    kind, arg, seed = str(z["kind"]), int(z["arg"]), int(z["seed"])
    if kind == "rmat":
        A = graphs.rmat(arg, 16, seed=seed)
    elif kind == "delaunay":
        A = graphs.delaunay3d(arg, seed=seed)
    elif kind == "rgg":
        A = graphs.rgg(arg, 10.0, seed=seed)
    else:
        raise ValueError(kind)
    h = hashlib.sha256()
    h.update(np.ascontiguousarray(A.indptr).tobytes())
    h.update(np.ascontiguousarray(A.indices).tobytes())
    assert h.hexdigest() == str(z["digest"]), "the generator no longer reproduces the cached graph"
    As, Ps = [graphs.canonical(A)], []
    for l in range(int(z["L"])):
        link, root_ids = unpack_i32(z["link%d" % l]), unpack_i32(z["roots%d" % l])
        assert link.shape[0] == As[-1].shape[0]
        P = graphs.aggregation_matrix(decode_aggregates(As[-1], link, root_ids), root_ids.shape[0])
        Ps.append(sp.csr_matrix((P.data, P.indices.astype(np.int32), P.indptr.astype(np.int32)), shape=P.shape))
        As.append(graphs.galerkin(As[-1], Ps[-1]))
    meta = dict(kind=kind, arg=arg, seed=seed, cf=float(z["cf"]),
                partition_seconds=float(z["partition_seconds"]))
    _REFHIER_CACHE[name] = (As, Ps, meta)
    return As, Ps, meta

"""ge_largest_component equals graphs.largest_component (scipy) exactly, and ge_layout_graph equals the
composed calls ge_largest_component -> ge_coarsen -> ge_embed bit for bit while no level's entries cross
PCIe."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp
from scipy.sparse.csgraph import connected_components

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bits(x):
    return np.ascontiguousarray(x, np.float64).view(np.uint64)


def _same(X, Y):
    assert X.shape == Y.shape
    assert np.array_equal(X.indptr, Y.indptr) and np.array_equal(X.indices, Y.indices)
    assert np.array_equal(_bits(X.data), _bits(Y.data))


def _disconnected(graphs):
    parts = [graphs.grid2d(40, 40), sp.csr_matrix((50, 50)), graphs.rgg(5000, 8.0, seed=4),
             graphs.grid2d(3, 1)]
    return graphs.canonical(sp.block_diag(parts))


def _permuted_path(graphs, n=1_000_000):
    """A path whose vertex ids are shuffled: chains of a million hooks in no particular order."""
    p = np.random.default_rng(7).permutation(n)
    r, c = p[:-1], p[1:]
    return graphs.canonical(sp.coo_matrix((np.ones(2 * (n - 1)), (np.r_[r, c], np.r_[c, r])), shape=(n, n)))


def _two_equal(graphs):
    G = graphs.grid2d(30, 30)
    return graphs.canonical(sp.block_diag([sp.csr_matrix((3, 3)), G, graphs.grid2d(10, 10), G]))


def _largest_not_first(graphs):
    return graphs.canonical(sp.block_diag([graphs.grid2d(5, 5), sp.csr_matrix((4, 4)), graphs.grid2d(60, 60)]))


def _real_weights(graphs):
    A = graphs.rgg(30000, 3.5, seed=9, largest=False)
    W = sp.triu(A, 1).tocsr()
    W.data = np.random.default_rng(2).random(W.nnz) * 3.0 + 0.01
    return graphs.canonical(W + W.T)


def _asymmetric(graphs):
    """Only the upper triangle of a disconnected graph: the components are weak ones."""
    return graphs.canonical(sp.triu(graphs.rgg(50000, 2.5, seed=3, largest=False), 1))


def _hub_graph(graphs):
    A = graphs.rgg(20000, 10.0, seed=8)
    n = A.shape[0]
    nb = np.random.default_rng(3).choice(n, 6000, replace=False)
    hub = np.full(nb.size, n)
    B = sp.coo_matrix((np.ones(2 * nb.size), (np.r_[hub, nb], np.r_[nb, hub])), shape=(n + 1, n + 1))
    return graphs.canonical(sp.bmat([[A, None], [None, sp.csr_matrix((1, 1))]]) + B)


CASES = {
    "rmat16_raw": lambda g: g.rmat(16, 16, seed=1, largest=False),
    "rmat18_raw": lambda g: g.rmat(18, 16, seed=2, largest=False),
    "rgg200k_sparse": lambda g: g.rgg(200_000, 3.0, seed=3, largest=False),
    "disconnected": _disconnected,
    "path1m": _permuted_path,
    "two_equal": _two_equal,
    "largest_not_first": _largest_not_first,
    "edgeless": lambda g: sp.csr_matrix((1000, 1000)),
    "connected": lambda g: g.grid2d(50, 50),
    "real_weights": _real_weights,
    "asymmetric": _asymmetric,
    "rgg100k_raw": lambda g: g.rgg(100_000, 10.0, seed=1, largest=False),
    "delaunay200k": lambda g: g.delaunay3d(200_000, seed=1),
    "hub": _hub_graph,
    "grid100": lambda g: g.grid2d(100, 100),
}
_GRAPHS = {}


def _graph(graphs, name):
    if name not in _GRAPHS:
        _GRAPHS[name] = graphs.canonical(CASES[name](graphs))
    return _GRAPHS[name]


@pytest.mark.parametrize("name", ["rmat16_raw", "rmat18_raw", "rgg200k_sparse", "disconnected", "path1m",
                                  "two_equal", "largest_not_first", "edgeless", "connected", "real_weights",
                                  "asymmetric"])
def test_largest_component_equals_scipy(ctx, graphs, name):
    A = _graph(graphs, name)
    B, vert, comps = ctx.largest_component(A)
    ncomp, label = connected_components(A, directed=False)
    assert comps == ncomp
    big = np.argmax(np.bincount(label))
    assert np.array_equal(vert, np.flatnonzero(label == big))
    _same(B, graphs.largest_component(A))
    if name == "edgeless":
        assert np.array_equal(vert, [0]) and B.shape == (1, 1)
    if name == "connected":
        assert comps == 1 and np.array_equal(vert, np.arange(A.shape[0]))
    if name == "two_equal":
        assert vert[0] == 3


def test_unit_weights_come_back_as_ones(ctx, capi, graphs):
    A = _graph(graphs, "disconnected")
    a = capi.CsrView(A, with_data=False)
    n, cap = A.shape[0], A.nnz
    vert, ptr, idx, val = np.zeros(n, np.int32), np.zeros(n + 1, np.int32), np.zeros(cap, np.int32), np.zeros(cap)
    k, nnz = C.c_int32(), C.c_int64()
    capi._check(capi.lib().ge_largest_component(ctx.h, a.ref(), capi._ptr(vert, capi._pi), C.byref(k),
                                                capi._ptr(ptr, capi._pi), capi._ptr(idx, capi._pi),
                                                capi._ptr(val, capi._pd), C.c_int64(cap), C.byref(nnz), None))
    ref = graphs.largest_component(A)
    assert k.value == ref.shape[0] and nnz.value == ref.nnz
    assert (val[:ref.nnz] == 1.0).all() and np.array_equal(idx[:ref.nnz], ref.indices)
    # too small a capacity: GE_ERR_INVALID, the size reported
    st = capi.lib().ge_largest_component(ctx.h, a.ref(), capi._ptr(vert, capi._pi), C.byref(k),
                                         capi._ptr(ptr, capi._pi), capi._ptr(idx, capi._pi),
                                         capi._ptr(val, capi._pd), C.c_int64(10), C.byref(nnz), None)
    assert st == capi.GE_ERR_INVALID and nnz.value == ref.nnz


def test_two_runs_are_identical(ctx, graphs):
    A = _graph(graphs, "rmat18_raw")
    B1, v1, c1 = ctx.largest_component(A)
    B2, v2, c2 = ctx.largest_component(A)
    _same(B1, B2)
    assert np.array_equal(v1, v2) and c1 == c2


def _composed(ctx, A, dim, cf, min_coarse, coarsen_seed, seed, precision, largest=True):
    h0, d0 = ctx.bytes_moved
    if largest:
        B, vert, _ = ctx.largest_component(A)
    else:
        B, vert = A, np.arange(A.shape[0], dtype=np.int32)
    As, Ps, _ = ctx.coarsen(B, cf, min_coarse, seed=coarsen_seed)
    x, _ = ctx.embed(As, Ps, dim, seed=seed, precision=precision)
    h1, d1 = ctx.bytes_moved
    return x, vert, As, Ps, (h1 - h0, d1 - d0)


def _fused(ctx, A, dim, cf, min_coarse, coarsen_seed, seed, precision, largest=True):
    h0, d0 = ctx.bytes_moved
    x, vert, st = ctx.layout(A, dim, cf, min_coarse, coarsen_seed=coarsen_seed, seed=seed, precision=precision,
                             largest_component=largest)
    h1, d1 = ctx.bytes_moved
    assert (st["h2d_bytes"], st["d2h_bytes"]) == (h1 - h0, d1 - d0)
    return x, vert, st


@pytest.mark.parametrize("name,dim,cf,precision,largest", [
    ("rmat16_raw", 3, 0.25, 0, True), ("rgg100k_raw", 2, 0.25, 0, True), ("delaunay200k", 3, 0.125, 0, True),
    ("real_weights", 2, 0.25, 0, True), ("hub", 3, 0.25, 0, True), ("rgg100k_raw", 2, 0.25, 1, True),
    ("grid100", 2, 0.25, 0, False),
])
def test_layout_equals_composed(ctx, capi, graphs, name, dim, cf, precision, largest):
    A = _graph(graphs, name)
    x, vert, st = _fused(ctx, A, dim, cf, 64, 5, 11, precision, largest)
    y, wert, As, Ps, _ = _composed(ctx, A, dim, cf, 64, 5, 11, precision, largest)
    assert np.array_equal(vert, wert)
    assert x.shape == y.shape and np.array_equal(_bits(x), _bits(y))
    assert np.isfinite(x).all()
    assert st["levels"] == len(Ps) and st["coarsen_ms"] > 0
    assert (st["components_ms"] > 0) == largest
    if largest:
        assert st["components"] == connected_components(A, directed=False)[0]


@pytest.mark.parametrize("name", ["rmat16_raw", "rmat18_raw"])
def test_no_level_entries_cross_pcie(ctx, graphs, name):
    A = _graph(graphs, name)
    _, _, st = _fused(ctx, A, 3, 0.25, 64, 1, 2, 0)
    _, _, As, Ps, (h2d, d2h) = _composed(ctx, A, 3, 0.25, 64, 1, 2, 0)
    E = sum(As[l].nnz * (4 + 8) for l in range(len(Ps)))  # index and weight arrays of levels 0..L-1
    assert len(Ps) >= 2 and E > 0
    assert h2d - st["h2d_bytes"] >= E
    assert d2h - st["d2h_bytes"] >= E


def test_multi_device_context(ctx, capi, graphs, monkeypatch):
    try:
        mc = capi.Context(devices=[0, 1])
    except capi.GeError as e:
        if e.status == capi.GE_ERR_INVALID and "more devices" in str(e):
            pytest.skip("box has fewer than 2 GPUs")
        raise
    monkeypatch.setenv("GE_SHARD_MIN_MPAIRS", "0.0001")  # shard every level of this small hierarchy
    A = _graph(graphs, "rmat16_raw")
    x2, v2, _ = _fused(mc, A, 3, 0.25, 64, 3, 4, 0)
    x1, v1, _ = _fused(ctx, A, 3, 0.25, 64, 3, 4, 0)
    y2, w2, _, _, _ = _composed(mc, A, 3, 0.25, 64, 3, 4, 0)
    assert np.array_equal(v2, v1) and np.array_equal(v2, w2)
    assert np.array_equal(_bits(x2), _bits(x1)) and np.array_equal(_bits(x2), _bits(y2))
    mc.close()


def test_errors(ctx, capi, graphs):
    def status(f):
        with pytest.raises(capi.GeError) as e:
            f()
        return e.value.status

    rect = sp.csr_matrix((3, 4))
    bad = sp.csr_matrix((np.ones(2), np.array([0, 7], dtype=np.int32), np.array([0, 1, 2], dtype=np.int32)),
                        shape=(2, 2))
    for A in (rect, bad):
        assert status(lambda: ctx.layout(A, 2, seed=1)) == capi.GE_ERR_INVALID
        assert status(lambda: ctx.largest_component(A)) == capi.GE_ERR_INVALID
    G = graphs.grid2d(20, 20)
    assert status(lambda: ctx.layout(G, 4, seed=1)) == capi.GE_ERR_INVALID
    As, Ps, _ = ctx.coarsen(G, 0.25, 64)
    assert status(lambda: ctx.embed(As, Ps, 4, seed=1)) == capi.GE_ERR_INVALID
    a = capi.CsrView(G)
    n = C.c_int32()
    assert capi.lib().ge_layout_graph(ctx.h, a.ref(), 2, 1, None, None, None, None, C.byref(n),
                                      None) == capi.GE_ERR_INVALID


def test_cpp_dropin_demo_layout(capi):
    exe = os.path.join(ROOT, "graph-embed_b200", "lib", "ge_dropin_demo")
    if not os.path.exists(exe):
        from graph_embed_b200 import build
        build.build_all()
    r = subprocess.run([exe, "60", "3", "--layout"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "layout: 3600 of 3660 vertices kept" in r.stdout and "embedded! in time" in r.stdout
    assert "NaN" not in r.stdout + r.stderr

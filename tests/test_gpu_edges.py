"""ge_graph_from_edges equals the host restatement (tests/edges_restatement.py) bit for bit for every
combination of its options, and ge_layout_edges equals ge_graph_from_edges -> ge_layout_graph bit for
bit while only the edge arrays go up."""
import ctypes as C
import itertools
import os
import subprocess

import numpy as np
import pytest

import edges_restatement as R

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bits(x):
    return np.ascontiguousarray(x, np.float64).view(np.uint64)


def _same(A, ref):
    indptr, indices, data = ref
    assert np.array_equal(A.indptr, indptr) and np.array_equal(A.indices, indices)
    assert np.array_equal(_bits(A.data), _bits(data))


def _weighted(rows, cols, n, seed):
    w = np.random.default_rng(seed).standard_normal(len(rows))
    return n, rows, cols, w


def _real_weights(g):
    rng = np.random.default_rng(6)
    n, E = 5000, 400_000
    src, dst = rng.integers(0, n, E), rng.integers(0, n, E)
    w = rng.standard_normal(E) * 10.0 ** rng.integers(-8, 9, E)
    w[rng.random(E) < 0.05] = -0.0
    k = np.arange(2000)  # order-sensitive runs: 1e16, 1, -1e16 on the same entry, both directions
    src = np.r_[src, np.repeat(k, 3), np.repeat(k + 1, 3)]
    dst = np.r_[dst, np.repeat(k + 1, 3), np.repeat(k, 3)]
    w = np.r_[w, np.tile([1e16, 1.0, -1e16], 2 * k.size)]
    return n, src, dst, w


def _long_run(g):
    m = 1 << 20
    src = np.r_[np.full(m, 3), 0, 5]
    dst = np.r_[np.full(m, 8), 1, 5]
    w = np.random.default_rng(1).random(m + 2) * np.r_[np.tile([1.0, -1e10, 1e-10, 3.0], m // 4), 1.0, 1.0]
    return 10, src, dst, w


def _self_loops(g):
    v = np.random.default_rng(2).integers(0, 1000, 50_000)
    return 1000, v, v, np.random.default_rng(3).standard_normal(v.size)


def _empty_ends(g):
    rng = np.random.default_rng(4)
    src, dst = rng.integers(100, 900, 20_000), rng.integers(100, 900, 20_000)
    return 1000, src, dst, rng.random(src.size)


def _wide(g):
    n = (1 << 24) + 3
    src = np.array([0, n - 1, 5, 1 << 23, n - 1, 5, 12345678])
    dst = np.array([n - 1, 0, 1 << 23, 5, n - 1, 1 << 23, 7])
    return n, src, dst, np.array([1.5, -2.0, 0.25, 0.5, 3.0, 1e300, -1e-300])


CASES = {
    "rmat16": lambda g: _weighted(*g.rmat_edges(16, 16, seed=1), seed=11),
    "rmat18": lambda g: _weighted(*g.rmat_edges(18, 16, seed=2), seed=12),
    "rgg": lambda g: _weighted(*g.rgg_edges(200_000, 8.0, seed=3), seed=13),
    "delaunay200k": lambda g: _weighted(*g.delaunay3d_edges(200_000, seed=1), seed=14),
    "real_weights": _real_weights,
    "long_run": _long_run,
    "self_loops": _self_loops,
    "empty": lambda g: (100, np.zeros(0, np.int64), np.zeros(0, np.int64), np.zeros(0)),
    "empty_ends": _empty_ends,
    "wide": _wide,
}
_EDGES = {}


def _edges(graphs, name):
    if name not in _EDGES:
        _EDGES[name] = CASES[name](graphs)
    return _EDGES[name]


OPTIONS = list(itertools.product([True, False], repeat=3))  # symmetrize, keep_self_loops, unit_weights


@pytest.mark.parametrize("name", sorted(CASES))
def test_equals_restatement(ctx, graphs, name):
    n, src, dst, w = _edges(graphs, name)
    for sym, keep, unit in OPTIONS:
        A, st = ctx.graph_from_edges(n, src, dst, w, symmetrize=sym, keep_self_loops=keep, unit_weights=unit)
        ref = R.build(n, src, dst, w, symmetrize=sym, keep_self_loops=keep, unit_weights=unit)
        _same(A, ref)
        loops = int(np.count_nonzero(np.asarray(src) == np.asarray(dst)))
        assert st["nnz"] == A.nnz and st["self_loops_dropped"] == (0 if keep else loops)
        S = R.slots(n, src, dst, w, sym, keep)[0].size
        assert st["duplicates_merged"] == S - A.nnz
        assert 0 <= st["device_ms"] <= st["total_ms"]
    # weights absent: 1.0 each
    A, _ = ctx.graph_from_edges(n, src, dst)
    _same(A, R.build(n, src, dst))


@pytest.mark.parametrize("name", ["rmat16", "rgg", "delaunay200k"])
def test_unit_mode_equals_finish(ctx, graphs, name):
    n, src, dst, _ = _edges(graphs, name)
    A, _ = ctx.graph_from_edges(n, src, dst, unit_weights=True)
    ref = graphs._finish(src, dst, n)
    _same(A, (ref.indptr, ref.indices, ref.data))


def test_two_runs_are_identical(ctx, graphs):
    n, src, dst, w = _edges(graphs, "rmat18")
    A, _ = ctx.graph_from_edges(n, src, dst, w)
    B, _ = ctx.graph_from_edges(n, src, dst, w)
    _same(A, (B.indptr, B.indices, B.data))


def test_errors(ctx, capi):
    def status(f):
        with pytest.raises(capi.GeError) as e:
            f()
        return e.value.status

    src, dst = np.array([0, 1, 2]), np.array([1, 2, 3])
    assert status(lambda: ctx.graph_from_edges(3, src, dst)) == capi.GE_ERR_INVALID
    assert status(lambda: ctx.graph_from_edges(4, np.array([0, -1, 2]), dst)) == capi.GE_ERR_INVALID
    assert status(lambda: ctx.graph_from_edges(4, src, np.array([1, 2, -5]))) == capi.GE_ERR_INVALID
    for bad in (np.nan, np.inf, -np.inf):
        w = np.array([1.0, bad, 2.0])
        assert status(lambda: ctx.graph_from_edges(4, src, dst, w)) == capi.GE_ERR_INVALID
        assert status(lambda: ctx.graph_from_edges(4, src, dst, w, unit_weights=True)) == capi.GE_ERR_INVALID
    assert status(lambda: ctx.graph_from_edges(-1, [], [])) == capi.GE_ERR_INVALID
    # n = 0 with no edges is the empty graph
    A, _ = ctx.graph_from_edges(0, [], [])
    assert A.shape == (0, 0) and A.nnz == 0
    L = capi.lib()
    s32, d32 = src.astype(np.int32), dst.astype(np.int32)
    ptr, idx, val = np.zeros(5, np.int32), np.zeros(6, np.int32), np.zeros(6)
    nnz = C.c_int64()

    def call(E, cap):
        return L.ge_graph_from_edges(ctx.h, C.c_int32(4), C.c_int64(E), capi._ptr(s32, capi._pi),
                                     capi._ptr(d32, capi._pi), None, None, capi._ptr(ptr, capi._pi),
                                     capi._ptr(idx, capi._pi), capi._ptr(val, capi._pd), C.c_int64(cap),
                                     C.byref(nnz), None)
    assert call(-1, 6) == capi.GE_ERR_INVALID
    assert call(1 << 30, 6) == capi.GE_ERR_INVALID  # 2^31 slots: checked before anything is read
    nnz.value = -1
    assert call(3, 5) == capi.GE_ERR_INVALID and nnz.value == 6
    assert np.array_equal(ptr, [0, 1, 3, 5, 6])
    assert call(3, 6) == capi.GE_OK and nnz.value == 6
    assert np.array_equal(idx, [1, 0, 2, 1, 3, 2]) and (val == 1.0).all()


def _composed(ctx, n, src, dst, w, dim, largest, xo, **lo):
    h0, _ = ctx.bytes_moved
    A, _ = ctx.graph_from_edges(n, src, dst, w, **xo)
    h1, _ = ctx.bytes_moved
    x, vert, st = ctx.layout(A, dim, largest_component=largest, **lo)
    return x, vert, h1 - h0, st, A


def _grid_edges(nx, ny):
    ids = np.arange(nx * ny).reshape(nx, ny)
    return np.r_[ids[:-1, :].ravel(), ids[:, :-1].ravel()], np.r_[ids[1:, :].ravel(), ids[:, 1:].ravel()], nx * ny


def _disconnected_edges():
    """A grid with random duplicate edges, 50 isolated vertices and a small second grid."""
    r1, c1, n1 = _grid_edges(40, 40)
    r2, c2, n2 = _grid_edges(10, 3)
    rng = np.random.default_rng(5)
    r = np.r_[r1, r2 + n1 + 50, rng.integers(0, n1, 500)]
    c = np.r_[c1, c2 + n1 + 50, rng.integers(0, n1, 500)]
    return n1 + 50 + n2, r, c, None


def _unweighted(rows, cols, n):
    return n, rows, cols, None


def _positive_weights(rows, cols, n):
    return n, rows, cols, np.random.default_rng(3).random(len(rows)) + 0.1


LAYOUT_CASES = {  # (n, src, dst, weights)
    "rmat16_raw": lambda g: _unweighted(*g.rmat_edges(16, 16, seed=1)),
    "disconnected": lambda g: _disconnected_edges(),
    "connected_grid": lambda g: _unweighted(*_grid_edges(70, 50)),
    "real_weights": lambda g: _positive_weights(*g.rgg_edges(50_000, 8.0, seed=7)),
}


@pytest.mark.parametrize("name,dim,largest,unit,precision", [
    ("rmat16_raw", 3, True, True, 0), ("disconnected", 2, True, False, 0), ("connected_grid", 2, False, True, 0),
    ("real_weights", 3, True, False, 0), ("real_weights", 2, False, False, 1),
])
def test_layout_edges_equals_composed(ctx, graphs, name, dim, largest, unit, precision):
    n, src, dst, w = LAYOUT_CASES[name](graphs)
    xo = dict(unit_weights=unit)
    lo = dict(coarsening_factor=0.25, min_coarse=64, coarsen_seed=5, seed=11, precision=precision)
    h0, d0 = ctx.bytes_moved
    x, vert, xs, st = ctx.layout_edges(n, src, dst, dim, w, largest_component=largest, **xo, **lo)
    h1, d1 = ctx.bytes_moved
    assert (st["h2d_bytes"], st["d2h_bytes"]) == (h1 - h0, d1 - d0)
    y, wert, h_build, st2, A = _composed(ctx, n, src, dst, w, dim, largest, xo, **lo)
    assert np.array_equal(vert, wert)
    assert x.shape == y.shape and np.array_equal(_bits(x), _bits(y)) and np.isfinite(x).all()
    assert xs["nnz"] == A.nnz and st["levels"] == st2["levels"]
    # up: the edge arrays, then exactly what ge_layout_graph moves besides its CSR (O(n))
    E = len(src)
    edge_bytes = E * 8 + (E * 8 if w is not None else 0)
    csr_bytes = (n + 1) * 4 + A.nnz * 12
    assert st["h2d_bytes"] - edge_bytes == st2["h2d_bytes"] - csr_bytes
    assert st["h2d_bytes"] < h_build + st2["h2d_bytes"]


def test_layout_edges_errors_match(ctx, capi, graphs):
    def status(f):
        try:
            f()
        except capi.GeError as e:
            return e.status
        return capi.GE_OK

    src, dst, n = _grid_edges(20, 20)
    for args in [(n, src, dst, 4), (n - 1, src, dst, 2), (n, src, dst, 2, np.r_[np.nan, np.ones(len(src) - 1)])]:
        fused = status(lambda: ctx.layout_edges(*args, seed=1))
        composed = status(lambda: ctx.layout(ctx.graph_from_edges(*args[:3], *args[4:])[0], args[3], seed=1))
        assert fused == composed == capi.GE_ERR_INVALID


def test_layout_edges_multi_device(ctx, capi, graphs, monkeypatch):
    try:
        mc = capi.Context(devices=[0, 1])
    except capi.GeError as e:
        if e.status == capi.GE_ERR_INVALID and "more devices" in str(e):
            pytest.skip("box has fewer than 2 GPUs")
        raise
    monkeypatch.setenv("GE_SHARD_MIN_MPAIRS", "0.0001")  # shard every level of this small hierarchy
    n, src, dst, w = LAYOUT_CASES["rmat16_raw"](graphs)
    x2, v2, _, _ = mc.layout_edges(n, src, dst, 3, coarsen_seed=3, seed=4)
    y2, w2, _ = mc.layout(mc.graph_from_edges(n, src, dst)[0], 3, coarsen_seed=3, seed=4)
    x1, v1, _, _ = ctx.layout_edges(n, src, dst, 3, coarsen_seed=3, seed=4)
    assert np.array_equal(v2, w2) and np.array_equal(v2, v1)
    assert np.array_equal(_bits(x2), _bits(y2)) and np.array_equal(_bits(x2), _bits(x1))
    mc.close()


def test_cpp_dropin_demo_edges(capi):
    exe = os.path.join(ROOT, "graph-embed_b200", "lib", "ge_dropin_demo")
    if not os.path.exists(exe):
        from graph_embed_b200 import build
        build.build_all()
    r = subprocess.run([exe, "60", "3", "--edges"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "equal to CooMatrix" in r.stdout and "layoutEdges: 3600 vertices" in r.stdout
    assert "NaN" not in r.stdout + r.stderr

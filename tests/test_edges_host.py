"""The host restatement of ge_graph_from_edges against graphs._finish and CooMatrix semantics, the
factored edge generators, and the edge-list entry points without a device."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp

import edges_restatement as R


def _bits(x):
    return np.ascontiguousarray(x, np.float64).view(np.uint64)


def _same(got, A):
    indptr, indices, data = got
    assert np.array_equal(indptr, A.indptr) and np.array_equal(indices, A.indices)
    assert np.array_equal(_bits(data), _bits(A.data))


def _grid_edges(nx, ny):
    ids = np.arange(nx * ny).reshape(nx, ny)
    return np.r_[ids[:-1, :].ravel(), ids[:, :-1].ravel()], np.r_[ids[1:, :].ravel(), ids[:, 1:].ravel()], nx * ny


EDGES = {
    "grid": lambda g: _grid_edges(30, 40),
    "rgg": lambda g: g.rgg_edges(20000, 6.0, seed=5),
    "rmat14": lambda g: g.rmat_edges(14, 16, seed=3),
    "delaunay": lambda g: g.delaunay3d_edges(3000, seed=2),
}


@pytest.mark.parametrize("name", sorted(EDGES))
def test_unit_mode_equals_finish(graphs, name):
    rows, cols, n = EDGES[name](graphs)
    _same(R.build(n, rows, cols, unit_weights=True), graphs._finish(rows, cols, n))


def test_sum_mode_equals_coo_matrix():
    rng = np.random.default_rng(4)
    n, E = 40, 3000
    src, dst = rng.integers(0, n, E), rng.integers(0, n, E)
    w = rng.standard_normal(E) * 10.0 ** rng.integers(-3, 4, E)
    w[:5] = -0.0
    # an order-sensitive run: (1e16 + 1) - 1e16 = 0 but (1e16 - 1e16) + 1 = 1
    src = np.r_[src, 7, 7, 7, 3, 3]
    dst = np.r_[dst, 9, 9, 9, 5, 5]
    w = np.r_[w, 1e16, 1.0, -1e16, 2.5, -2.5]
    for sym in (True, False):
        for keep in (True, False):
            got = R.build(n, src, dst, w, symmetrize=sym, keep_self_loops=keep)
            ref = R.coo_matrix_dict(n, src, dst, w, symmetrize=sym, keep_self_loops=keep)
            for a, b in zip(got[:2], ref[:2]):
                assert np.array_equal(a, b)
            assert np.array_equal(_bits(got[2]), _bits(ref[2]))
    indptr, indices, data = R.build(n, [7, 7, 7, 1], [9, 9, 9, 1], [1e16, 1.0, -1e16, -0.0])
    assert data[indptr[7]] == 0.0  # the 1.0 is absorbed by 1e16 first
    assert indptr[2] - indptr[1] == 0  # the self-loop is dropped


def test_negative_zero_alone_becomes_positive_zero():
    _, _, data = R.build(3, [0], [2], [-0.0])
    assert np.array_equal(_bits(data), _bits([0.0, 0.0]))


def test_long_runs_sum_in_order():
    vals = np.r_[np.full(100, 1e-16), 1.0, np.full(5, 3.0)]
    starts, lengths = np.array([0, 101]), np.array([101, 5])
    s = R.run_sums(vals, starts, lengths)
    acc = 0.0
    for v in vals[:101]:
        acc += v
    assert s[0] == acc and s[1] == 15.0


@pytest.mark.parametrize("make,edges", [
    (lambda g, **k: g.rmat(12, **k), lambda g: g.rmat_edges(12)),
    (lambda g, **k: g.rgg(20000, 3.0, seed=5, **k), lambda g: g.rgg_edges(20000, 3.0, seed=5)),
    (lambda g, **k: g.delaunay3d(2000, seed=2, **k), lambda g: g.delaunay3d_edges(2000, seed=2)),
])
def test_edge_generators_reproduce_graphs(graphs, make, edges):
    A = graphs._finish(*edges(graphs))
    B = make(graphs, largest=False)
    assert np.array_equal(A.indptr, B.indptr) and np.array_equal(A.indices, B.indices)
    assert np.array_equal(_bits(A.data), _bits(B.data))


def test_edge_entry_points_without_device(capi):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    src = np.array([0, 1, 2], np.int32)
    dst = np.array([1, 2, 3], np.int32)
    ptr, idx, val = np.zeros(5, np.int32), np.zeros(6, np.int32), np.zeros(6)
    nnz = C.c_int64()
    L = capi.lib()
    st = L.ge_graph_from_edges(None, C.c_int32(4), C.c_int64(3), capi._ptr(src, capi._pi), capi._ptr(dst, capi._pi),
                               None, None, capi._ptr(ptr, capi._pi), capi._ptr(idx, capi._pi),
                               capi._ptr(val, capi._pd), C.c_int64(6), C.byref(nnz), None)
    assert st == capi.GE_ERR_NO_DEVICE
    x = np.zeros((4, 2))
    n = C.c_int32()
    st = L.ge_layout_edges(None, C.c_int32(4), C.c_int64(3), capi._ptr(src, capi._pi), capi._ptr(dst, capi._pi),
                           None, None, 2, 1, None, None, capi._ptr(x, capi._pd), None, C.byref(n), None, None)
    assert st == capi.GE_ERR_NO_DEVICE


def test_python_rejects_ids_beyond_int32(capi):
    with pytest.raises(capi.GeError) as e:
        capi.EdgeList(4, np.array([0, 2 ** 31]), np.array([1, 2]))
    assert e.value.status == capi.GE_ERR_INVALID
    with pytest.raises(capi.GeError):
        capi.EdgeList(2 ** 31, np.array([0]), np.array([1]))
    el = capi.EdgeList(4, np.array([0, 3], np.int64), np.array([1, 2], np.int64), [0.5, 2.0])
    assert el.src.dtype == np.int32 and el.E == 2 and el.w.dtype == np.float64


def test_restatement_shapes():
    indptr, indices, data = R.build(5, [], [], None)
    assert np.array_equal(indptr, np.zeros(6)) and indices.size == 0 and data.size == 0
    indptr, indices, data = R.build(6, [4, 1, 1], [4, 1, 1], [2.0, 3.0, 4.0], keep_self_loops=True)
    assert np.array_equal(indptr, [0, 0, 1, 1, 1, 2, 2]) and np.array_equal(indices, [1, 4])
    assert np.array_equal(data, [7.0, 2.0])
    A = sp.csr_matrix((data, indices, indptr), shape=(6, 6))
    assert A[1, 1] == 7.0

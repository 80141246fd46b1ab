"""ge_largest_component / ge_layout_graph without a device, and the raw generator graphs (largest=False)."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp


def _same(X, Y):
    assert X.shape == Y.shape
    assert np.array_equal(X.indptr, Y.indptr) and np.array_equal(X.indices, Y.indices)
    assert np.array_equal(X.data.view(np.uint64), Y.data.view(np.uint64))


def test_entry_points_without_device(capi):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    A = sp.identity(4, format="csr")
    a = capi.CsrView(A)
    vert, ptr, idx, val = (np.zeros(4, np.int32), np.zeros(5, np.int32), np.zeros(4, np.int32), np.zeros(4))
    n, nnz, comps = C.c_int32(), C.c_int64(), C.c_int64()
    st = capi.lib().ge_largest_component(None, a.ref(), capi._ptr(vert, capi._pi), C.byref(n),
                                         capi._ptr(ptr, capi._pi), capi._ptr(idx, capi._pi),
                                         capi._ptr(val, capi._pd), C.c_int64(4), C.byref(nnz), C.byref(comps))
    assert st == capi.GE_ERR_NO_DEVICE
    x = np.zeros((4, 2))
    st = capi.lib().ge_layout_graph(None, a.ref(), 2, 1, None, None, capi._ptr(x, capi._pd), None, C.byref(n),
                                    None)
    assert st == capi.GE_ERR_NO_DEVICE


@pytest.mark.parametrize("make", [lambda g, **k: g.rmat(12, **k), lambda g, **k: g.rgg(20000, 3.0, seed=5, **k),
                                  lambda g, **k: g.delaunay3d(2000, seed=2, **k)])
def test_raw_generators(graphs, make):
    raw = make(graphs, largest=False)
    _same(graphs.largest_component(raw), make(graphs))
    _same(make(graphs, largest=True), make(graphs))

"""The hierarchy builder of ge_coarsen restated on the host (tests/coarsen_restatement.py): its hash, the
properties of the hierarchies it builds, its edge cases, and the C entry point without a device."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp

import coarsen_restatement as R


def _mix64_int(x):
    """splitmix64's finaliser on Python integers: a second writing of the definition."""
    M = 2**64 - 1
    x = (x + 0x9E3779B97F4A7C15) & M
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & M
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & M
    return x ^ (x >> 31)


def test_hash_known_answers(oracle):
    # splitmix64 seeded with 0 outputs 0xe220a8397b1dcdaf first
    assert int(R.mix64(0)) == 0xE220A8397B1DCDAF == _mix64_int(0)
    assert int(R.mix64(1)) == 0x910A2DEC89025CC1
    assert int(R.coarsen_hash(0, 0, 0, 0, 0)) == 0xA706DD2F4D197E6F
    assert int(R.coarsen_hash(7, 2, 3, 1, 12345)) == 0x678F92BB74959DD4
    assert int(R.coarsen_hash(0xFFFFFFFF, 31, 100, 2, (5 << 32) | 9)) == 0xAC93A13722DAD66B
    v = np.arange(0, 5000, 7, dtype=np.uint64)
    base = _mix64_int((3 << 32) | (1 << 20) | (2 << 4) | 1)
    assert [int(h) for h in R.coarsen_hash(3, 1, 2, 1, v)] == [_mix64_int(base ^ int(x)) for x in v]


def _check_hierarchy(As, Ps, cf, min_coarse, exact=True, bound=True):
    for l, P in enumerate(Ps):
        n, m = As[l].shape[0], As[l + 1].shape[0]
        assert P.shape == (m, n)
        # a partition of the vertices, members ascending, no empty aggregate
        assert np.array_equal(np.sort(P.indices), np.arange(n))
        sizes = np.diff(P.indptr)
        assert (sizes > 0).all()
        for a in range(m):
            mem = P.indices[P.indptr[a]:P.indptr[a + 1]]
            assert (np.diff(mem) > 0).all()
        if bound:  # (a level can run out of candidates first: isolated vertices never merge)
            assert m <= max(int(np.floor(cf * n)), min_coarse)
        assert m < n
        ref = (P @ As[l] @ P.T).tocsr()
        ref.sort_indices()
        got = As[l + 1]
        if exact:
            assert abs(got - ref).max() == 0
        else:
            assert abs(got - ref).max() <= 1e-12 * abs(ref).max()
    return [A.shape[0] for A in As]


@pytest.mark.parametrize("name,cf,min_coarse", [("grid", 0.25, 64), ("rgg", 0.25, 30), ("rmat", 0.125, 50),
                                                ("rgg", 0.5, 10)])
def test_restatement_properties(oracle, graphs, name, cf, min_coarse):
    A = {"grid": lambda: graphs.grid2d(40, 40), "rgg": lambda: graphs.rgg(4000, 10.0, seed=2),
         "rmat": lambda: graphs.rmat(12, 16, seed=3)}[name]()
    As, Ps = R.coarsen(A, cf, min_coarse=min_coarse, seed=11)
    sizes = _check_hierarchy(As, Ps, cf, min_coarse)
    assert len(Ps) >= 2 and sizes[-1] <= max(min_coarse, int(cf * sizes[-2]))
    # levels keep the diagonal (intra-aggregate weight) and the total weight
    for l in range(len(Ps)):
        assert As[l + 1].sum() == pytest.approx(As[l].sum())


def test_restatement_is_a_function_of_the_seed(oracle, graphs):
    A = graphs.rgg(3000, 10.0, seed=4)
    As1, Ps1 = R.coarsen(A, 0.25, 32, seed=0)
    As2, Ps2 = R.coarsen(A, 0.25, 32, seed=0)
    As3, Ps3 = R.coarsen(A, 0.25, 32, seed=1)
    assert len(Ps1) == len(Ps2)
    for P, Q in zip(Ps1, Ps2):
        assert np.array_equal(P.indptr, Q.indptr) and np.array_equal(P.indices, Q.indices)
    for X, Y in zip(As1, As2):
        assert np.array_equal(X.indices, Y.indices) and np.array_equal(X.data, Y.data)
    assert not (Ps3[0].shape == Ps1[0].shape and np.array_equal(Ps3[0].indices, Ps1[0].indices))


def test_real_weights_equal_the_product_to_rounding(oracle, graphs):
    A = graphs.rgg(3000, 10.0, seed=5)
    rng = np.random.default_rng(1)
    W = sp.triu(A, 1)
    W.data = rng.random(W.nnz) + 0.1
    W = (W + W.T).tocsr()
    W.sort_indices()
    As, Ps = R.coarsen(W, 0.25, 30, seed=2)
    _check_hierarchy(As, Ps, 0.25, 30, exact=False)


def test_max_levels_and_small_graphs(oracle, graphs):
    A = graphs.grid2d(30, 30)
    As, Ps = R.coarsen(A, 0.25, 8, max_levels=2)
    assert len(Ps) == 2 and len(As) == 3
    As, Ps = R.coarsen(A, 0.25, 8, max_levels=0)
    assert len(Ps) == 0 and len(As) == 1
    As, Ps = R.coarsen(A, 0.25, 900)       # n <= min_coarse: nothing to do
    assert len(Ps) == 0
    As, Ps = R.coarsen(sp.csr_matrix((500, 500)), 0.25, 8)   # no edges: nothing merges
    assert len(Ps) == 0 and len(As) == 1


def test_isolated_vertices_and_several_components(oracle, graphs):
    G = graphs.grid2d(20, 20)
    Q = graphs.rgg(800, 8.0, seed=6)
    A = sp.block_diag([G, sp.csr_matrix((37, 37)), Q, sp.csr_matrix((5, 5))]).tocsr()
    A.sort_indices()
    As, Ps = R.coarsen(A, 0.25, 16, seed=3)
    _check_hierarchy(As, Ps, 0.25, 16, bound=False)
    # isolated vertices never merge and no aggregate spans two components
    comp = np.concatenate([np.zeros(400), np.arange(1, 38), np.full(Q.shape[0], 38),
                           np.arange(39, 44)]).astype(int)
    for P in Ps:
        agg_comp = np.full(P.shape[0], -1)
        v_A = oracle.vertex_to_aggregate(P)
        for v, a in enumerate(v_A):
            assert agg_comp[a] in (-1, comp[v])
            agg_comp[a] = comp[v]
        comp = agg_comp
    assert len(Ps) >= 1


def test_coarsen_without_device(capi):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    A = sp.identity(4, format="csr")
    a = capi.CsrView(A)
    opt = capi.CoarsenOptions()
    capi.lib().ge_coarsen_options_default(C.byref(opt))
    assert (opt.coarsening_factor, opt.min_coarse, opt.max_levels, opt.seed) == (0.25, 64, 32, 0)
    h = C.c_void_p()
    st = capi.lib().ge_coarsen(None, a.ref(), C.byref(opt), C.byref(h), None)
    assert st == capi.GE_ERR_NO_DEVICE and not h.value
    assert capi.lib().ge_hierarchy_levels(None) == 0

"""ge_coarsen: the hierarchy built on the device equals the host restatement
(tests/coarsen_restatement.py) exactly -- integer arrays equal, weights bit for bit -- and feeds
ge_embed."""
import os
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp

import coarsen_restatement as R

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _same(X, Y):
    assert X.shape == Y.shape
    assert np.array_equal(X.indptr, Y.indptr) and np.array_equal(X.indices, Y.indices)
    assert np.array_equal(np.asarray(X.data, np.float64).view(np.uint64),
                          np.asarray(Y.data, np.float64).view(np.uint64))


def _same_hierarchy(got, ref):
    (As, Ps), (Rs, Qs) = got, ref
    assert len(Ps) == len(Qs) and len(As) == len(Rs)
    for P, Q in zip(Ps, Qs):
        _same(P, Q)
    for A, B in zip(As[1:], Rs[1:]):
        _same(A, B)


def _hub_graph(graphs):
    """An RGG plus a vertex joined to 6000 others: a row beyond 4096 entries, so the proposal takes
    the CTA-per-row path and the Galerkin product segments beyond shared memory."""
    A = graphs.rgg(20000, 10.0, seed=8)
    n = A.shape[0]
    nb = np.random.default_rng(3).choice(n, 6000, replace=False)
    hub = np.full(nb.size, n)
    B = sp.coo_matrix((np.ones(2 * nb.size), (np.r_[hub, nb], np.r_[nb, hub])), shape=(n + 1, n + 1))
    return graphs.canonical(sp.bmat([[A, None], [None, sp.csr_matrix((1, 1))]]) + B)


def _real_weights(graphs):
    A = graphs.rgg(30000, 10.0, seed=9)
    W = sp.triu(A, 1).tocsr()
    W.data = np.random.default_rng(2).random(W.nnz) * 3.0 + 0.01
    return graphs.canonical(W + W.T)


def _disconnected(graphs):
    parts = [graphs.grid2d(40, 40), sp.csr_matrix((50, 50)), graphs.rgg(5000, 8.0, seed=4),
             graphs.grid2d(3, 1)]
    return graphs.canonical(sp.block_diag(parts))


CASES = {
    "grid100": lambda g: g.grid2d(100, 100),
    "rgg100k": lambda g: g.rgg(100_000, 10.0, seed=1),
    "rmat16": lambda g: g.rmat(16, 16, seed=1),
    "delaunay200k": lambda g: g.delaunay3d(200_000, seed=1),
    "real_weights": _real_weights,
    "hub": _hub_graph,
    "disconnected": _disconnected,
}
_GRAPHS = {}


def _graph(graphs, name):
    if name not in _GRAPHS:
        _GRAPHS[name] = CASES[name](graphs)
    return _GRAPHS[name]


@pytest.mark.parametrize("name,cf,min_coarse,seed", [
    ("grid100", 0.25, 64, 0), ("grid100", 0.5, 10, 7),
    ("rgg100k", 0.25, 64, 0), ("rgg100k", 0.125, 100, 3),
    ("rmat16", 0.25, 64, 0), ("rmat16", 0.25, 30, 12345),
    ("delaunay200k", 0.125, 64, 1),
    ("real_weights", 0.25, 50, 5),
    ("hub", 0.25, 64, 2), ("hub", 0.5, 200, 9),
    ("disconnected", 0.25, 16, 4),
])
def test_device_hierarchy_equals_restatement(ctx, oracle, graphs, name, cf, min_coarse, seed):
    A = _graph(graphs, name)
    As, Ps, st = ctx.coarsen(A, cf, min_coarse=min_coarse, seed=seed)
    Rs, Qs = R.coarsen(A, cf, min_coarse=min_coarse, seed=seed)
    _same_hierarchy((As, Ps), (Rs, Qs))
    assert len(Ps) >= 1 and st["rounds"] >= len(Ps) and st["kernel_launches"] > 0
    assert 0 < st["device_ms"] <= st["total_ms"]


def test_no_weights_array_means_unit_weights(ctx, capi, oracle, graphs):
    import ctypes as C
    A = graphs.rgg(20000, 10.0, seed=2)
    As, Ps, _ = ctx.coarsen(A, 0.25, 32, seed=6)
    a = capi.CsrView(A, with_data=False)
    opt = capi.CoarsenOptions(0.25, 32, 32, 6)
    h = C.c_void_p()
    capi._check(capi.lib().ge_coarsen(ctx.h, a.ref(), C.byref(opt), C.byref(h), None))
    try:
        assert capi.lib().ge_hierarchy_levels(h) == len(Ps)
        for l in range(len(Ps)):
            c = capi.Csr()
            capi._check(capi.lib().ge_hierarchy_aggregation(h, l, C.byref(c)))
            _same(capi._csr_copy(c), Ps[l])
            capi._check(capi.lib().ge_hierarchy_graph(h, l + 1, C.byref(c)))
            _same(capi._csr_copy(c), As[l + 1])
        c = capi.Csr()
        assert capi.lib().ge_hierarchy_graph(h, 0, C.byref(c)) == capi.GE_ERR_INVALID
        assert capi.lib().ge_hierarchy_aggregation(h, len(Ps), C.byref(c)) == capi.GE_ERR_INVALID
    finally:
        capi.lib().ge_hierarchy_destroy(h)


def test_edge_cases(ctx, capi, graphs):
    A = graphs.grid2d(30, 30)
    assert len(ctx.coarsen(A, 0.25, 8, max_levels=2)[1]) == 2
    assert len(ctx.coarsen(A, 0.25, 900)[1]) == 0
    As, Ps, _ = ctx.coarsen(sp.csr_matrix((500, 500)), 0.25, 8)
    assert len(Ps) == 0 and len(As) == 1
    with pytest.raises(capi.GeError) as e:
        ctx.coarsen(sp.csr_matrix((3, 4)), 0.25, 1)
    assert e.value.status == capi.GE_ERR_INVALID
    bad = sp.csr_matrix((np.ones(2), np.array([0, 7], dtype=np.int32), np.array([0, 1, 2], dtype=np.int32)),
                        shape=(2, 2))
    with pytest.raises(capi.GeError) as e:
        ctx.coarsen(bad, 0.25, 1)
    assert e.value.status == capi.GE_ERR_INVALID
    with pytest.raises(capi.GeError):
        ctx.coarsen(A, 0.0, 8)


def test_two_runs_are_identical(ctx, graphs):
    A = _graph(graphs, "rmat16")
    As1, Ps1, _ = ctx.coarsen(A, 0.25, 64, seed=77)
    As2, Ps2, _ = ctx.coarsen(A, 0.25, 64, seed=77)
    _same_hierarchy((As1, Ps1), (As2, Ps2))


def test_multi_device_context_gives_the_same_hierarchy(ctx, capi, graphs):
    try:
        mc = capi.Context(devices=[0, 1])
    except capi.GeError as e:
        if e.status == capi.GE_ERR_INVALID and "more devices" in str(e):
            pytest.skip("box has fewer than 2 GPUs")
        raise
    A = _graph(graphs, "rgg100k")
    got = mc.coarsen(A, 0.25, 64, seed=1)
    ref = ctx.coarsen(A, 0.25, 64, seed=1)
    _same_hierarchy(got[:2], ref[:2])
    mc.close()


@pytest.mark.parametrize("name,cf", [("rmat16", 0.25), ("delaunay200k", 0.125)])
def test_embed_on_device_built_hierarchy(ctx, capi, graphs, name, cf):
    As, Ps, _ = ctx.coarsen(_graph(graphs, name), cf, 64, seed=0)
    dim = 3
    x, st = ctx.embed(As, Ps, dim, seed=1)
    assert np.isfinite(x).all() and x.shape == (As[0].shape[0], dim)
    v_A = capi.vertex_to_aggregate(Ps[0])
    cent = np.zeros((Ps[0].shape[0], dim))
    np.add.at(cent, v_A, x)
    cent /= np.diff(Ps[0].indptr)[:, None]
    spread = np.linalg.norm(x - cent[v_A], axis=1).mean()
    extent = np.linalg.norm(x - x.mean(0), axis=1).max()
    assert spread < 0.05 * extent
    pairs = 100000.0 * As[-1].shape[0] * (As[-1].shape[0] - 1) + 100.0 * sum(
        float((np.diff(P.indptr).astype(np.int64) * (np.diff(P.indptr) - 1)).sum()) for P in Ps)
    assert st["pair_interactions"] == pytest.approx(pairs)


def test_cpp_dropin_demo_coarsen(capi):
    exe = os.path.join(ROOT, "graph-embed_b200", "lib", "ge_dropin_demo")
    if not os.path.exists(exe):
        from graph_embed_b200 import build
        build.build_all()
    r = subprocess.run([exe, "60", "3", "--coarsen"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "coarsen:" in r.stdout and "embedded! in time" in r.stdout
    assert "NaN" not in r.stdout + r.stderr

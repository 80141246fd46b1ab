"""Host restatement of ge_coarsen (include/graph_embed_b200.h): the level and round loop of the
stand-in generator graphs.coarsen with counter-based randomness, so that host and device draw the
same values.  The device must reproduce it exactly.  Test infrastructure (tests/, tools/); each
round is contracted with oracle_galerkin, the C restatement of the Galerkin product whose summation
order the device kernels share."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _oracle():
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    import __graft_entry__ as entry
    return entry.load_oracle()


_U64 = np.uint64


def mix64(x):
    """The splitmix64 finaliser on uint64 (wrapping arithmetic)."""
    x = np.asarray(x, dtype=_U64)
    with np.errstate(over="ignore"):
        x = x + _U64(0x9E3779B97F4A7C15)
        x = (x ^ (x >> _U64(30))) * _U64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> _U64(27))) * _U64(0x94D049BB133111EB)
    return x ^ (x >> _U64(31))


def coarsen_hash(seed, level, rnd, tag, v):
    """H(tag, v) = mix64(mix64(seed << 32 | level << 20 | round << 4 | tag) ^ v) in uint64."""
    base = mix64(_U64(((int(seed) << 32) | (int(level) << 20) | (int(rnd) << 4) | int(tag)) & (2**64 - 1)))
    return mix64(base ^ np.asarray(v, dtype=_U64))


def _aggregation(agg, m):
    """P_T (m x n, unit data) of a vertex -> aggregate map, members ascending per row."""
    import scipy.sparse as sp
    n = agg.shape[0]
    order = np.argsort(agg, kind="stable").astype(np.int32)
    indptr = np.zeros(m + 1, dtype=np.int32)
    np.cumsum(np.bincount(agg, minlength=m), out=indptr[1:])
    return sp.csr_matrix((np.ones(n), order, indptr), shape=(m, n))


def _coarsen_round(S, seed, level, rnd, max_merges):
    m = S.shape[0]
    ptr, idx = S.indptr, S.indices.astype(np.int64)
    w = S.data
    rows = np.repeat(np.arange(m, dtype=np.int64), np.diff(ptr))
    k = np.bincount(rows, weights=w, minlength=m)       # adds each row in CSR order, from 0.0
    k = np.where(k > 0, k, 1.0)
    head = (coarsen_hash(seed, level, rnd, 0, np.arange(m)) >> _U64(63)).astype(bool)
    ok = (rows != idx) & ~head[rows] & head[idx]
    r, c, wv = rows[ok], idx[ok], w[ok]
    if r.size == 0:
        return None
    score = wv / (k[r] * k[c])
    tie = coarsen_hash(seed, level, rnd, 2, (r.astype(_U64) << _U64(32)) | c.astype(_U64))
    order = np.lexsort((c, tie, -score, r))               # per tail: best score, hash, id first
    rs = r[order]
    first = np.r_[True, rs[1:] != rs[:-1]]
    tails, heads = rs[first], c[order][first]
    if tails.size > max_merges:
        keep = np.lexsort((tails, coarsen_hash(seed, level, rnd, 1, tails)))[:max_merges]
        keep.sort()
        tails, heads = tails[keep], heads[keep]
    label = np.arange(m)
    label[tails] = heads
    survive = np.ones(m, dtype=bool)
    survive[tails] = False
    newid = np.cumsum(survive) - 1                        # = np.unique(label, return_inverse=True)
    return newid[label], int(survive.sum())


def coarsen(A, coarsening_factor=0.25, min_coarse=64, max_levels=32, seed=0):
    """ge_coarsen restated: the level and round loop of graphs.coarsen with counter-based
    randomness.  -> (As, P_Ts); As[0] is A itself (int32 / float64 CSR, entry order kept)."""
    import scipy.sparse as sp
    A = sp.csr_matrix(A)
    data = A.data if A.data is not None else np.ones(A.nnz)
    A = sp.csr_matrix((np.ascontiguousarray(data, dtype=np.float64), np.ascontiguousarray(A.indices, dtype=np.int32),
                       np.ascontiguousarray(A.indptr, dtype=np.int32)), shape=A.shape)
    As, P_Ts = [A], []
    while As[-1].shape[0] > min_coarse and len(P_Ts) < max_levels:
        level, N = len(P_Ts), As[-1].shape[0]
        agg, M, S = np.arange(N), N, As[-1]
        target = max(int(np.floor(coarsening_factor * N)), min_coarse)
        rnd = 0
        while M > target:
            res = _coarsen_round(S, seed, level, rnd, M - target)
            rnd += 1
            if res is None:
                break
            new, M = res
            agg = new[agg]
            S = _oracle().galerkin(S, _aggregation(new, M))
        if M == N:
            break
        P_Ts.append(_aggregation(agg, M))
        As.append(S)
    return As, P_Ts

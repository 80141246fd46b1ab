"""Host restatement of ge_graph_from_edges (include/graph_embed_b200.h): the CSR that linalgcpp's
CooMatrix returns after Add(src, dst, w) for every kept edge, then Add(dst, src, w) when symmetrising
a non-loop edge.  The device must reproduce it bit for bit.  Test infrastructure (tests/, tools/).

Contribution `mirror` of edge e is slot 2e + mirror.  The kept slots are sorted stably on the packed
key (row << b) | col, so equal entries stay in slot order; each run is then summed in that order
from +0.0, one addition at a time, exactly as CooMatrix's `+=` does."""
import numpy as np


def key_bits(n):
    """b: the bit width of n - 1 (at least 1); keys are (row << b) | col."""
    return max(1, int(n - 1).bit_length()) if n > 1 else 1


def slots(n, src, dst, w=None, symmetrize=True, keep_self_loops=False):
    """The kept slots in slot order: (rows, cols, values), int64 / float64."""
    src = np.asarray(src, dtype=np.int64).ravel()
    dst = np.asarray(dst, dtype=np.int64).ravel()
    E = src.size
    w = np.ones(E) if w is None else np.asarray(w, dtype=np.float64).ravel()
    loop = src == dst
    keep = np.empty(2 * E, dtype=bool)
    keep[0::2] = ~loop | bool(keep_self_loops)
    keep[1::2] = ~loop & bool(symmetrize)
    rows = np.empty(2 * E, dtype=np.int64)
    cols = np.empty(2 * E, dtype=np.int64)
    rows[0::2], rows[1::2] = src, dst
    cols[0::2], cols[1::2] = dst, src
    return rows[keep], cols[keep], np.repeat(w, 2)[keep]


def run_sums(vals, starts, lengths):
    """Sum of every run vals[starts[r] : starts[r] + lengths[r]], in order, from +0.0: the k-th
    member of every run still open is added in step k.  The last few long runs are finished one
    value at a time (Python floats are IEEE doubles: the same additions)."""
    sums = np.zeros(starts.size)
    active = np.arange(starts.size)
    k = 0
    while active.size > 8:
        sums[active] += vals[starts[active] + k]
        k += 1
        active = active[lengths[active] > k]
    for r in active:
        acc = float(sums[r])
        for v in vals[starts[r] + k:starts[r] + lengths[r]].tolist():
            acc += v
        sums[r] = acc
    return sums


def build(n, src, dst, w=None, symmetrize=True, keep_self_loops=False, unit_weights=False):
    """(indptr int32 [n+1], indices int32, data float64) of ge_graph_from_edges."""
    rows, cols, vals = slots(n, src, dst, w, symmetrize, keep_self_loops)
    b = key_bits(n)
    key = (rows << b) | cols
    order = np.argsort(key, kind="stable")
    key, vals = key[order], vals[order]
    S = key.size
    head = np.ones(S, dtype=bool)
    head[1:] = key[1:] != key[:-1]
    starts = np.flatnonzero(head)
    lengths = np.diff(np.r_[starts, S])
    ukey = key[starts]
    urow, ucol = ukey >> b, ukey & ((1 << b) - 1)
    data = np.ones(starts.size) if unit_weights else run_sums(vals, starts, lengths)
    indptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(urow, minlength=n), out=indptr[1:])
    return indptr.astype(np.int32), ucol.astype(np.int32), data


def coo_matrix_dict(n, src, dst, w=None, symmetrize=True, keep_self_loops=False):
    """CooMatrix itself, in plain Python: a dict of running sums in call order, read out sorted."""
    acc = {}
    ws = [1.0] * len(src) if w is None else [float(x) for x in w]
    for s, d, x in zip([int(v) for v in src], [int(v) for v in dst], ws):
        if s == d and not keep_self_loops:
            continue
        acc[(s, d)] = acc.get((s, d), 0.0) + x
        if symmetrize and s != d:
            acc[(d, s)] = acc.get((d, s), 0.0) + x
    entries = sorted(acc.items())
    indptr = np.zeros(n + 1, dtype=np.int32)
    for (r, _), _v in entries:
        indptr[r + 1] += 1
    indptr = np.cumsum(indptr).astype(np.int32)
    return indptr, np.array([c for (_, c), _ in entries], dtype=np.int32), np.array([v for _, v in entries])

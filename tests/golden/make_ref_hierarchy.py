"""Caches hierarchies produced by the REFERENCE's own partitioner for the large BASELINE configs.

  python tests/golden/make_ref_hierarchy.py rmat20      -> tests/golden/refhier_rmat20.npz
  python tests/golden/make_ref_hierarchy.py delaunay N   -> tests/golden/refhier_delaunayN.npz

Runs `partition::partition(A, cf, false, true, 1.0, 2, false)` (src/partitioner.cpp:1550-1893, the call
shape of examples/embedder.cpp:187) through oracle/_ref (the unmodified reference compiled by
oracle/Makefile) on the synthetic graph the generator in graph-embed_b200/graphs.py produces for the
given seed, and stores ONLY the vertex->aggregate map of every level, relative to that level's graph
(tests/helpers.py::encode_aggregates), plus the generator's arguments and a checksum of the graph: the
graph itself is regenerated from the seed wherever the fixture is used
(tests/helpers.py::load_ref_hierarchy), and the checksum catches a generator that drifted.
Needs /root/reference (build container only); the partition of R-MAT-20 takes ~20 CPU-minutes, which
is why the result is committed.
"""
import hashlib
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
import __graft_entry__ as entry  # noqa: E402
from helpers import pack_i32, encode_aggregates  # noqa: E402

entry.load_package()
O = entry.load_oracle()
from graph_embed_b200 import graphs as G  # noqa: E402


def graph_digest(A):
    h = hashlib.sha256()
    h.update(np.ascontiguousarray(A.indptr).tobytes())
    h.update(np.ascontiguousarray(A.indices).tobytes())
    return h.hexdigest()


def build_graph(kind, arg, seed):
    if kind == "rmat":
        return G.rmat(int(arg), 16, seed=seed), 0.25
    if kind == "delaunay":
        return G.delaunay3d(int(arg), seed=seed), 0.125
    if kind == "rgg":
        return G.rgg(int(arg), 10.0, seed=seed), 0.25
    raise SystemExit("unknown graph kind")


def main():
    kind = sys.argv[1]
    arg = int(sys.argv[2])
    seed = int(sys.argv[3]) if len(sys.argv) > 3 else 1
    threads = int(os.environ.get("GE_PART_THREADS", "8"))
    O.build(ref=True)
    assert O.ref_available("fast"), "oracle/_ref missing (needs /root/reference)"
    t = time.time()
    A, cf = build_graph(kind, arg, seed)
    print("graph", A.shape[0], A.nnz, "in %.1f s" % (time.time() - t), flush=True)
    t = time.time()
    Ps = O.ref_partition(A, cf, matching_iterations=2, nthreads=threads, kind="fast")
    secs = time.time() - t
    print("partition: %d levels in %.1f s" % (len(Ps), secs), flush=True)
    out = {"kind": kind, "arg": np.int64(arg), "seed": np.int64(seed), "cf": np.float64(cf),
           "n": np.int64(A.shape[0]), "nnz": np.int64(A.nnz), "digest": graph_digest(A),
           "L": np.int32(len(Ps)), "partition_seconds": np.float64(secs),
           "partition_threads": np.int32(threads)}
    As = G.hierarchy_from(A, Ps)
    for l, P in enumerate(Ps):
        # P_T has one unit entry per column and members ascending per row (interpolationMatrix,
        # src/partitioner.cpp:29-65): the vertex->aggregate map determines it completely.
        agg = np.zeros(P.shape[1], dtype=np.int32)
        agg[P.indices] = np.repeat(np.arange(P.shape[0], dtype=np.int32), np.diff(P.indptr))
        rebuilt = G.aggregation_matrix(agg, P.shape[0])
        assert np.array_equal(rebuilt.indptr, P.indptr) and np.array_equal(rebuilt.indices, P.indices), \
            "members not ascending: the map does not determine P_T at level %d" % l
        link, root_ids = encode_aggregates(As[l], P)
        out["link%d" % l], out["roots%d" % l] = pack_i32(link), pack_i32(root_ids)
        s = np.diff(P.indptr).astype(np.int64)
        print("level", l, "n", P.shape[1], "aggregates", P.shape[0], "max", int(s.max()),
              "pairs", int((s * (s - 1)).sum()), flush=True)
    name = "refhier_%s%d.npz" % (kind, arg)
    np.savez(os.path.join(HERE, name), **out)  # the members are xz-compressed already
    print("wrote", name, os.path.getsize(os.path.join(HERE, name)), "bytes")


if __name__ == "__main__":
    main()

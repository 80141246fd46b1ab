"""ge_coarsen at full size: the hierarchy built on the device for a 1M-vertex RGG, the R-MAT-20
largest component and the 1M-point Delaunay graph.  Per graph: the call's wall and device time
(3 untimed calls, then the median of 5), equality with the host restatement
(tests/coarsen_restatement.py), the level shapes, and -- for R-MAT-20 and Delaunay 1M -- the per-level
modularity, ge_embed time and layout statistics of this hierarchy next to the reference
partitioner's (tests/golden/refhier_*.npz).  Kernel time by name from torch.profiler (CUDA
activities) for one call per graph.  Needs a B200.

    python tools/run_coarsen.py [--out profiles/r03_coarsen.json] [--graphs rgg1m,rmat20,delaunay1m]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import __graft_entry__ as entry  # noqa: E402

entry.load_package()
from graph_embed_b200 import capi, graphs  # noqa: E402
import coarsen_restatement  # noqa: E402
from helpers import layout_stats, load_ref_hierarchy  # noqa: E402

# graph, coarsening factor and dimension of the BASELINE config it belongs to
CASES = {"rgg1m": (0.25, 2), "rmat20": (0.25, 3), "delaunay1m": (0.125, 3)}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
        return dict(name=name, power_limit=power)
    except Exception as e:  # the numbers still stand, with the card named by the runtime
        import torch
        return dict(name=torch.cuda.get_device_name(0), power_limit="unknown (%s)" % e)


def modularity(A, P):
    """Newman modularity of the partition P (m x n aggregation) of the weighted graph A."""
    v_A = capi.vertex_to_aggregate(P)
    k = np.asarray(A.sum(axis=1)).ravel()
    two_m = k.sum()
    coo = A.tocoo()
    intra = coo.data[v_A[coo.row] == v_A[coo.col]].sum()
    K = np.bincount(v_A, weights=k, minlength=P.shape[0])
    return float(intra / two_m - ((K / two_m) ** 2).sum())


def same(X, Y):
    return (X.shape == Y.shape and np.array_equal(X.indptr, Y.indptr) and np.array_equal(X.indices, Y.indices)
            and np.array_equal(np.asarray(X.data).view(np.uint64), np.asarray(Y.data).view(np.uint64)))


def kernel_times(ctx, A, cf):
    """Device time per kernel name over one ge_coarsen call (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.coarsen(A, cf, 64, seed=0)
    rows = []
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = getattr(ev, "cuda_time_total", 0.0)
        if t > 0:
            rows.append(dict(name=ev.key[:100], calls=int(ev.count), ms=t / 1000.0))
    rows.sort(key=lambda r: -r["ms"])
    return rows[:15]


def upload_ms(As, Ps):
    """Host -> device copy of the level graphs ge_embed uploads again (pageable numpy arrays)."""
    import torch
    arrs = []
    for A in As[1:]:
        arrs += [A.indptr, A.indices, A.data]
    for P in Ps:
        arrs += [P.indptr, P.indices]
    nbytes = sum(a.nbytes for a in arrs)
    for rep in range(2):
        torch.cuda.synchronize()
        t = time.perf_counter()
        for a in arrs:
            torch.from_numpy(np.ascontiguousarray(a)).to("cuda", non_blocking=False)
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t) * 1e3
    return dict(bytes=int(nbytes), ms=ms)


def graph_of(name):
    """-> (A, the reference partitioner's (As, P_Ts) or None)"""
    if name == "rgg1m":
        return graphs.rgg(1_000_000, 10.0, seed=1), None
    ref = load_ref_hierarchy(graphs, "rmat20" if name == "rmat20" else "delaunay1000000")
    return ref[0][0], ref


def restatement(name):
    """The host restatement on one graph (runs in a worker process, one host core)."""
    A, _ = graph_of(name)
    t = time.perf_counter()
    Rs, Qs = coarsen_restatement.coarsen(A, CASES[name][0], 64, seed=0)
    return Rs, Qs, time.perf_counter() - t


def run(ctx, name, check):
    cf, dim = CASES[name]
    A, ref = graph_of(name)
    out = dict(graph=name, n=int(A.shape[0]), nnz=int(A.nnz), coarsening_factor=cf, min_coarse=64, seed=0)
    for _ in range(3):
        ctx.coarsen(A, cf, 64, seed=0)
    tot, dev, wall = [], [], []
    for _ in range(5):
        t = time.perf_counter()
        As, Ps, st = ctx.coarsen(A, cf, 64, seed=0)
        wall.append((time.perf_counter() - t) * 1e3)
        tot.append(st["total_ms"])
        dev.append(st["device_ms"])
    out.update(total_ms_median=float(np.median(tot)), device_ms_median=float(np.median(dev)),
               python_wall_ms_median=float(np.median(wall)), total_ms_all=tot, device_ms_all=dev,
               rounds=int(st["rounds"]), kernel_launches=int(st["kernel_launches"]), levels=len(Ps))
    out["level_shapes"] = graphs.level_stats(As, Ps)
    out["kernels"] = kernel_times(ctx, A, cf)
    if check is not None:
        Rs, Qs, secs = check.result()
        out["restatement_seconds"] = secs
        out["equal_to_restatement"] = bool(len(Qs) == len(Ps) and all(same(P, Q) for P, Q in zip(Ps, Qs))
                                           and all(same(X, Y) for X, Y in zip(As[1:], Rs[1:])))
    out["modularity"] = [modularity(As[l], P) for l, P in enumerate(Ps)]
    out["level_graph_upload"] = upload_ms(As, Ps)
    hier = {"device": (As, Ps)}
    if ref is not None:
        hier["reference_partitioner"] = (ref[0], ref[1])
        out["reference_modularity"] = [modularity(ref[0][l], P) for l, P in enumerate(ref[1])]
        out["reference_level_shapes"] = graphs.level_stats(ref[0], ref[1])
    out["embed"] = {}
    for key, (Xs, Zs) in hier.items():
        ctx.embed(Xs, Zs, dim, seed=1)                        # warm-up
        x, est = ctx.embed(Xs, Zs, dim, seed=1)
        out["embed"][key] = dict(dim=dim, total_ms=est["total_ms"], h2d_bytes=est["h2d_bytes"],
                                 pair_interactions=est["pair_interactions"],
                                 layout=layout_stats(Xs[0], x))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_coarsen.json"))
    ap.add_argument("--graphs", default="rgg1m,rmat20,delaunay1m")
    ap.add_argument("--no-check", action="store_true", help="skip the host restatement")
    args = ap.parse_args()
    names = args.graphs.split(",")
    checks = {}
    if not args.no_check:  # the host restatements run beside the device measurements
        import multiprocessing
        from concurrent.futures import ProcessPoolExecutor
        pool = ProcessPoolExecutor(max_workers=len(names), mp_context=multiprocessing.get_context("spawn"))
        checks = {name: pool.submit(restatement, name) for name in names}
    ctx = capi.Context(0)
    res = dict(card=card(), graphs=[])
    for name in names:
        r = run(ctx, name, checks.get(name))
        print(json.dumps({k: v for k, v in r.items() if k not in ("level_shapes", "reference_level_shapes",
                                                                  "kernels")}), flush=True)
        res["graphs"].append(r)
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    ctx.close()
    if checks:
        pool.shutdown()


if __name__ == "__main__":
    main()

"""ge_graph_from_edges and ge_layout_edges at full size, on the raw edges of R-MAT-20 (16.8 M edges,
cf 0.25, d = 3), the 1M-vertex RGG (its pairs, cf 0.25, d = 2) and the 1M-point Delaunay graph (six
edges per tetrahedron, cf 0.125, d = 3).  Per graph, in one process, the arms alternated:
  gfe_unit     ge_graph_from_edges, unit mode (the graph graphs._finish builds)
  gfe_sum      ge_graph_from_edges, sum mode with random real weights
  host_finish  graphs._finish (scipy COO -> CSR + sum_duplicates) on this host
  layout_csr   ge_layout_graph on the CSR host_finish built (prebuilt CSR)
  layout_edges ge_layout_edges, unit mode
  composed     ge_graph_from_edges (unit) -> ge_layout_graph
Arm (a) of the issue is host_finish + layout_csr, timed in the same iteration.  3 untimed rounds,
then the median of 5; byte counters; bit equality of the graphs and of the three layouts (seed != 0);
in a separate torch.profiler run, the device time of the CUB sort and of the project's kernels of one
ge_graph_from_edges call per mode, and the bytes the project's kernels move against the HBM data-sheet
bandwidth.  The card's name and power limit are read in the same run.  Needs a B200.

    python tools/run_edges.py [--out profiles/r05_edges.json] [--graphs rmat20,rgg1m,delaunay1m]
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
import __graft_entry__ as entry  # noqa: E402

entry.load_package()
from graph_embed_b200 import capi, graphs  # noqa: E402

CASES = {
    "rmat20": (lambda: graphs.rmat_edges(20, 16), 0.25, 3),
    "rgg1m": (lambda: graphs.rgg_edges(1_000_000, 10.0), 0.25, 2),
    "delaunay1m": (lambda: graphs.delaunay3d_edges(1_000_000), 0.125, 3),
}
SEED, COARSEN_SEED = 1, 0
HBM_BPS = 7.7e12  # HGX B200 data sheet, one GPU


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
        return dict(name=name, power_limit=power)
    except Exception as e:  # the numbers still stand, with the card named by the runtime
        import torch
        return dict(name=torch.cuda.get_device_name(0), power_limit="unknown (%s)" % e)


def timed(ctx, f):
    h0, d0 = ctx.bytes_moved
    t0 = time.perf_counter()
    out = f()
    wall = (time.perf_counter() - t0) * 1e3
    h1, d1 = ctx.bytes_moved
    return out, dict(wall_ms=wall, h2d_bytes=h1 - h0, d2h_bytes=d1 - d0)


def one_round(ctx, n, src, dst, w, cf, dim):
    lo = dict(coarsening_factor=cf, min_coarse=64, coarsen_seed=COARSEN_SEED, seed=SEED)
    rec, out = {}, {}
    (A, st), m = timed(ctx, lambda: ctx.graph_from_edges(n, src, dst, unit_weights=True))
    rec["gfe_unit"] = dict(m, total_ms=st["total_ms"], device_ms=st["device_ms"], nnz=st["nnz"],
                           duplicates_merged=st["duplicates_merged"], self_loops_dropped=st["self_loops_dropped"],
                           kernel_launches=st["kernel_launches"])
    out["gfe_unit"] = A
    (B, st), m = timed(ctx, lambda: ctx.graph_from_edges(n, src, dst, w))
    rec["gfe_sum"] = dict(m, total_ms=st["total_ms"], device_ms=st["device_ms"], nnz=st["nnz"],
                          kernel_launches=st["kernel_launches"])
    t0 = time.perf_counter()
    H = graphs._finish(src, dst, n)
    rec["host_finish"] = dict(wall_ms=(time.perf_counter() - t0) * 1e3)
    out["host_finish"] = H
    (x, v, st), m = timed(ctx, lambda: ctx.layout(H, dim, **lo))
    rec["layout_csr"] = dict(m, total_ms=st["total_ms"])
    rec["a_host_finish_plus_layout_csr"] = dict(wall_ms=rec["host_finish"]["wall_ms"] + m["wall_ms"])
    out["layout_csr"] = (x, v)
    (x, v, xs, st), m = timed(ctx, lambda: ctx.layout_edges(n, src, dst, dim, unit_weights=True, **lo))
    rec["layout_edges"] = dict(m, total_ms=st["total_ms"], build_ms=xs["total_ms"], build_device_ms=xs["device_ms"],
                               components_ms=st["components_ms"], coarsen_ms=st["coarsen_ms"],
                               embed_ms=st["embed_ms"], levels=st["levels"])
    out["layout_edges"] = (x, v)

    def composed():
        G, _ = ctx.graph_from_edges(n, src, dst, unit_weights=True)
        return ctx.layout(G, dim, **lo)
    (x, v, st), m = timed(ctx, composed)
    rec["b_gfe_plus_layout_csr"] = m
    out["composed"] = (x, v)
    return rec, out


def bits_equal(A, B):
    return (np.array_equal(A.indptr, B.indptr) and np.array_equal(A.indices, B.indices)
            and np.array_equal(A.data.view(np.uint64), B.data.view(np.uint64)))


def layouts_equal(p, q):
    return np.array_equal(p[1], q[1]) and np.array_equal(p[0].view(np.uint64), q[0].view(np.uint64))


def model_bytes(E, S, U, n, weights):
    """Bytes the project's kernels of one build read and write, from the shapes (E edges, S kept
    slots, U entries); neighbouring reads that hit the same lines are counted once."""
    wv = 8 * E if weights else 0
    sv = 8 * S if weights else 0
    return {
        "k_edges_check": 8 * E + wv + 4 * E,
        "k_scan": 8 * E + 8 * S,  # the two scans (counts over E, run heads over S)
        "k_edges_emit": 8 * E + 4 * E + wv + 8 * S + sv,
        "k_edges_heads": 8 * S + 4 * S,
        "k_edges_reduce": 4 * S + 8 * S + sv + 8 * U + 8 * U,
        "k_edges_rowptr": 4 * U + 4 * (n + 1),
    }


def kernel_split(ctx, n, src, dst, w, unit):
    """Device time per kernel name of one ge_graph_from_edges call (torch.profiler)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        A, st = ctx.graph_from_edges(n, src, dst, None if unit else w, unit_weights=unit)
    rows = []
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = getattr(ev, "cuda_time_total", 0.0)
        if t > 0:
            rows.append(dict(name=ev.key[:120], calls=int(ev.count), ms=t / 1000.0))
    rows.sort(key=lambda r: -r["ms"])
    own = [r for r in rows if "k_edges" in r["name"] or "k_scan" in r["name"]]
    sort = [r for r in rows if "cub" in r["name"].lower() or "radix" in r["name"].lower()
            or "onesweep" in r["name"].lower()]
    E = len(src)
    S = st["nnz"] + st["duplicates_merged"]
    mb = model_bytes(E, S, st["nnz"], n, not unit)
    own_ms = sum(r["ms"] for r in own)
    own_bytes = sum(mb.values())
    return dict(kernels=rows[:20], sort_ms=sum(r["ms"] for r in sort), own_ms=own_ms,
                other_ms=sum(r["ms"] for r in rows) - own_ms - sum(r["ms"] for r in sort),
                own_model_bytes=mb, own_bytes_per_s=own_bytes / (own_ms * 1e-3) if own_ms else None,
                own_share_of_hbm=own_bytes / (own_ms * 1e-3) / HBM_BPS if own_ms else None)


def median(runs, arm, key):
    return float(np.median([r[arm][key] for r in runs]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_edges.json"))
    ap.add_argument("--graphs", default="rmat20,rgg1m,delaunay1m")
    args = ap.parse_args()
    ctx = capi.Context(0)
    result = dict(card=card(), seed=SEED, coarsen_seed=COARSEN_SEED, graphs={})
    for name in args.graphs.split(","):
        make, cf, dim = CASES[name]
        rows, cols, n = make()
        src, dst = rows.astype(np.int32), cols.astype(np.int32)  # the C ABI's id type, converted once
        w = np.random.default_rng(7).random(len(src)) + 0.5
        for _ in range(3):
            one_round(ctx, n, src, dst, w, cf, dim)
        runs, equal = [], dict(graph_unit_vs_finish=True, layout_edges_vs_a=True, layout_edges_vs_b=True)
        for _ in range(5):
            rec, out = one_round(ctx, n, src, dst, w, cf, dim)
            runs.append(rec)
            equal["graph_unit_vs_finish"] &= bits_equal(out["gfe_unit"], out["host_finish"])
            equal["layout_edges_vs_a"] &= layouts_equal(out["layout_edges"], out["layout_csr"])
            equal["layout_edges_vs_b"] &= layouts_equal(out["layout_edges"], out["composed"])
        med = {arm: {k: median(runs, arm, k) for k in runs[0][arm]} for arm in runs[0]}
        rec = dict(n=n, edges=len(src), edge_bytes_int32=8 * len(src), cf=cf, dim=dim,
                   bit_equal={k: bool(v) for k, v in equal.items()}, median=med, runs=runs,
                   profile_unit=kernel_split(ctx, n, src, dst, w, True),
                   profile_sum=kernel_split(ctx, n, src, dst, w, False))
        rec["layout_edges_minus_layout_csr_ms"] = med["layout_edges"]["wall_ms"] - med["layout_csr"]["wall_ms"]
        result["graphs"][name] = rec
        print(name, json.dumps({k: rec[k] for k in ("n", "edges", "bit_equal", "median",
                                                     "layout_edges_minus_layout_csr_ms")}), flush=True)
        print(name, "profile", json.dumps({k: rec["profile_unit"][k] for k in ("sort_ms", "own_ms", "other_ms",
                                                                              "own_share_of_hbm")}),
              json.dumps({k: rec["profile_sum"][k] for k in ("sort_ms", "own_ms", "other_ms", "own_share_of_hbm")}),
              flush=True)
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()

"""ge_layout_graph at full size: raw R-MAT-20 (cf 0.25, d = 3), a raw 1M-vertex RGG (average degree 10,
cf 0.25, d = 2) and the 1M-point Delaunay graph (cf 0.125, d = 3).  Per graph, in one process:
  (i)   ge_layout_graph (Context.layout) and its parts from ge_layout_stats;
  (ii)  the composed device path with its host round trips: ge_largest_component, ge_coarsen,
        ge_embed (Context.largest_component / coarsen / embed), alternated with (i);
  (iii) scipy's largest component (graphs.largest_component) for context.
3 untimed calls of (i) and (ii), then the median of 5 of each; byte counters of (i) and (ii); whether
(i) and (ii) are bit-equal (seed != 0); device time per kernel name of the component step from
torch.profiler (CUDA activities) in a separate call.  The card's name and power limit are read in the
same run.  Needs a B200.

    python tools/run_layout.py [--out profiles/r04_layout.json] [--graphs rmat20,rgg1m,delaunay1m]
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

# raw generator output (no largest-component step), coarsening factor, dimension
CASES = {
    "rmat20": (lambda: graphs.rmat(20, 16, largest=False), 0.25, 3),
    "rgg1m": (lambda: graphs.rgg(1_000_000, 10.0, largest=False), 0.25, 2),
    "delaunay1m": (lambda: graphs.delaunay3d(1_000_000, largest=False), 0.125, 3),
}
SEED, COARSEN_SEED = 1, 0


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
        return dict(name=name, power_limit=power)
    except Exception as e:  # the numbers still stand, with the card named by the runtime
        import torch
        return dict(name=torch.cuda.get_device_name(0), power_limit="unknown (%s)" % e)


def fused(ctx, A, cf, dim):
    h0, d0 = ctx.bytes_moved
    t0 = time.perf_counter()
    x, vert, st = ctx.layout(A, dim, cf, 64, coarsen_seed=COARSEN_SEED, seed=SEED)
    wall = (time.perf_counter() - t0) * 1e3
    h1, d1 = ctx.bytes_moved
    return x, vert, dict(wall_ms=wall, h2d_bytes=h1 - h0, d2h_bytes=d1 - d0,
                         **{k: st[k] for k in ("total_ms", "components_ms", "coarsen_ms", "embed_ms",
                                               "components", "levels", "kernel_launches")})


def composed(ctx, A, cf, dim):
    h0, d0 = ctx.bytes_moved
    t0 = time.perf_counter()
    B, vert, comps = ctx.largest_component(A)
    t1 = time.perf_counter()
    As, Ps, cst = ctx.coarsen(B, cf, 64, seed=COARSEN_SEED)
    t2 = time.perf_counter()
    x, est = ctx.embed(As, Ps, dim, seed=SEED)
    t3 = time.perf_counter()
    h1, d1 = ctx.bytes_moved
    return x, vert, dict(wall_ms=(t3 - t0) * 1e3, largest_component_ms=(t1 - t0) * 1e3,
                         coarsen_ms=(t2 - t1) * 1e3, embed_ms=(t3 - t2) * 1e3, h2d_bytes=h1 - h0,
                         d2h_bytes=d1 - d0, levels=len(Ps))


def kernel_times(ctx, A):
    """Device time per kernel name over one ge_largest_component call."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.largest_component(A)
    rows = []
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = getattr(ev, "cuda_time_total", 0.0)
        if t > 0:
            rows.append(dict(name=ev.key[:100], calls=int(ev.count), ms=t / 1000.0))
    rows.sort(key=lambda r: -r["ms"])
    return rows[:15]


def median(runs, key):
    return float(np.median([r[key] for r in runs]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_layout.json"))
    ap.add_argument("--graphs", default="rmat20,rgg1m,delaunay1m")
    args = ap.parse_args()
    ctx = capi.Context(0)
    result = dict(card=card(), seed=SEED, coarsen_seed=COARSEN_SEED, graphs={})
    for name in args.graphs.split(","):
        make, cf, dim = CASES[name]
        A = make()
        t0 = time.perf_counter()
        ref = graphs.largest_component(A)
        scipy_ms = (time.perf_counter() - t0) * 1e3
        for _ in range(3):
            fused(ctx, A, cf, dim)
            composed(ctx, A, cf, dim)
        fr, cr, equal = [], [], True
        for _ in range(5):
            x, v, f = fused(ctx, A, cf, dim)
            y, w, c = composed(ctx, A, cf, dim)
            fr.append(f)
            cr.append(c)
            equal = equal and np.array_equal(v, w) and np.array_equal(x.view(np.uint64), y.view(np.uint64))
        rec = dict(n=A.shape[0], nnz=int(A.nnz), lcc_n=ref.shape[0], lcc_nnz=int(ref.nnz), cf=cf, dim=dim,
                   bit_equal=bool(equal), scipy_lcc_ms=scipy_ms,
                   fused={k: median(fr, k) for k in fr[0]}, composed={k: median(cr, k) for k in cr[0]},
                   fused_runs=fr, composed_runs=cr, component_kernels=kernel_times(ctx, A))
        rec["fused_minus_composed_ms"] = rec["fused"]["wall_ms"] - rec["composed"]["wall_ms"]
        result["graphs"][name] = rec
        print(name, json.dumps({k: rec[k] for k in ("n", "lcc_n", "bit_equal", "scipy_lcc_ms", "fused",
                                                     "composed")}), flush=True)
    ctx.close()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()

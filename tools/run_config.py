"""One-off full-size runs of the BASELINE configs through ge_embed (single GPU):
  python tools/run_config.py config3 | config5 [n_points] | config2 | config1  [--ref] [--cpu-ref]
--ref      use the hierarchy of the REFERENCE's partitioner cached under tests/golden/refhier_*.npz
           (config3: R-MAT-20; config5: Delaunay of n_points = 1000000) instead of the
           stand-in generator graphs.coarsen
--gpus=N   one context over N GPUs of the box (large levels sharded by aggregates)
--cpu-ref  also time the compiled reference's embed() (oracle/_ref, all host threads) on the same
           hierarchy -- minutes of CPU
Prints one JSON line: hierarchy shape, embed() wall time, per-phase times, properties."""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry

entry.load_package()
from graph_embed_b200 import capi, graphs


def build(name, arg):
    if name == "config1":
        return graphs.grid2d(100, 100), 0.25, 2
    if name == "config2":
        return graphs.rgg(100_000, 10.0, seed=12345), 0.25, 2
    if name == "config3":
        return graphs.rmat(int(arg or 20), 16, seed=1), 0.25, 3
    if name == "config5":
        return graphs.delaunay3d(int(arg or 4_000_000), seed=1), 0.125, 3
    raise SystemExit("unknown config")


def main():
    flags = [a for a in sys.argv[1:] if a.startswith("--")]
    pos = [a for a in sys.argv[1:] if not a.startswith("--")]
    name = pos[0]
    arg = pos[1] if len(pos) > 1 else None
    use_ref = "--ref" in flags
    t = time.time()
    if use_ref:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from helpers import load_ref_hierarchy
        key = {"config3": "rmat20", "config5": "delaunay%d" % int(arg or 1_000_000)}[name]
        As, Ps, meta = load_ref_hierarchy(graphs, key)
        A, cf, dim = As[0], meta["cf"], 3
        t_gen, t_coarsen = time.time() - t, meta["partition_seconds"]
    else:
        A, cf, dim = build(name, arg)
        t_gen = time.time() - t
        t = time.time()
        As, Ps = graphs.coarsen(A, cf, min_coarse=64)
        t_coarsen = time.time() - t
    stats = graphs.level_stats(As, Ps)
    gpu_list = [1]
    for f in flags:
        if f.startswith("--gpus="):
            gpu_list = [int(v) for v in f.split("=")[1].split(",")]
    # --gpus=N[,M...]: one context over N GPUs (ge_context_create_multi); large levels are sharded
    # by aggregates.  The first entry is the run the main figures describe; every entry is listed
    # under "scaling" (same hierarchy, same process).
    scaling = []
    for gi, g in enumerate(gpu_list):
        c = capi.Context(0) if g == 1 else capi.Context(devices=list(range(g)))
        c.embed(As[-2:], Ps[-1:], dim, seed=1, coarse_iterations=100)  # warm-up (context, pool)
        c.embed(As, Ps, dim, seed=0, coarse_iterations=100)            # warm-up (NCCL channels, pools of every device)
        w = []
        for rep in range(2):   # seed 0: the reference's own (std::random_device) mode
            t = time.time()
            xg, sg = c.embed(As, Ps, dim, seed=0)
            w.append(time.time() - t)
        scaling.append({"gpus": g, "embed_wall_s": min(w), "coarse_ms": sg["coarse_ms"], "levels_ms": sg["levels_ms"],
                        "grid_tier_ms": sg["grid_tier_ms"], "device_radii_ms": sg["device_radii_ms"],
                        "finite": bool(np.isfinite(xg).all())})
        if gi == 0:
            ctx, x, st, walls = c, xg, sg, w
        else:
            c.close()
    gpus = gpu_list[0]
    t = time.time()
    ctx.embed(As, Ps, dim, seed=1)
    wall_seeded = time.time() - t
    # the same hierarchy's coarse graphs rebuilt on the device (ge_galerkin), level by level
    gal = {"device_ms": 0.0, "total_ms": 0.0, "segments_global": 0, "exact": True}
    for l, P in enumerate(Ps):
        ctx.galerkin(As[l], P)  # first call at this size grows the memory pool
        C, gs = ctx.galerkin(As[l], P, with_stats=True)
        gal["device_ms"] += gs["device_ms"]
        gal["total_ms"] += gs["total_ms"]
        gal["segments_global"] += gs["segments_global"]
        gal["exact"] = bool(gal["exact"] and np.array_equal(C.indptr, As[l + 1].indptr)
                            and np.array_equal(C.indices, As[l + 1].indices)
                            and np.array_equal(C.data, As[l + 1].data))
    v_A = capi.vertex_to_aggregate(Ps[0])
    cent = np.zeros((Ps[0].shape[0], dim))
    np.add.at(cent, v_A, x)
    cent /= np.diff(Ps[0].indptr)[:, None]
    spread = float(np.linalg.norm(x - cent[v_A], axis=1).mean())
    extent = float(np.linalg.norm(x - x.mean(0), axis=1).max())
    cpu = None
    if "--cpu-ref" in flags:
        O = entry.load_oracle()
        threads = len(os.sched_getaffinity(0))
        fd = os.dup(1)
        os.dup2(2, 1)   # the reference prints progress lines on stdout
        try:
            _, secs = O.ref_embed(As, Ps, dim, seed=1, nthreads=threads, kind="fast")
        finally:
            os.dup2(fd, 1)
            os.close(fd)
        cpu = {"embed_wall_s": secs, "threads": threads, "kind": "reference (oracle/_ref, -O3, OpenMP)"}
    out = {"config": name, "gpus": gpus, "scaling": scaling, "hierarchy": ("reference partitioner (src/partitioner.cpp:1550-1893), cached"
                                         if use_ref else "stand-in generator graphs.coarsen"),
           "cpu_reference": cpu, "grid_tier_ms": st["grid_tier_ms"], "device_radii_ms": st["device_radii_ms"],
           "grid_tier_share_of_levels": st["grid_tier_ms"] / max(st["levels_ms"], 1e-9),
           "n": A.shape[0], "nnz": int(A.nnz), "dim": dim, "coarsening": cf,
           "levels": [s["n"] for s in stats], "max_aggregate": [s["max_size"] for s in stats],
           "pairs_per_iteration": [s["pairs"] for s in stats],
           "embed_wall_s": min(walls), "embed_wall_s_fixed_seed": wall_seeded, "coarse_ms": st["coarse_ms"], "levels_ms": st["levels_ms"],
           "host_radii_ms": st["host_radii_ms"], "kernel_launches": st["kernel_launches"],
           "pair_interactions": st["pair_interactions"], "edge_visits": st["edge_visits"],
           "galerkin_all_levels": gal, "finite": bool(np.isfinite(x).all()), "aggregate_spread_over_extent": spread / extent,
           "host_generate_s": t_gen, "host_coarsen_s": t_coarsen}
    print(json.dumps(out))


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py -- ForceAtlas iterations/s and pair-interactions/s on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR] [--workload ...]

Workload (config.workload): BASELINE config 4, the flat single-level ForceAtlas iteration on a
500 000-vertex random geometric graph (avg degree 10), all-pairs repulsion, d = 2, FP64 like the
reference.  It is the configuration the metric (iterations/s, pair-interactions/s at 1/2/4/8 B200)
is quoted on, it fits one GPU, and it is the path that shards (row blocks + one coordinate
all-gather per iteration), so the same workload is measured at every N ("scaling": "strong").
A step = one ForceAtlas iteration (include/forceatlas.hpp:146-270) over the whole graph.
At N = 1 the same run also reports embed() wall time on BASELINE config 2 (RGG 100k, multilevel,
d = 2) under "embed", and the FP32 variant of the flat kernels under "fp32".

One JSON line on stdout (rank 0); everything else goes to stderr.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry  # noqa: E402


def log(*a):
    print(*a, file=sys.stderr, flush=True)


class stdout_to_stderr:
    """The reference prints progress lines on std::cout (src/embed.cpp:583, 613); keep the
    process's stdout for the one JSON line by pointing fd 1 at stderr while reference code runs."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def __exit__(self, *exc):
        try:
            import ctypes
            ctypes.CDLL(None).fflush(None)
        except Exception:
            pass
        os.dup2(self.saved, 1)
        os.close(self.saved)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "MEASURED_PEAKS.json (driver-measured copy bandwidth)"
    return 6650.0, "fallback of B200_PROFILING.md (MEASURED_PEAKS.json absent)"


def algorithmic(n, nnz, dim, w):
    """SURVEY.md section 8d: 5d+4 flops per ordered pair; attraction+step bytes per iteration =
    nnz*(4+w) [indices+weights] + n*(4 + w + 5*d*w) [indptr, mass; own coords, repulsion sum,
    previous force read; new coords, previous force written]."""
    return dict(pairs=float(n) * (n - 1), flops_per_pair=5 * dim + 4,
                step_bytes=float(nnz) * (4 + w) + float(n) * (4 + w + 5 * dim * w))


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons during the timed region (pynvml, 100 ms)."""
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
            0x4: "sw_power_cap", 0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            while not self.stop_flag:
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                r = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(
                    pynvml, "nvmlDeviceGetCurrentClocksEventReasons") else \
                    pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in self.BITS.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.1)
        except Exception as e:  # pragma: no cover
            self.reasons.add("sampler_error:%s" % type(e).__name__)

    def result(self):
        self.stop_flag = True
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def flat_graph(n, seed=7):
    entry.load_package()
    from graph_embed_b200 import graphs
    t = time.time()
    A = graphs.rgg(n, 10.0, seed=seed)
    log("[bench] rgg n=%d nnz=%d (%.1fs)" % (A.shape[0], A.nnz, time.time() - t))
    return A


# ------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation (oracle/_ref), all host threads
# ------------------------------------------------------------------------------------------------
def cpu_flat_rate(O, dim, n_sample, iters, threads, kind):
    """pair-interactions/s of partition::forceAtlas on an n_sample-vertex graph of the same
    generator; returns (rate, seconds)."""
    from graph_embed_b200 import graphs
    A = graphs.rgg(n_sample, 10.0, seed=7)
    n = A.shape[0]
    x0 = O.mt_uniform(23, n * dim).reshape(n, dim)
    t = time.time()
    if kind == "reference":
        O.ref_flat(A, dim, x0, O.Params(iterations=iters), nthreads=threads, kind="fast")
    else:
        O.flat_run(A, dim, x0, O.Params(iterations=iters))
    dt = time.time() - t
    return float(n) * (n - 1) * iters / dt, dt, n


def host_threads():
    """Threads the CPU arm uses: every core this process may run on.  torchrun exports
    OMP_NUM_THREADS=1 into its workers, so omp_get_max_threads() is not the box's core count
    there; the affinity mask is."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:  # pragma: no cover
        return max(1, os.cpu_count() or 1)


REF_ITERS_PER_STEP = 2  # the same sample shape in --impl reference and in cpu_baseline


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    entry.load_package()
    O = entry.load_oracle()
    kind = "reference" if O.ref_available("fast") else "port"
    threads = host_threads() if kind == "reference" else 1
    n_sample = args.ref_n
    for _ in range(min(args.warmup, 1)):
        cpu_flat_rate(O, args.dim, n_sample, 1, threads, kind)
    t_total, pairs_total, n_eff = 0.0, 0.0, 0
    for _ in range(args.steps):
        rate, dt, n_eff = cpu_flat_rate(O, args.dim, n_sample, REF_ITERS_PER_STEP, threads, kind)
        t_total += dt
        pairs_total += rate * dt
    value = pairs_total / t_total
    sample = ("flat forceAtlas, %d iterations per step on a %d-vertex RGG (avg degree 10) from the "
              "same generator as the %d-vertex workload (a direct run is ~100 s per iteration); "
              "pair-interactions/s is size-independent for the O(n^2) kernel, so the rate is "
              "quoted for the workload's n" % (REF_ITERS_PER_STEP, n_eff, args.n))
    line = {"impl": "reference", "metric": "forceatlas_pair_interactions_per_sec", "value": value,
            "unit": "pair-interactions/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "iters_per_sec_at_workload_n": value / (float(args.n) * (args.n - 1)),
            "config": dict(workload_config(args), reference_sample_n=n_eff,
                           reference_iterations_per_step=REF_ITERS_PER_STEP,
                           reference_threads=threads),
            "cpu_baseline": {"value": value, "unit": "pair-interactions/s", "cores": threads,
                             "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "pair-interactions/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def workload_config(args):
    return {"workload": "config4: flat single-level ForceAtlas, RGG n=%d avg degree 10, all-pairs "
                        "repulsion, dim=%d" % (args.n, args.dim),
            "n": args.n, "dim": args.dim, "avg_degree": 10,
            "parallelism": ("single GPU" if args.gpus == 1 else
                            "row-block x%d + coordinate all-gather per iteration" % args.gpus
                            if (getattr(args, "ordered", False) or args.n < 32768) else
                            "unordered pairs shared x%d (reduce-scatter of pair sums) + row-block x%d "
                            "attraction/step + coordinate all-gather per iteration" % (args.gpus, args.gpus)),
            "l2": "flushed between timed steps (256 MiB device write outside the timed events)"}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    entry.load_package()
    from graph_embed_b200 import capi, graphs, sharding

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the CUDA path is the only path (no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node N for --gpus N"
    dev = torch.device("cuda", local)
    # a non-default stream: the library launches on it, torch/NCCL order against it, and the CUDA
    # events of the timed region are recorded on it (torch.cuda.Event sees only this stream)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    ctx = capi.Context(local, stream=stream.cuda_stream)

    A = flat_graph(args.n)
    n, nnz, dim = A.shape[0], A.nnz, args.dim
    prec = capi.GE_F64
    w = 8
    alg = algorithmic(n, nnz, dim, w)
    params = capi.flat_params(precision=prec)
    x0 = capi.reference_uniform(23, n * dim).reshape(n, dim)

    # row blocks: ld is a multiple of 256, hence of every N in {1,2,4,8}
    r0, r1, R, probe_ld = sharding.row_block(n, world, rank)
    # N > 1: symmetric plan -- each rank evaluates 1/N of the unordered pairs over the full length,
    # one reduce-scatter of the pair sums, then attraction + step on its row block, one all-gather
    # of the new coordinates.  --ordered keeps the ordered row-block sweep (no reduce-scatter).
    sym_ranks = world > 1 and not args.ordered and n >= 32768  # below: ordered row-block plans
    if sym_ranks:
        plan = ctx.flat_plan(A, dim, params, symmetric=(rank, world))
        assert plan.rows == (r0, r1)
    else:
        plan = ctx.flat_plan(A, dim, params, rows=(r0, r1))
    ld = plan.ld
    assert ld == probe_ld
    tdt = torch.float64
    bufs = [torch.zeros(dim * ld, dtype=tdt, device=dev) for _ in range(2)]
    plan.bind_coords(bufs[0].data_ptr(), bufs[1].data_ptr())
    plan.upload(x0)
    ptr_to_buf = {bufs[0].data_ptr(): bufs[0], bufs[1].data_ptr(): bufs[1]}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    sums = None
    if sym_ranks:
        sums = torch.zeros(dim * ld, dtype=tdt, device=dev)
        plan.bind_pair_sums(sums.data_ptr())

    def one_step():
        if sym_ranks:
            plan.launch_repulsion()
            sharding.reduce_scatter_pair_sums(dist, sums.view(dim, ld), rank, R)
            plan.launch_step()
        else:
            plan.launch_iteration()
        if world > 1:  # in-place: own slice sits at rank*R of the output
            sharding.allgather_coords(dist, ptr_to_buf[plan.next_ptr()].view(dim, ld), rank, R)
        plan.swap()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        one_step()
    barrier()

    sampler = ClockSampler(local)
    sampler.start()
    launches0 = ctx.launches
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    t_wall = time.time()
    for s in range(args.steps):
        flush.fill_(s & 0xFF)  # evict L2 between timed steps (outside the event pair)
        ev[s][0].record(stream)
        one_step()
        ev[s][1].record(stream)
    barrier()
    t_wall = time.time() - t_wall
    launches = ctx.launches - launches0
    ms = sum(a.elapsed_time(b) for a, b in ev)
    clocks = sampler.result()
    if args.dump_outputs and rank == 0:
        outputs = {"coords": plan.download()}
        if world == 1:  # at N > 1 each rank holds the forces of its own rows only
            outputs["forces"] = plan.download_forces()
        dump_outputs(args.dump_outputs, outputs)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    ms_per_step = ms / args.steps
    value = alg["pairs"] * args.steps / (ms * 1e-3)

    # ---- per-kernel device time (CUDA events inside the library, on the launching stream) -------
    plan.profile(True)
    for _ in range(3):
        flush.fill_(1)
        one_step()
    barrier()
    prof = plan.profile_get()
    plan.profile(False)
    rep_ms = prof["repulsion_ms"] / max(prof["repulsion_launches"], 1)
    step_ms = prof["attract_step_ms"] / max(prof["attract_step_launches"], 1)
    rows_frac = (r1 - r0) / float(n)
    hbm_peak, hbm_src = measured_peaks()
    out = None
    if rank == 0:
        fp64_peak = ctx.fma_peak_tflops(capi.GE_F64)
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            traffic = json.load(open(tpath)).get(
                "%s_f64_d%d_bytes_per_launch" % ("k_repulsion_sym" if plan.symmetric else "k_repulsion", dim))
        rep_flops = alg["pairs"] * rows_frac * alg["flops_per_pair"]
        roof = {"kernel": "%s<double,%d>%s" % ("k_repulsion_sym" if plan.symmetric else "k_repulsion", dim,
                                                " (+ k_sym_reduce)" if plan.symmetric else ""),
                "bound": "fp64", "unit": "TFLOP/s",
                "achieved": rep_flops / (rep_ms * 1e-3) / 1e12, "peak": fp64_peak,
                "peak_source": "measured live: ge_measure_fma_peak (independent DFMA chains, all SMs, CUDA events)",
                "traffic": traffic, "ms_per_launch": rep_ms, "share_of_step": rep_ms / (rep_ms + step_ms),
                "pairs_per_launch": alg["pairs"] * rows_frac, "flops_per_pair": alg["flops_per_pair"]}
        roof["frac"] = roof["achieved"] / roof["peak"]
        step_bytes = alg["step_bytes"] * rows_frac
        roof2 = {"kernel": "k_attract_step_staged<double,%d>" % dim, "bound": "hbm", "unit": "GB/s",
                 "achieved": step_bytes / (step_ms * 1e-3) / 1e9, "peak": hbm_peak, "peak_source": hbm_src,
                 "traffic": None, "ms_per_launch": step_ms, "bytes_per_launch": step_bytes}
        roof2["frac"] = roof2["achieved"] / roof2["peak"]
        out = {"metric": "forceatlas_pair_interactions_per_sec", "value": value,
               "unit": "pair-interactions/s", "n_gpus": world, "steps": args.steps,
               "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
               "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
               "iters_per_sec": 1e3 / ms_per_step, "wall_s_timed_region": t_wall,
               "config": workload_config(args), "gpu_launches": launches, "clocks": clocks,
               "roofline": roof, "roofline_attraction": roof2}

    # ---- parity at this N (outside the timed region) ---------------------------------------------
    parity = bench_parity(args, torch, dist, capi, ctx, plan, A, x0, params, world, rank, r0, r1, one_step, barrier, dev)
    if rank == 0:
        out.update(parity)

    # ---- e2e: host buffers in, host buffers out, every step -------------------------------------
    e2e = bench_e2e(args, torch, dist, capi, sharding, ctx, plan, A, x0, world, rank, R, ptr_to_buf, ld, alg, barrier, one_step)
    if rank == 0:
        out["e2e"] = e2e

    if rank == 0 and world == 1:
        out["fp32"] = bench_fp32(args, capi, ctx, A, x0, alg)
        if not args.no_attraction:
            out["roofline_attraction_large"] = bench_attraction_large(args, capi, ctx, graphs, hbm_peak, hbm_src)
        if not args.no_embed:
            out["embed"] = bench_embed(args, capi, ctx, graphs)
        if not args.no_embed:
            out["embed_config1"] = bench_embed_config1(args, capi, ctx, graphs)
        if not args.no_embed and not args.no_refhier:
            out["embed_config3"] = bench_embed_refhier(args, capi, ctx, graphs)
        if not args.no_galerkin:
            out["galerkin"] = bench_galerkin(args, capi, ctx, graphs, hbm_peak, hbm_src)
        if not args.no_cpu:
            out["cpu_baseline"] = bench_cpu_baseline(args)
    if rank == 0:
        print(json.dumps(out), flush=True)
    plan.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if parity["parity_max_err"] > PARITY_TOL or not parity["parity_ok"]:
        log("[bench] PARITY FAILURE: %r" % (parity,))
        sys.exit(3)


DUMP_BYTES = 60 << 20  # under 64 MB in all, .npy headers included


def dump_outputs(path, arrays):
    """Writes each n-row array as <path>/<name>.npy (float64).  Above DUMP_BYTES in all, the same
    fixed, seeded sample of rows is written for every array, with the row indices as rows.npy."""
    os.makedirs(path, exist_ok=True)
    n = next(iter(arrays.values())).shape[0]
    row_bytes = sum(a[0].nbytes for a in arrays.values())
    if n * row_bytes > DUMP_BYTES:
        k = DUMP_BYTES // (row_bytes + 8)
        rows = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))
        arrays = dict({name: a[rows] for name, a in arrays.items()}, rows=rows.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))
    log("[bench] outputs of the last timed step written to %s: %s" % (path, sorted(arrays)))


PARITY_TOL = 1e-10  # FP64 forces, relative to the vertex's conditioning scale (tests/helpers.py)


def bench_parity(args, torch, dist, capi, ctx, plan, A, x0, params, world, rank, r0, r1, one_step, barrier, dev):
    """One more step from the known state x0, checked on every rank: the forces of sampled owned
    rows against the CPU oracle (include/forceatlas.hpp:148-212 restated, oracle/ -- the checker,
    never the thing measured), the positions of those rows against the oracle's forces pushed
    through the step formula (:244-261), and at N > 1 every position against a single-GPU plan of
    the same graph on rank 0.  The errors are max-reduced over the ranks."""
    O = entry.load_oracle()
    n, dim = A.shape[0], args.dim
    plan.upload(x0)
    barrier()
    one_step()
    barrier()
    F = plan.download_forces()   # owned rows, forces of the step just taken
    x1 = plan.download()         # all rows (gathered)
    per_rank = max(4, 32 // world)
    rng = np.random.default_rng(1234 + rank)
    rows = np.sort(rng.choice(np.arange(r0, r1), size=min(per_rank, r1 - r0), replace=False))
    ferr = xerr = 0.0
    p = O.Params()
    for r in rows:
        Fr, S = O.flat_forces(A, dim, x0, p, rows=(int(r), int(r) + 1))
        f, sc = Fr[r], max(S[r], 1e-300)
        ferr = max(ferr, float(np.linalg.norm(F[r - r0] - f) / sc))
        # step (:244-261) from zero previous forces: swing = |f|, speed = ks / (1 + sqrt(swing)),
        # capped at ksmax / |f|
        fn = float(np.sqrt((f * f).sum()))
        speed = p.ks * p.tolerate / (1.0 + p.tolerate * np.sqrt(fn))
        if fn > 0:
            speed = min(speed, p.ksmax / fn)
        xr = x0[r] + f * speed
        # a force error of 1e-10*scale moves the vertex by at most speed * that
        xerr = max(xerr, float(np.linalg.norm(x1[r] - xr) / max(speed * sc, 1e-300)))
    t = torch.tensor([ferr, xerr], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ferr, xerr = float(t[0].item()), float(t[1].item())
    out = {"parity_max_err": max(ferr, xerr), "parity_force_err": ferr, "parity_position_err": xerr,
           "parity_rows_checked": int(per_rank * world), "parity_tolerance": PARITY_TOL,
           "parity_vs_single_gpu_plan": None, "parity_ok": True}
    if world > 1:
        ok = 1.0
        if rank == 0:  # the same step on ONE GPU: positions of every vertex
            single = ctx.flat_plan(A, dim, params)
            single.upload(x0)
            single.iterate(1)
            xs = single.download()
            single.close()
            extent = float(np.abs(xs).max())
            d = float(np.abs(x1 - xs).max() / extent)
            out["parity_vs_single_gpu_plan"] = d
            ok = 1.0 if d < 1e-9 else 0.0
        t = torch.tensor([ok], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        out["parity_ok"] = bool(t.item() > 0.5)
    log("[bench] parity: %r" % (out,))
    return out


def bench_e2e(args, torch, dist, capi, sharding, ctx, plan, A, x0, world, rank, R, ptr_to_buf, ld, alg, barrier, one_step):
    """Same metric through the public host-buffer API, host<->device copies inside the timed
    region.  N = 1: ge_flat_forceatlas (the forceAtlas drop-in: graph + coordinates in from pinned
    host memory, coordinates out), one call per step.  N > 1: the row-block plan API with the
    coordinates uploaded and downloaded every step (the graph stays resident)."""
    n, dim = A.shape[0], args.dim
    steps = max(2, min(args.steps, 5))
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
    x = pin(x0.copy())
    h0, d0 = ctx.bytes_moved
    if world == 1:
        import scipy.sparse as sp
        Ap = sp.csr_matrix((pin(A.data), pin(A.indices), pin(A.indptr)), shape=A.shape)
        p1 = capi.flat_params(iterations=1)
        for _ in range(3):  # warm-up (memory pools, staging rings)
            ctx.flat_forceatlas(Ap, dim, x, p1)
        barrier()
        h0, d0 = ctx.bytes_moved
        t = time.time()
        for _ in range(steps):
            ctx.flat_forceatlas(Ap, dim, x, p1, inplace=True)
        dt = time.time() - t
        note = "ge_flat_forceatlas(host CSR, host coords, iterations=1) per step"
    else:
        # N > 1: the same public call, ge_flat_forceatlas, on a context that owns all N GPUs
        # (ge_context_create_multi: one process, NCCL inside the library).  Rank 0 makes the call;
        # the other ranks' processes hold their GPUs idle behind the barriers.
        import scipy.sparse as sp
        dt = 0.0
        note = ("ge_flat_forceatlas(host CSR, host coords, iterations=1) per step on a %d-GPU context "
                "(ge_context_create_multi), called from rank 0" % world)
        # the other ranks wait on a CPU (gloo) barrier: an NCCL barrier would park a spinning kernel
        # on their GPUs, which rank 0's context is about to use
        cpu_group = dist.new_group(backend="gloo")
        barrier()
        if rank == 0:
            mctx = capi.Context(devices=list(range(world)))
            Ap = sp.csr_matrix((pin(A.data), pin(A.indices), pin(A.indptr)), shape=A.shape)
            p1 = capi.flat_params(iterations=1)
            for _ in range(3):  # warm-up (NCCL channels, memory pools of every device)
                mctx.flat_forceatlas(Ap, dim, x, p1)
            h0, d0 = mctx.bytes_moved
            t = time.time()
            for _ in range(steps):
                mctx.flat_forceatlas(Ap, dim, x, p1, inplace=True)
            dt = time.time() - t
            h1, d1 = mctx.bytes_moved
            mctx.close()
        dist.barrier(group=cpu_group)
        tt = torch.tensor([dt, 0.0, 0.0], dtype=torch.float64, device="cuda")
        if rank == 0:
            tt[1], tt[2] = (h1 - h0) / steps, (d1 - d0) / steps
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt[0].item())
        return {"value": alg["pairs"] * steps / dt, "unit": "pair-interactions/s", "steps": steps,
                "ms_per_step": 1e3 * dt / steps, "h2d_bytes_per_step": float(tt[1].item()),
                "d2h_bytes_per_step": float(tt[2].item()), "api": note, "host_memory": "pinned"}
    tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dt = float(tt.item())
    h1, d1 = ctx.bytes_moved
    return {"value": alg["pairs"] * steps / dt, "unit": "pair-interactions/s", "steps": steps,
            "ms_per_step": 1e3 * dt / steps, "h2d_bytes_per_step": (h1 - h0) / steps,
            "d2h_bytes_per_step": (d1 - d0) / steps, "api": note, "host_memory": "pinned"}


def bench_fp32(args, capi, ctx, A, x0, alg):
    """FP32 variant of the same kernels (reduced precision: reported beside, never as, the headline)."""
    n, dim = A.shape[0], args.dim
    plan = ctx.flat_plan(A, dim, capi.flat_params(precision=capi.GE_F32))
    plan.upload(x0)
    plan.iterate(3)
    plan.sync()
    plan.profile(True)
    plan.iterate(5)
    prof = plan.profile_get()
    kname = "k_repulsion_sym<float,%d> (+ k_sym_reduce)" if plan.symmetric else "k_repulsion<float,%d>"
    plan.close()
    rep_ms = prof["repulsion_ms"] / prof["repulsion_launches"]
    step_ms = prof["attract_step_ms"] / prof["attract_step_launches"]
    peak = ctx.fma_peak_tflops(capi.GE_F32)
    ach = alg["pairs"] * alg["flops_per_pair"] / (rep_ms * 1e-3) / 1e12
    return {"dtype": "f32", "pair_interactions_per_sec": alg["pairs"] / ((rep_ms + step_ms) * 1e-3),
            "iters_per_sec": 1e3 / (rep_ms + step_ms),
            "roofline": {"kernel": kname % dim, "bound": "fp32", "unit": "TFLOP/s",
                         "achieved": ach, "peak": peak, "frac": ach / peak, "ms_per_launch": rep_ms,
                         "peak_source": "measured live: ge_measure_fma_peak"}}


def bench_attraction_large(args, capi, ctx, graphs, hbm_peak, hbm_src):
    """The CSR attraction + step kernel alone on a graph whose arrays exceed L2 (n = 2M-vertex RGG,
    ~20M entries, ~0.5 GB of algorithmic traffic): achieved HBM GB/s against the measured copy bandwidth."""
    n = args.attr_n
    t = time.time()
    A = graphs.rgg(n, 10.0, seed=11)
    n, nnz = A.shape[0], A.nnz
    log("[bench] attraction graph n=%d nnz=%d (%.1fs)" % (n, nnz, time.time() - t))
    out = {}
    for prec, w, name, dim in ((capi.GE_F64, 8, "f64", 3), (capi.GE_F32, 4, "f32", 3), (capi.GE_F64, 8, "f64_d2", 2)):
        plan = ctx.flat_plan(A, dim, capi.flat_params(precision=prec))
        plan.upload(capi.reference_uniform(5, n * dim).reshape(n, dim))
        plan.select_kernels(2)  # attraction + step only: 4e12 ordered pairs per repulsion pass here
        plan.iterate(2)
        plan.sync()
        plan.profile(True)
        plan.iterate(5)
        prof = plan.profile_get()
        plan.close()
        ms = prof["attract_step_ms"] / prof["attract_step_launches"]
        b = algorithmic(n, nnz, dim, w)["step_bytes"]
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if w == 8 and dim == 3 and n > 1_900_000 and os.path.exists(tpath):
            traffic = json.load(open(tpath)).get("k_attract_step_f64_d3_n2m_bytes_per_launch")
        out[name] = {"kernel": "k_attract_step_staged<%s,%d>" % ("double" if w == 8 else "float", dim), "bound": "hbm",
                     "graph": "RGG n=%d avg degree 10 (the graph the launch shape was tuned on)" % n,
                     "traffic": traffic,
                     "unit": "GB/s", "achieved": b / (ms * 1e-3) / 1e9, "peak": hbm_peak,
                     "frac": b / (ms * 1e-3) / 1e9 / hbm_peak, "peak_source": hbm_src, "ms_per_launch": ms,
                     "bytes_per_launch": b, "n": n, "nnz": nnz, "edge_visits_per_sec": nnz / (ms * 1e-3)}
    # held-out graphs: not used for any tuning decision (another generator, another degree
    # distribution); same frozen launch heuristics
    held = []
    t = time.time()
    held.append(("heldout_delaunay3d", "Delaunay tetrahedralisation, %d points (avg degree ~15.5)" % args.heldout_n,
                 graphs.delaunay3d(args.heldout_n, seed=3)))
    held.append(("heldout_rmat", "R-MAT scale %d, edge factor 16, largest component (power-law rows)" % args.heldout_rmat,
                 graphs.rmat(args.heldout_rmat, 16, seed=5)))
    log("[bench] held-out attraction graphs (%.1fs)" % (time.time() - t))
    for key, desc, H in held:
        hn, hnnz = H.shape[0], H.nnz
        for dim in (2, 3):
            plan = ctx.flat_plan(H, dim, capi.flat_params(precision=capi.GE_F64))
            plan.upload(capi.reference_uniform(5, hn * dim).reshape(hn, dim))
            plan.select_kernels(2)
            plan.iterate(2)
            plan.sync()
            plan.profile(True)
            plan.iterate(5)
            prof = plan.profile_get()
            plan.close()
            ms = prof["attract_step_ms"] / prof["attract_step_launches"]
            b = algorithmic(hn, hnnz, dim, 8)["step_bytes"]
            out["%s_f64_d%d" % (key, dim)] = {
                "kernel": "k_attract_step*<double,%d>" % dim, "bound": "hbm", "graph": desc, "traffic": None,
                "unit": "GB/s", "achieved": b / (ms * 1e-3) / 1e9, "peak": hbm_peak,
                "frac": b / (ms * 1e-3) / 1e9 / hbm_peak, "peak_source": hbm_src, "ms_per_launch": ms,
                "bytes_per_launch": b, "n": hn, "nnz": hnnz, "edge_visits_per_sec": hnnz / (ms * 1e-3)}
    return out


def bench_galerkin(args, capi, ctx, graphs, hbm_peak, hbm_src):
    """SURVEY section 8 row f3: the Galerkin coarse graph P_T A P_T^T (examples/embedder.cpp:213-216)
    of one level of a 1M-vertex RGG on the device, against its compulsory HBM bytes, next to the
    oracle's row-by-row accumulation on one host core."""
    t = time.time()
    A = graphs.rgg(args.galerkin_n, 10.0, seed=13)
    As, Ps = graphs.coarsen(A, 0.25, min_coarse=1000, max_levels=1)
    P = Ps[0]
    n, m, nnz = A.shape[0], P.shape[0], A.nnz
    log("[bench] galerkin level n=%d -> m=%d nnz=%d (%.1fs)" % (n, m, nnz, time.time() - t))
    ctx.galerkin(A, P)  # warm-up (pool, kernel attributes)
    best = None
    for _ in range(3):
        C, st = ctx.galerkin(A, P, with_stats=True)
        if best is None or st["device_ms"] < best["device_ms"]:
            best = st
    assert np.array_equal(C.indptr, As[1].indptr) and np.array_equal(C.indices, As[1].indices)
    assert np.array_equal(C.data, As[1].data)
    b = nnz * 12.0 + n * 16.0 + m * 12.0 + C.nnz * 12.0  # A once, row pointers / maps, A_c once
    out = {"kernel": "k_gal_warp / k_gal_segment (+ scan, k_gal_compact)", "bound": "hbm", "unit": "GB/s", "n": n, "m": m,
           "nnz": nnz, "nnz_out": int(C.nnz), "device_ms": best["device_ms"], "total_ms": best["total_ms"],
           "bytes": b, "achieved": b / (best["device_ms"] * 1e-3) / 1e9, "peak": hbm_peak,
           "peak_source": hbm_src, "entries_per_sec": nnz / (best["device_ms"] * 1e-3),
           "segments_shared": best["segments_shared"], "segments_global": best["segments_global"],
           "kernel_launches": best["kernel_launches"]}
    out["frac"] = out["achieved"] / hbm_peak
    if not args.no_cpu:
        O = entry.load_oracle()
        t = time.time()
        O.galerkin(A, P)
        out["cpu_port_ms"] = 1e3 * (time.time() - t)
        out["cpu_port_cores"] = 1
    return out


def bench_embed(args, capi, ctx, graphs):
    """BASELINE config 2: embed() wall time, bracketed like examples/embedder.cpp:219-222
    (hierarchy already built, coordinates returned to the host)."""
    t = time.time()
    A = graphs.rgg(100_000, 10.0, seed=12345)
    As, Ps = graphs.coarsen(A, 0.25, min_coarse=100)
    log("[bench] config2 hierarchy %s (%.1fs)" % ([a.shape[0] for a in As], time.time() - t))
    ctx.embed(As, Ps, 2, seed=1, coarse_iterations=1000)  # warm-up
    walls, st = [], None
    for rep in range(3):   # seed 0 = the reference's own mode (std::random_device)
        t = time.time()
        x, st = ctx.embed(As, Ps, 2, seed=0)
        walls.append(time.time() - t)
    assert np.isfinite(x).all()
    wall = float(np.median(walls))
    t = time.time()
    ctx.embed(As, Ps, 2, seed=1)  # fixed seed: the reference's mt19937 stream is reproduced on the host
    wall_seeded = time.time() - t
    out = {"workload": "config2: RGG n=%d avg degree 10, multilevel embed, dim=2, coarsening 0.25, "
                       "levels %s" % (As[0].shape[0], [a.shape[0] for a in As]),
           "embed_wall_s": wall, "embed_wall_s_fixed_seed": wall_seeded,
           "pair_interactions": st["pair_interactions"],
           "pair_interactions_per_sec": st["pair_interactions"] / wall,
           "iterations": 100000 + 100 * len(Ps), "iters_per_sec": (100000 + 100 * len(Ps)) / wall,
           "coarse_ms": st["coarse_ms"], "levels_ms": st["levels_ms"], "host_radii_ms": st["host_radii_ms"],
           "kernel_launches": st["kernel_launches"], "h2d_bytes": st["h2d_bytes"], "d2h_bytes": st["d2h_bytes"]}
    if not args.no_cpu:
        O = entry.load_oracle()
        if O.ref_available("fast"):
            threads = host_threads()
            best = None
            for nt in sorted({1, threads}):
                with stdout_to_stderr():
                    _, secs = O.ref_embed(As, Ps, 2, seed=1, nthreads=nt, kind="fast")
                if best is None or secs < best[0]:
                    best = (secs, nt)
            out["cpu_reference_embed_wall_s"], out["cpu_reference_threads"] = best
    return out


def bench_embed_config1(args, capi, ctx, graphs):
    """BASELINE config 1 (configs[0], the reference's own CPU-runnable case): the pipeline of
    examples/embedder.cpp on a 100 x 100 grid, coarsening 0.25, d = 2, hierarchy from the
    reference's own partitioner (tests/golden/config1_grid100.npz); embed() wall time next to the
    compiled reference on this box's host cores."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import load_config1_golden
    As, Ps, z = load_config1_golden(graphs)
    ctx.embed(As, Ps, 2, seed=0, coarse_iterations=1000)  # warm-up
    walls, st = [], None
    for rep in range(3):
        t = time.time()
        x, st = ctx.embed(As, Ps, 2, seed=0)
        walls.append(time.time() - t)
    assert np.isfinite(x).all()
    out = {"workload": "config1: 100x100 grid, coarsening 0.25, dim=2, hierarchy of the reference partitioner, "
                       "levels %s" % [a.shape[0] for a in As],
           "embed_wall_s": float(np.median(walls)), "coarse_ms": st["coarse_ms"], "levels_ms": st["levels_ms"],
           "device_radii_ms": st["device_radii_ms"], "kernel_launches": st["kernel_launches"],
           "pair_interactions": st["pair_interactions"], "h2d_bytes": st["h2d_bytes"], "d2h_bytes": st["d2h_bytes"]}
    if not args.no_cpu:
        O = entry.load_oracle()
        if O.ref_available("fast"):
            best = None
            for nt in sorted({1, host_threads()}):   # the reference is slower multi-threaded on small levels
                with stdout_to_stderr():
                    _, secs = O.ref_embed(As, Ps, 2, seed=1, nthreads=nt, kind="fast")
                if best is None or secs < best[0]:
                    best = (secs, nt)
            out["cpu_reference_embed_wall_s"], out["cpu_reference_threads"] = best
    return out


def bench_embed_refhier(args, capi, ctx, graphs):
    """BASELINE config 3 on the hierarchy of the REFERENCE's own partitioner (R-MAT scale 20,
    largest component, coarsening 0.25, d = 3; tests/golden/refhier_rmat20.npz): embed() wall time
    with the device-side phases.  The compiled reference's embed() on the same hierarchy takes
    minutes (profiles/r02_config3_rmat20_ref.json: 213.7 s on 16 host threads) and is not re-run
    here."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import load_ref_hierarchy
    t = time.time()
    As, Ps, meta = load_ref_hierarchy(graphs, "rmat20")
    log("[bench] config3 reference hierarchy %s (%.1fs)" % ([a.shape[0] for a in As], time.time() - t))
    ctx.embed(As, Ps, 3, seed=0, coarse_iterations=1000)  # warm-up
    walls, st = [], None
    for rep in range(3):
        t = time.time()
        x, st = ctx.embed(As, Ps, 3, seed=0)
        walls.append(time.time() - t)
    assert np.isfinite(x).all()
    sizes = [int(np.diff(P.indptr).max()) for P in Ps]
    pairs = [float((np.diff(P.indptr).astype(np.int64) * (np.diff(P.indptr) - 1)).sum()) for P in Ps]
    ref_s, ref_threads = None, None
    prof = os.path.join(ROOT, "profiles", "r02_config3_rmat20_ref.json")
    if os.path.exists(prof):
        d = json.load(open(prof))
        if d.get("cpu_reference"):
            ref_s, ref_threads = d["cpu_reference"]["embed_wall_s"], d["cpu_reference"]["threads"]
    return {"workload": "config3: R-MAT scale 20 largest component (n=%d, %d entries), hierarchy of the "
                        "reference partitioner, multilevel embed, dim=3" % (As[0].shape[0], As[0].nnz),
            "levels": [a.shape[0] for a in As], "max_aggregate": sizes, "pairs_per_iteration": pairs,
            "embed_wall_s": float(np.median(walls)), "coarse_ms": st["coarse_ms"], "levels_ms": st["levels_ms"],
            "grid_tier_ms": st["grid_tier_ms"], "device_radii_ms": st["device_radii_ms"],
            "host_radii_ms": st["host_radii_ms"], "h2d_bytes": st["h2d_bytes"], "d2h_bytes": st["d2h_bytes"],
            "pair_interactions": st["pair_interactions"],
            "pair_interactions_per_sec": st["pair_interactions"] / float(np.median(walls)),
            "kernel_launches": st["kernel_launches"],
            "cpu_reference_embed_wall_s_recorded": ref_s, "cpu_reference_threads_recorded": ref_threads,
            "cpu_reference_source": "profiles/r02_config3_rmat20_ref.json (tools/run_config.py config3 --ref --cpu-ref)"}


def bench_cpu_baseline(args):
    """The reference's own flat forceAtlas (oracle/_ref, -O3, OpenMP, all host threads) on a bounded
    sample of the same workload, ~10-30 s of CPU work."""
    O = entry.load_oracle()
    kind = "reference" if O.ref_available("fast") else "port"
    threads = host_threads() if kind == "reference" else 1
    cpu_flat_rate(O, args.dim, 6000, 1, threads, kind)      # warm the thread pool / page in the library
    # the same sample as `--impl reference` (args.ref_n vertices, 2 iterations per step, 2 steps)
    t_total, pairs_total, n = 0.0, 0.0, 0
    for _ in range(2):
        rate, dt, n = cpu_flat_rate(O, args.dim, args.ref_n, REF_ITERS_PER_STEP, threads, kind)
        t_total += dt
        pairs_total += rate * dt
    return {"value": pairs_total / t_total, "unit": "pair-interactions/s", "cores": threads, "kind": kind,
            "seconds": t_total,
            "sample": "flat forceAtlas, 2 steps of %d iterations on a %d-vertex RGG (avg degree 10) of the "
                      "same generator (the --impl reference sample); the O(n^2) kernel's pair rate is "
                      "size-independent" % (REF_ITERS_PER_STEP, n)}


def main():
    # stdout carries exactly one JSON line: everything else that writes to fd 1 (NCCL's version
    # banner, the reference's progress lines) is pointed at stderr for the life of the process.
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(json_fd, "w")
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=500_000)
    ap.add_argument("--dim", type=int, default=2)
    ap.add_argument("--ref-n", type=int, default=30_000)
    ap.add_argument("--attr-n", type=int, default=2_000_000)
    ap.add_argument("--heldout-n", type=int, default=1_000_000, help="points of the held-out Delaunay graph")
    ap.add_argument("--heldout-rmat", type=int, default=20, help="scale of the held-out R-MAT graph")
    ap.add_argument("--ordered", action="store_true",
                    help="N > 1: ordered row-block sweep instead of the symmetric pair shares")
    ap.add_argument("--no-embed", action="store_true")
    ap.add_argument("--no-refhier", action="store_true", help="skip config 3 on the reference hierarchy")
    ap.add_argument("--no-galerkin", action="store_true")
    ap.add_argument("--galerkin-n", type=int, default=1_000_000)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-attraction", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the coordinates (and at N = 1 the forces) of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native large-steps hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload plane1000|...] [--dump-outputs DIR]

metric   : from_differential solves/sec @ 1M verts  (BASELINE.json)
step     : one from_differential solve of a (V,3) right-hand side (forward solve of the optimisation step)
workload : BASELINE config 3 -- plane 1000x1000 (V = 1,000,000, nnz(M) = 6,992,002), uniform Laplacian, alpha = 0.95,
           3-RHS Jacobi-PCG to rtol 1e-7 from a cold start -- one mesh per GPU (seed = rank) at every N: weak scaling,
           no collective on the solve path (SURVEY.md 8e); NCCL only gathers a checksum at the end.
value    : whole-job solves/s with the right-hand sides already in HBM (CUDA events, max over ranks)
e2e      : same through the public API with HOST (pinned) buffers: H2D of u and D2H of v inside the timed region
roofline : the HBM figure of record is the SpMV (BASELINE metric part 2): the stand-alone in-solver SpMM+dot kernel timed
           alone with CUDA events, rotating over 4 copies of matrix + vectors (336 MB > 126 MB L2) so every launch streams
           from HBM; algorithmic bytes 8 nnz + 4 (V+1) + 8 k V (SURVEY 8d).  The solve kernel (one launch per solve, the
           dominant kernel of the timed region) is reported beside it as `solve_kernel`: it is L2-resident by construction
           (pattern-only matrix copy + shared-memory residency), so its DRAM traffic -- measured by ncu, source file named --
           is far below any algorithmic byte model and an HBM fraction would be meaningless; its byte model and time are given.
cpu_baseline / --impl reference : the reference's path on the box's host cores: the C/OpenMP port of its
           ConjugateGradientSolver (threads chosen around the cgroup CPU quota, median of 3) and the SuperLU direct solve that
           stands in for its default cholespy/CHOLMOD CholeskySolver (1 core, factorisation untimed); the faster one is `value`.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "large-steps-pytorch_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "from_differential solves/sec @1M verts"
WORKLOADS = {
    "plane1000": dict(kind="plane", n=1000, alpha=0.95, desc="plane 1000x1000, V=1000000, nnz=6992002, uniform L, alpha=0.95 (BASELINE config 3)"),
    "plane500": dict(kind="plane", n=500, alpha=0.95, desc="plane 500x500, V=250000, nnz=1746002, uniform L, alpha=0.95 (BASELINE config 4, one per GPU)"),
    "plane2000": dict(kind="plane", n=2000, alpha=0.95, desc="plane 2000x2000, V=4000000, uniform L, alpha=0.95 (working set >> L2)"),
    "icosphere": dict(kind="ico", level=4, lam=10.0, desc="icosphere level 4, V=2562, uniform L, lambda=10 (BASELINE config 1)"),
    "bunny": dict(kind="bunny", lam=19.0, desc="bunny.obj subdivided x2, V=52786, cot L, lambda=19 (BASELINE config 2)"),
}
RTOL = 1e-7


def build_mesh(wl, seed):
    from largesteps_b200 import workloads as W
    if wl["kind"] == "plane":
        v, f = W.plane(wl["n"], seed=seed)
        return v, f, dict(lambda_=1.0, alpha=wl["alpha"])
    if wl["kind"] == "ico":
        v, f = W.icosphere(wl["level"])
        return v, f, dict(lambda_=wl["lam"])
    d = np.load(os.path.join(ROOT, "tests", "golden", "bunny_mesh.npz"))
    v, f = W.subdivide(*W.subdivide(d["verts"], d["faces"].astype(np.int64)))
    return v.astype(np.float32), f, dict(lambda_=wl["lam"], cotan=True)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed regions (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.proc = None
        self.path = f"/tmp/ls_clocks_{os.getpid()}.csv"
        self.gpu = gpu_index

    def start(self):
        try:
            self.fh = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=self.fh, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()           # exact PID we started
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.fh.close()
        sm, mx, pw = [], [], []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        seen = set()
        for line in open(self.path):
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
                pw.append(float(parts[2]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    seen.add(nm)
        try:
            os.remove(self.path)
        except OSError:
            pass
        if sm:
            out = {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(seen),
                   "samples": len(sm), "power_w_max": max(pw)}
        return out


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def shared_config(wl_name, wl, V, nnz):
    """Identical in both arms, so that the driver can tell they ran the same workload."""
    return {"workload": wl_name, "desc": wl["desc"], "V": int(V), "nnz": int(nnz), "rhs_columns": 3, "rtol": RTOL,
            "l2": "4 rotating right-hand sides; the GPU solve's working set is L2-resident by design (pattern-only matrix "
                  "copy), the stand-alone SpMV is timed HBM-cold by rotating 4 matrix+vector copies (336 MB > 126 MB L2)"}


def cpu_reference_leg(v, f, kw, bs, repeats=3, warm=False):
    """The reference's solve path on this box's host cores, both ports, each `repeats` times (median + spread):
       (a) C/OpenMP port of ConjugateGradientSolver (oracle/cg_port.c; abs tol 1e-5 as in the reference), threads chosen
           around the cgroup CPU quota and pinned; cold start unless `warm` (the reference keeps its previous solution),
       (b) SuperLU fp32 symmetric-mode direct solve, 1 core, factorisation untimed: stand-in for cholespy/CHOLMOD."""
    import oracle
    from oracle.cport import CPortCG, host_cpu_budget, pin_to_allowed_cores
    budget = host_cpu_budget()
    r, c, val, V = oracle.compute_matrix(v, f, **kw)
    cg = CPortCG(r, c, val, V)
    cg.autotune_threads(bs[1 % len(bs)])
    pinned = pin_to_allowed_cores(cg.threads)
    cg.guess_fwd = None
    cg.solve(bs[1 % len(bs)])                   # untimed: first-touch page faults, thread pool
    t_cgs = []
    for i in range(repeats):
        if not warm:
            cg.guess_fwd = None
        t0 = time.perf_counter()
        cg.solve(bs[i % len(bs)])
        t_cgs.append(time.perf_counter() - t0)
    t0 = time.perf_counter()
    ds = oracle.DirectSolver(r, c, val, V, dtype=np.float32)
    t_fac = time.perf_counter() - t0
    t_dss = []
    for i in range(repeats):
        t0 = time.perf_counter()
        ds.solve(bs[i % len(bs)])
        t_dss.append(time.perf_counter() - t0)
    med = statistics.median
    return {"cg": cg, "ds": ds, "V": V, "nnz": len(val), "t_cg": t_cgs, "t_ds": t_dss, "t_fac": t_fac, "budget": budget,
            "pinned_cpus": len(pinned) if pinned else None,
            "record": {"reference_cg_port": {"solves_per_s": 1.0 / med(t_cgs), "median_s": med(t_cgs), "min_s": min(t_cgs),
                                             "max_s": max(t_cgs), "cores": cg.threads, "iterations_per_axis": cg.iters,
                                             "note": "oracle/cg_port.c: C/OpenMP restatement of the reference CG (fp32, absolute tol 1e-5), "
                                                     + ("warm starts" if warm else "cold start")},
                       "direct_solve": {"solves_per_s": 1.0 / med(t_dss), "median_s": med(t_dss), "min_s": min(t_dss),
                                        "max_s": max(t_dss), "cores": 1, "factor_s": t_fac, "factor_nnz": ds.factor_nnz,
                                        "note": "scipy SuperLU fp32 symmetric mode: stand-in for cholespy/CHOLMOD (not installable offline)"},
                       "cpu": cpu_model(), "host_cores": os.cpu_count(), "affinity_cpus": budget["affinity_cpus"],
                       "cgroup_cpu_max": budget["cgroup_cpu_max"], "quota_cores": budget["quota_cores"],
                       "pinned_cpus": len(pinned) if pinned else None}}


def run_reference(args, wl, wl_name):
    """CPU arm: the reference's path restated on the host (the reference itself is Python + an un-installable wheel).
    Both CPU ports are measured (median of 3); the faster one runs the K timed steps.  The SuperLU figure is printed every time."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    v, f, kw = build_mesh(wl, seed=0)
    import oracle
    r, c, val, V = oracle.compute_matrix(v, f, **kw)
    A = oracle.coo_to_scipy(r, c, val, V, dtype=np.float32)
    rng = np.random.default_rng(100)
    bs = [(A @ (v + rng.normal(0, 0.01, v.shape).astype(np.float32))).astype(np.float32) for _ in range(2)]
    leg = cpu_reference_leg(v, f, kw, bs, repeats=3, warm=True)
    cg, ds = leg["cg"], leg["ds"]
    t_cg, t_ds = statistics.median(leg["t_cg"]), statistics.median(leg["t_ds"])
    use_cg = t_cg < t_ds
    step = (lambda i: cg.solve(bs[i % 2])) if use_cg else (lambda i: ds.solve(bs[i % 2]))
    for i in range(args.warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        x_last = step(i)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "solution.npy"), np.asarray(x_last, dtype=np.float32))
    val_sps = args.steps / dt
    cores = cg.threads if use_cg else 1
    sample = (f"{args.steps} solves of a (V,3) fp32 RHS at V={V} with the faster of two CPU ports of the reference: "
              f"{'C/OpenMP port of its ConjugateGradientSolver (abs tol 1e-5, warm starts) on ' + str(cg.threads) + ' pinned threads' if use_cg else 'SuperLU direct solve (stand-in for cholespy/CHOLMOD), 1 core'}"
              f"; probes (median of 3): CG port {t_cg:.3f} s, direct {t_ds:.3f} s after an untimed {leg['t_fac']:.1f} s factorisation")
    cb = dict(leg["record"])
    cb.update({"value": val_sps, "unit": "solves/s", "cores": cores, "kind": "port", "sample": sample})
    line = {
        "impl": "reference", "metric": METRIC, "value": val_sps, "unit": "solves/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": shared_config(wl_name, wl, V, len(val)),
        "solver": "CPU port of the reference path: " + ("ConjugateGradientSolver (C/OpenMP)" if use_cg else "direct solve (SuperLU)"),
        "cpu_baseline": cb,
        "e2e": {"value": val_sps, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def run_b200(args, wl, wl_name):
    import torch
    import torch.distributed as dist
    from largesteps_b200 import _native as N, distributed as D
    from largesteps_b200.geometry import compute_matrix
    from largesteps_b200.parameterize import to_differential, from_differential, _cache
    from largesteps_b200.solvers import PCGSolver

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a GPU (there is no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    N.lib()

    # ---- setup (untimed): one mesh per rank -----------------------------------------------------------
    v, f, kw = build_mesh(wl, seed=rank)
    V = v.shape[0]
    tv = torch.from_numpy(v).to(dev)
    tf = torch.from_numpy(f).to(dev)
    M = compute_matrix(tv, tf, **kw)              # first call pays library / context warm-up and the allocator's first cudaMallocs
    torch.cuda.synchronize()
    del M                                         # as in a remesh: the old matrix is dropped, its blocks return to torch's caching allocator
    t0 = time.perf_counter()
    M = compute_matrix(tv, tf, **kw)              # steady-state assembly time (round 1 timed this with the first M still alive:
    torch.cuda.synchronize()                      #  ~250 MB of fresh cudaMalloc inside the timed region, 28.6 ms instead of ~2 ms)
    t_assemble = time.perf_counter() - t0
    nnz = M._nnz()
    R = 4
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    us = []
    for i in range(R):
        vv = tv + 0.01 * torch.randn(V, 3, device=dev, generator=gen)
        us.append((to_differential(M, vv) + 0.01 * torch.randn(V, 3, device=dev, generator=gen)).contiguous())
    t0 = time.perf_counter()
    x = from_differential(M, us[0], "Cholesky")          # builds + caches the solver handle
    torch.cuda.synchronize()
    t_first = time.perf_counter() - t0
    solver = _cache[(id(M), "Cholesky")][0]

    def timed(fn, steps, warmup):
        for i in range(warmup):
            fn(i)
        torch.cuda.synchronize()
        D.barrier()
        n0 = N.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        D.barrier()
        ms = e0.elapsed_time(e1)
        return D.max_over_ranks(ms, device=dev), N.launch_count() - n0

    sampler = ClockSampler(local)       # every rank watches its own GPU (VERDICT r1: per-rank clock skew was unobserved)
    sampler.start()
    time.sleep(0.3)

    # ---- value: device-resident right-hand sides ---------------------------------------------------------
    iters = []
    last = {}

    def step_dev(i):
        with torch.no_grad():
            x = from_differential(M, us[i % R], "Cholesky")     # asynchronous: one persistent-kernel launch per solve
        if i == args.steps - 1:
            last["x"] = x

    ms_total, launches = timed(step_dev, args.steps, args.warmup)
    x_last = last.pop("x").cpu()                                # what the last timed step returned (for --dump-outputs)
    for i in range(R):                                          # iteration counts per right-hand side (untimed)
        with torch.no_grad():
            from_differential(M, us[i], "Cholesky")
        iters.append(solver.iterations)
        solver.raise_for_status()
    it_mean = float(np.mean(iters))
    value = world * args.steps / (ms_total * 1e-3)

    # ---- fwd+bwd pairs (what one optimiser step does: scripts/main.py:173,206) ---------------------------
    gsmall = [(1e-4 * torch.randn(V, 3, device=dev, generator=gen)) for _ in range(2)]

    def step_pair(i):
        u = us[i % R].detach().requires_grad_(True)
        xx = from_differential(M, u, "Cholesky")
        xx.backward(gsmall[i % 2])

    pair_steps = max(3, args.steps // 4)
    ms_pair, _ = timed(step_pair, pair_steps, min(args.warmup, 3))
    pairs_per_s = world * pair_steps / (ms_pair * 1e-3)

    # ---- e2e: host buffers through the public API ----------------------------------------------------------
    # Every step copies its right-hand side from pinned host memory, solves, and copies the solution back.  Two independent
    # pipelines (stream + matrix object with its own solver handle + device/host buffers) alternate, so the copies of one step
    # overlap the solve of the other on the copy engines -- the solves themselves cannot overlap (each occupies all 148 SMs).
    # `e2e_serial` is the same thing on one stream (copy -> solve -> copy, nothing overlapped).
    h_in = [u.cpu().pin_memory() for u in us]
    M_b = compute_matrix(tv, tf, **kw)
    with torch.no_grad():
        from_differential(M_b, us[0], "Cholesky")
    pipes = []
    for Mx in (M, M_b):
        pipes.append({"M": Mx, "stream": torch.cuda.Stream(device=dev), "d_u": torch.empty(V, 3, dtype=torch.float32, device=dev),
                      "h_out": torch.empty(V, 3, dtype=torch.float32).pin_memory()})

    def step_serial(i):
        pp = pipes[0]
        with torch.no_grad():
            pp["d_u"].copy_(h_in[i % R], non_blocking=True)
            xx = from_differential(pp["M"], pp["d_u"], "Cholesky")
            pp["h_out"].copy_(xx, non_blocking=True)

    ms_ser, _ = timed(step_serial, args.steps, args.warmup)

    def timed_pipelined(steps, warmup):
        def one(i):
            pp = pipes[i % 2]
            with torch.cuda.stream(pp["stream"]), torch.no_grad():
                pp["d_u"].copy_(h_in[i % R], non_blocking=True)
                xx = from_differential(pp["M"], pp["d_u"], "Cholesky")
                pp["h_out"].copy_(xx, non_blocking=True)
        for i in range(warmup):
            one(i)
        torch.cuda.synchronize()
        D.barrier()
        cur = torch.cuda.current_stream(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(cur)
        for pp in pipes:
            pp["stream"].wait_event(e0)
        for i in range(steps):
            one(i)
        for pp in pipes:
            cur.wait_stream(pp["stream"])
        e1.record(cur)
        torch.cuda.synchronize()
        D.barrier()
        return D.max_over_ranks(e0.elapsed_time(e1), device=dev)

    ms_e2e = timed_pipelined(args.steps, args.warmup)
    e2e_value = world * args.steps / (ms_e2e * 1e-3)
    e2e_serial = world * args.steps / (ms_ser * 1e-3)
    bytes_io = V * 3 * 4
    with torch.no_grad():                      # the pipelined results are the real solutions
        last = args.steps - 1
        ref_x = from_differential(M, h_in[last % R].to(dev), "Cholesky")
        chk_pipe = float((pipes[last % 2]["h_out"].to(dev) - ref_x).abs().max())
    del M_b

    # ---- BASELINE config 4: 8 independent 250K-vertex meshes, mesh i -> rank i mod N, aggregate solves/s -----------
    cfg4 = None
    if not args.no_config4:
        wl4 = WORKLOADS["plane500"]
        mine = D.assign(8, rank, world)
        items = []
        for i in mine:
            v4, f4, kw4 = build_mesh(wl4, seed=i)
            t4 = torch.from_numpy(v4).to(dev)
            M4 = compute_matrix(t4, torch.from_numpy(f4).to(dev), **kw4)
            u4 = (to_differential(M4, t4) + 0.01 * torch.randn(t4.shape[0], 3, device=dev, generator=gen)).contiguous()
            from_differential(M4, u4, "Cholesky")
            items.append((M4, u4, v4))
        reps4 = 10

        def step4(i):
            with torch.no_grad():
                for (M4, u4, _) in items:
                    from_differential(M4, u4, "Cholesky")

        ms4, _ = timed(step4, reps4, 3)
        with torch.no_grad():
            err4 = max(float((from_differential(M4, to_differential(M4, torch.from_numpy(v4).to(dev)), "Cholesky").cpu()
                              - torch.from_numpy(v4)).norm() / torch.from_numpy(v4).norm()) for (M4, _, v4) in items[:1]) if items else 0.0
        cfg4 = {"workload": "plane500", "desc": wl4["desc"], "meshes": 8, "meshes_per_rank": len(mine),
                "solves_per_s": 8 * reps4 / (ms4 * 1e-3), "ms_per_round_of_8": ms4 / reps4,
                "roundtrip_rel_l2_first_mesh": err4,
                "how": "each rank solves its share of the 8 meshes back to back; CUDA events, max over ranks; no collective on the solve path"}
        del items

    # ---- roofline ---------------------------------------------------------------------------------------------
    # HBM figure of record: the stand-alone in-solver SpMM+dot kernel (BASELINE metric part 2), CUDA events over 400 launches
    # issued from C, rotating over 4 copies of matrix + vectors = 336 MB > L2, so every launch streams from HBM.
    # The solve kernel (dominant kernel of the timed region, one launch per solve) is described beside it.
    roof = None
    extra_more = {}
    if rank == 0:
        from largesteps_b200.solvers import bench_kernels
        desc = solver.describe()
        peak, peak_src = measured_peak()
        k = 3
        b_spmm = solver.spmm_bytes(k)
        extra_h = [PCGSolver(M) for _ in range(3)]
        handles = [solver] + extra_h
        L = 400

        def time_kernels(which, hs):
            bench_kernels(hs, which, 8)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            bench_kernels(hs, which, L)
            e1.record()
            torch.cuda.synchronize()
            return 1e3 * e0.elapsed_time(e1) / L

        us_cold_dot = time_kernels(0, handles)          # SpMM + p.Ap epilogue, as the graph-mode CG iteration launches it
        us_hot_dot = time_kernels(0, handles[:1])
        us_cold = time_kernels(4, handles)              # the plain SpMV y = A x of BASELINE's metric (same kernel, no dot epilogue)
        us_hot = time_kernels(4, handles[:1])
        spmv_kernel = "lsk::spmm_sell_tma_kernel<3,DOT=false,...> (SELL-32 entry stream staged by cp.async.bulk into per-warp shared-memory rings)"
        if os.environ.get("LS_SELL_TMA") == "0":
            spmv_kernel = "lsk::spmm_sell_kernel<3,DOT>"
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "spmv_traffic.json")
        if os.path.exists(tp) and wl_name == "plane1000":
            try:
                tj = json.load(open(tp))
                traffic, traffic_src = tj["dram_bytes_per_launch"], tj.get("source")
            except Exception:
                pass
        roof = {"bound": "hbm", "achieved": b_spmm / (us_cold * 1e-6) / 1e9, "peak": peak, "unit": "GB/s",
                "frac": b_spmm / (us_cold * 1e-6) / 1e9 / peak, "traffic": traffic, "traffic_source": traffic_src,
                "kernel": spmv_kernel, "algorithmic_bytes": b_spmm, "us_per_launch": us_cold, "l2_resident_us_per_launch": us_hot,
                "peak_source": peak_src,
                "how": "CUDA events over 400 back-to-back launches from C (programmatic dependent launch) rotating over 4 matrix+vector "
                       "copies (336 MB > L2); bytes = 8 nnz + 4 (V+1) + 8 k V (SURVEY 8d)",
                "with_dot_epilogue": {"us_per_launch": us_cold_dot, "l2_resident_us_per_launch": us_hot_dot,
                                      "frac": b_spmm / (us_cold_dot * 1e-6) / 1e9 / peak,
                                      "note": "same kernel + deterministic grid reduction of p.Ap (what a graph-mode CG iteration launches)"}}
        # the solve kernel: L2-resident by design -- say so with numbers instead of an HBM fraction
        t_solve_s = ms_total * 1e-3 / args.steps
        pat = desc.get("sell_engine") == 2
        b_iter = (4 * (nnz - V) + 4 * V if pat else 8 * nnz) + 32 * V + 48 * V     # matrix stream, z write+gather, p and x read+write
        st_traffic, st_src = None, None
        tp2 = os.path.join(ROOT, "profiles", "solve_traffic.json")
        if os.path.exists(tp2) and wl_name == "plane1000":
            try:
                tj = json.load(open(tp2))
                st_traffic, st_src = tj["dram_bytes_per_launch"], tj.get("source")
            except Exception:
                pass
        roof["solve_kernel"] = {
            "kernel": "lsf::pcg_fused_kernel<3,RES=%d,...> (whole solve, 1 launch)" % desc.get("residency", -1) if desc.get("algo") == "fused"
                      else "lsp::pcg_persistent_kernel (round-1 kernel)",
            "us_per_launch": 1e6 * t_solve_s, "cg_iterations": it_mean, "us_per_iteration": 1e6 * t_solve_s / max(it_mean, 1),
            "bound": "L2 / latency (working set L2-resident: pattern-only matrix copy 4 B/entry, r/s/D^-1 in shared memory)",
            "algorithmic_bytes_per_iteration": b_iter, "algorithmic_GBs": it_mean * b_iter / t_solve_s / 1e9,
            "dram_bytes_per_launch": st_traffic, "dram_traffic_source": st_src,
            "note": "algorithmic_GBs may exceed the HBM peak because the data never leaves L2; it is NOT an HBM roofline fraction",
            "solver": desc}
        if wl_name == "plane1000" and not args.no_spmv_4m:
            # SURVEY 8(d): the same kernel on a plane whose working set is far beyond L2 (2000 x 2000: V = 4e6, 336 MB per launch)
            v4, f4, kw4 = build_mesh(WORKLOADS["plane2000"], seed=0)
            tv4, tf4 = torch.from_numpy(v4).to(dev), torch.from_numpy(f4).to(dev)
            M4 = compute_matrix(tv4, tf4, **kw4)
            s4 = PCGSolver(M4)
            us4 = time_kernels(4, [s4])
            b4 = s4.spmm_bytes(k)
            with torch.no_grad():
                s4.solve(to_differential(M4, tv4))
                t0 = time.perf_counter()
                s4.solve(to_differential(M4, tv4))
                torch.cuda.synchronize()
                t4m = time.perf_counter() - t0
            roof["spmv_4M"] = {"workload": WORKLOADS["plane2000"]["desc"], "algorithmic_bytes": b4, "us_per_launch": us4,
                               "achieved_GBs": b4 / (us4 * 1e-6) / 1e9, "frac": b4 / (us4 * 1e-6) / 1e9 / peak,
                               "solve_ms": 1e3 * t4m, "solve_iterations": s4.iterations,
                               "how": "CUDA events over 400 back-to-back launches from C; 336 MB per launch >> 126 MB L2"}
            del s4, M4, tv4, tf4
        if desc.get("persistent"):
            # per-phase SM cycles of the solve kernel (profiling instantiation of the same kernel, CTA 0)
            os.environ["LS_PCG_PROFILE"] = "1"
            try:
                solver.solve(us[0])
                pc = solver.phase_cycles()
            finally:
                del os.environ["LS_PCG_PROFILE"]
            itn = max(pc["iterations"], 1)
            roof["solve_kernel"]["phase_cycles_per_iteration"] = {kk: round(vv / itn) for kk, vv in pc.items() if kk not in ("_", "_0", "iterations")}
        del extra_h, handles

        # ---- the other BASELINE configs and the section 8(f) rows, so that the driver sees them -----------------------
        def solve_ms(Mx, ux, reps=50):
            sx = _cache[(id(Mx), "Cholesky")][0] if (id(Mx), "Cholesky") in _cache else None
            with torch.no_grad():
                from_differential(Mx, ux, "Cholesky")
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(reps):
                    from_differential(Mx, ux, "Cholesky")
                e1.record()
                torch.cuda.synchronize()
            sx = _cache[(id(Mx), "Cholesky")][0]
            return e0.elapsed_time(e1) / reps, sx.iterations, sx.describe()

        for cname, wname in (("config1_icosphere", "icosphere"), ("config2_bunny", "bunny")):
            vv_, ff_, kw_ = build_mesh(WORKLOADS[wname], seed=0)
            tvx, tfx = torch.from_numpy(vv_).to(dev), torch.from_numpy(ff_).to(dev)
            Mx = compute_matrix(tvx, tfx, **kw_)
            ux = (to_differential(Mx, tvx) + 0.01 * torch.randn(tvx.shape[0], 3, device=dev, generator=gen)).contiguous()
            msx, itx, dx = solve_ms(Mx, ux)
            extra_more[cname] = {"V": int(tvx.shape[0]), "solve_ms": msx, "iterations": itx, "us_per_iteration": 1e3 * msx / max(itx, 1),
                                 "cluster": dx.get("cluster"), "grid": dx.get("grid")}
            if wname == "bunny":
                # config 5 stand-in: Tutorial-shaped loop (two solves + fused AdamUniform per step, no renderer) at 52.8K
                from largesteps_b200.optimize import AdamUniform
                target = (tvx * (1.0 + 0.3 * torch.sin(3 * tvx[:, :1]) * torch.cos(2 * tvx[:, 1:2]))).detach()
                uu = to_differential(Mx, tvx).clone().requires_grad_(True)
                opt = AdamUniform([uu], lr=0.01)

                def loop(n):
                    for _ in range(n):
                        xx = from_differential(Mx, uu, "Cholesky")
                        loss = ((xx - target) ** 2).mean()
                        opt.zero_grad()
                        loss.backward()
                        opt.step()

                loop(20)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                loop(500)
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                extra_more["config5_loop_standin"] = {"V": int(tvx.shape[0]), "steps": 500, "it_per_s": 500 / dt,
                                                      "note": "from_differential -> MSE loss -> backward -> AdamUniform; no renderer (nvdiffrast needs GL)"}
            del Mx
        # re-parameterisation after a remesh (8 f4): assemble + solver build + first solve, arena reused
        from largesteps_b200.remesh import Reparameterizer
        for nm, nplane in (("250K", 500), ("1M", 1000)):
            vv_, ff_ = build_mesh(WORKLOADS["plane500" if nplane == 500 else "plane1000"], seed=3)[:2]
            tvx, tfx = torch.from_numpy(vv_).to(dev), torch.from_numpy(ff_).to(dev)
            rp = Reparameterizer(lambda_=1.0, alpha=0.95)
            Mx, ux = rp.update(tvx, tfx)                      # first call sizes the arena
            with torch.no_grad():
                from_differential(Mx, ux)
            ts = []
            for _ in range(3):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                Mx, ux = rp.update(tvx, tfx)
                with torch.no_grad():
                    from_differential(Mx, ux)
                torch.cuda.synchronize()
                ts.append(time.perf_counter() - t0)
            extra_more["reparameterize_" + nm] = {"ms_median": 1e3 * statistics.median(ts), "ms_min": 1e3 * min(ts),
                                                  "what": "Reparameterizer.update (assembly + to_differential + solver build) + first from_differential, wall clock"}
            del rp, Mx, ux

    clocks = sampler.stop()
    if world > 1:
        import torch.distributed as tdist
        allc = [None] * world
        tdist.all_gather_object(allc, clocks)            # outside every timed region
        if rank == 0:
            meds = [c["sm_mhz"] for c in allc if c and c.get("sm_mhz") is not None]
            clocks = {"sm_mhz": min(meds) if meds else None,
                      "sm_max_mhz": max([c["sm_max_mhz"] for c in allc if c and c.get("sm_max_mhz")] or [None]),
                      "reasons": sorted(set(r for c in allc if c for r in c.get("reasons", []))),
                      "samples": sum(c.get("samples", 0) for c in allc if c),
                      "what": "sm_mhz = lowest per-rank median under load; reasons = union over ranks",
                      "per_rank": [{"rank": i, "sm_mhz": c.get("sm_mhz"), "reasons": c.get("reasons"),
                                    "power_w_max": c.get("power_w_max")} for i, c in enumerate(allc) if c]}

    # ---- trivial gather (the only collective): checksum of every rank's last solution ---------------------
    with torch.no_grad():
        xs = from_differential(M, us[0], "Cholesky")
    chk = D.gather_solutions(xs.double().sum(dim=0, keepdim=True).float())

    # ---- CPU baseline beside it (rank 0, N = 1 only) ------------------------------------------------------
    cpu = None
    parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        b_host = [us[0].cpu().numpy(), us[1].cpu().numpy()]
        leg = cpu_reference_leg(v, f, kw, b_host, repeats=3, warm=False)
        xd = leg["ds"].solve(b_host[0]).astype(np.float64)
        parity = float(np.linalg.norm(xs.cpu().numpy().astype(np.float64) - xd) / np.linalg.norm(xd))
        t_cg, t_ds = statistics.median(leg["t_cg"]), statistics.median(leg["t_ds"])
        use_cg = t_cg < t_ds
        cpu = dict(leg["record"])
        cpu.update({"value": max(1.0 / t_cg, 1.0 / t_ds), "unit": "solves/s", "cores": leg["cg"].threads if use_cg else 1, "kind": "port",
                    "sample": (f"median of 3 single (V,3) fp32 solves at V={V}: C/OpenMP port of the reference CG on {leg['cg'].threads} "
                               f"pinned threads, cold start ({t_cg:.3f} s) vs SuperLU direct solve, 1 core ({t_ds:.3f} s after an untimed "
                               f"{leg['t_fac']:.1f} s factorisation; stand-in for cholespy/CHOLMOD); the faster is `value`")})

    if rank == 0:
        extra = {"fwd_bwd_pairs_per_s": pairs_per_s, "us_per_cg_iteration": 1e3 * (ms_total / args.steps) / max(it_mean, 1),
                 "assembly_ms": 1e3 * t_assemble, "first_solve_incl_solver_build_ms": 1e3 * t_first,
                 "parity_rel_l2_vs_cpu_direct": parity, "checksums": chk.flatten().tolist()[:6], "config4": cfg4}
        extra.update(extra_more)
        line = {
            "metric": METRIC, "value": value, "unit": "solves/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": shared_config(wl_name, wl, V, nnz),
            "solver": "Jacobi-PCG, cold start, one fused persistent kernel per solve; cg_iterations_mean=%.1f; %d independent mesh(es), "
                      "one per GPU, no collective on the solve path" % (it_mean, world),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "solves/s", "h2d_bytes_per_step": bytes_io, "d2h_bytes_per_step": bytes_io,
                    "ms_per_step": ms_e2e / args.steps, "serial_one_stream_value": e2e_serial,
                    "how": "two alternating pipelines (stream + solver handle + buffers each): the H2D/D2H copies of one step overlap "
                           "the solve of the other; serial_one_stream_value = copy -> solve -> copy on one stream",
                    "max_abs_diff_last_result_vs_device_resident_solve": chk_pipe},
            "gpu_launches": int(launches),
            "roofline": roof,
            "cpu_baseline": cpu,
            "extra": extra,
        }
        print(json.dumps(line))
    if rank == 0 and args.dump_outputs:
        # the solution (V, 3) of the last timed step, for output-for-output comparison of two builds on the same inputs
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "solution.npy"), x_last.numpy().astype(np.float32))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=os.environ.get("LS_BENCH_WORKLOAD", "plane1000"), choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-spmv-4m", action="store_true", help="skip the 4M-vertex SpMV roofline measurement")
    ap.add_argument("--no-config4", action="store_true", help="skip the config-4 sub-record (8 x 250K meshes over the ranks)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the solution of the last one to DIR/solution.npy (float32, V x 3)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        return run_reference(args, wl, args.workload)
    return run_b200(args, wl, args.workload)


if __name__ == "__main__":
    sys.exit(main())

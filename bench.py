#!/usr/bin/env python
"""bench.py -- V-cycles/s of the B200 AMG solve-phase engine on BASELINE.json's configurations.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg3|cfg2|cfg4|cfg5]
                    [--grid G] [--configs cfg2,cfg5,cfg4] [--dump-outputs DIR]

Headline workload (config.workload): BASELINE.json configs[2] -- gallery.poisson((256,256,256)) 7-pt fp64,
ruge_stuben_solver hierarchy (classical strength 0.25, RS splitting, classical interpolation), multi-colour
Gauss-Seidel (symmetric, gauss_seidel_indexed over colour-sorted rows) pre and post, 'pinv' coarse solve;
rhs = default_rng(20260922).random(n), x0 = 0.  The hierarchy is built by this repo's host-side setup
(pyamg_b200.classical: 28 s instead of ~150 s with the reference; validated to reproduce the reference's
hierarchies, tests/test_setup.py).  At N = 1 the same line carries, under `configs`, BASELINE configs[1] (cfg2),
configs[4] (cfg5) and configs[3] (cfg4) with the same measurements each.

A "step" is one V-cycle plus the per-cycle residual-norm check, exactly what one iteration of the
reference's MultilevelSolver.solve does (pyamg/multilevel.py:558-582).
  value    : V-cycles/s with b, x resident in HBM (CUDA events on the launching stream, max over ranks)
  e2e      : V-cycles/s through the C-ABI amgb_solve_ex with pinned HOST b/x, one cycle per call (the
             aspreconditioner() pattern): H2D b and D2H x inside the timed region every step
  roofline : the dominant kernel class of the cycle, algorithmic bytes / CUDA-event time, vs
             MEASURED_PEAKS.json hbm_gbs; traffic = DRAM bytes per launch from the committed ncu capture of the
             SAME library build (profiles/r02_ncu_traffic.json), else null
  fine_level : level-0 SpMV and the fused Jacobi+residual kernel in isolation, outputs checked at size
  cpu_baseline / --impl reference : the REAL pyamg.MultilevelSolver.solve of the unmodified reference
             (baseline/_ref, installed by oracle/build.py; travels to the GPU box) on the same operators and
             smoother parameters, 1 host core (the reference is single-threaded and holds the GIL); falls back to
             the oracle's restatement over the compiled relaxation.h when the package is absent
  --gpus N : torchrun, one rank per GPU: cfg3 and cfg4 row-partitioned (pyamg_b200/dist.py), peer-memory halo
             exchange, one CUDA graph per rank, parity_vs_n1, time_model_us
Inputs are far larger than L2 (level-0 operator alone is 1.4 GB), so no explicit L2 flush is needed.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
SEED = 20260922


def log(*a):
    if int(os.environ.get("RANK", "0")) == 0:
        print("[bench]", *a, file=sys.stderr, flush=True)


def peak_hbm():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


WORKLOAD = {"name": "cfg3"}      # set by --workload; the default is BASELINE.json's headline config


def build_hierarchy(grid, stream=None, device=0):
    """cfg3 (default): poisson(grid) + RS hierarchy + multi-colour symmetric GS on every level (BASELINE
    configs[2]).  cfg2: 2-D poisson(grid[:2]) + smoothed aggregation + weighted Jacobi (BASELINE configs[1]).
    cfg4: stencil_grid(rotated anisotropic diffusion, grid[:2]) + smoothed aggregation + weighted Jacobi (BASELINE
    configs[3], the multi-GPU configuration).  cfg5: linear_elasticity(grid[:2]) BSR(2,2) + smoothed aggregation on the rigid-body modes + block Jacobi
    (BASELINE configs[4])."""
    from pyamg_b200.gallery import poisson
    from pyamg_b200.classical import ruge_stuben_solver
    from pyamg_b200.aggregation import smoothed_aggregation_solver
    t0 = time.time()
    np.random.seed(SEED)
    if WORKLOAD["name"] == "cfg2":
        A = poisson(tuple(grid)[:2])
        t1 = time.time()
        sm = ("jacobi", {"omega": 4.0 / 3.0})
        ml = smoothed_aggregation_solver(A, presmoother=sm, postsmoother=sm, device=device, stream=stream)
    elif WORKLOAD["name"] == "cfg4":
        # BASELINE configs[3]: anisotropic rotated diffusion (eps = 0.001, theta = pi/6, FE stencil), SA + Jacobi -- the
        # row-partitioned multi-GPU configuration.  Strength of connection is the SA default ('symmetric'), which
        # the host setup offers; SURVEY.md 8(d)-4: with it the stand-alone V-cycle does not converge on this
        # operator (the reference needs strength='evolution' for that) -- throughput is unaffected.
        from pyamg_b200.gallery import stencil_grid, diffusion_stencil_2d
        A = stencil_grid(diffusion_stencil_2d(epsilon=0.001, theta=np.pi / 6, type="FE"), tuple(grid)[:2], format="csr")
        t1 = time.time()
        sm = ("jacobi", {"omega": 4.0 / 3.0})
        ml = smoothed_aggregation_solver(A, presmoother=sm, postsmoother=sm, device=device, stream=stream)
    elif WORKLOAD["name"] == "cfg5":
        from pyamg_b200.gallery import linear_elasticity
        A, B = linear_elasticity(tuple(grid)[:2])
        t1 = time.time()
        ml = smoothed_aggregation_solver(A, B=B, presmoother="block_jacobi", postsmoother="block_jacobi",
                                         device=device, stream=stream)
    else:
        A = poisson(grid)
        t1 = time.time()
        sm = ("gauss_seidel_indexed", {"sweep": "symmetric"})
        ml = ruge_stuben_solver(A, presmoother=sm, postsmoother=sm, device=device, stream=stream)
    t2 = time.time()
    log(f"gallery {t1 - t0:.1f}s, setup {t2 - t1:.1f}s, levels {[lv.A.shape[0] for lv in ml.levels]}, "
        f"op-cx {ml.operator_complexity():.3f}")
    return ml


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.stop_flag = gpu, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.gpu)], capture_output=True, text=True, timeout=5).stdout
                for ln in out.strip().splitlines():
                    self.rows.append([c.strip() for c in ln.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def sample_once(self):
        try:
            out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                  "-i", str(self.gpu)], capture_output=True, text=True, timeout=20).stdout
            for ln in out.strip().splitlines():
                self.rows.append([c.strip() for c in ln.split(",")])
        except Exception:
            pass

    def summary(self):
        self.stop_flag = True
        if not self.rows:
            self.sample_once()      # the region was shorter than one nvidia-smi round trip
        sm = [float(r[1]) for r in self.rows if len(r) > 2 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v == "Active":
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def reference_solver(ml):
    """The reference's CPU implementation of the path for hierarchy `ml`: (callable cycles(b, k) -> x after k
    V-cycles from x0 = 0 incl. the per-cycle residual checks, kind, description).

    With baseline/_ref present (the unmodified reference, compiled in place by oracle/build.py; it travels to
    the GPU box) this is the REAL ``pyamg.MultilevelSolver.solve`` (multilevel.py:398-582) on the same operators
    and smoother parameters (oracle/reference_adapter.py); otherwise the oracle's restatement of ``__solve`` driving
    the compiled ``relaxation.h`` (oracle/_ref/libamg_ref.so) or, last, the C port."""
    import oracle
    try:
        from oracle.reference_adapter import to_reference
        ref = to_reference(ml)
        return (lambda b, k: ref.solve(b, tol=0, maxiter=k)), "reference", \
            "pyamg.MultilevelSolver.solve of the unmodified reference (baseline/_ref), amg_core + SciPy matvec"
    except ImportError:
        pass
    kernels = "ref" if oracle.have_ref() else "oracle"
    cyc = oracle.Cycle(oracle.hierarchy_spec(ml), coarse_pinv=ml.coarse_solver.dense_operator(ml.levels[-1].A),
                       kernels=kernels)
    return (lambda b, k: cyc.solve(b, tol=0, maxiter=k)), ("reference" if kernels == "ref" else "port"), \
        ("compiled reference relaxation.h + SciPy matvec under the oracle's __solve restatement" if kernels == "ref"
         else "oracle C port")


def cpu_cycles_per_s(ml, b, ncyc):
    """The reference's CPU path on this host: (V-cycles/s, seconds, x after ncyc cycles, kind, description) -- x
    doubles as a full-size parity check."""
    cycles, kind, desc = reference_solver(ml)
    t0 = time.perf_counter()
    x = cycles(b, ncyc)
    dt = time.perf_counter() - t0
    return ncyc / dt, dt, x, kind, desc


def run_reference(args, grid):
    """--impl reference: the reference's own CPU implementation of the path, rank 0 only.  One call
    ``solve(b, tol=0, maxiter=steps)`` is timed: `steps` V-cycles, each followed by the residual check, exactly
    the reference's iteration (plus the one initial residual of the call)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    ml = build_hierarchy(grid)
    n = ml.levels[0].A.shape[0]
    b = np.random.default_rng(SEED).random(n)
    cycles, kind, desc = reference_solver(ml)
    if args.warmup > 0:
        cycles(b, args.warmup)
    t0 = time.perf_counter()
    cycles(b, args.steps)
    dt = time.perf_counter() - t0
    v = args.steps / dt
    print(json.dumps({
        "impl": "reference", "metric": "V-cycles/sec", "value": v, "unit": "V-cycles/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(grid, ml, 1),
        "cpu_baseline": {"value": v, "unit": "V-cycles/s", "cores": 1, "kind": kind,
                         "sample": f"one solve(b, tol=0, maxiter={args.steps}) = {args.steps} x (V-cycle + residual "
                                   f"check) on the full hierarchy; {desc}; host has {os.cpu_count()} cores, the "
                                   "reference path is single-threaded (GIL held, no OpenMP)"},
        "e2e": {"value": v, "unit": "V-cycles/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def workload_config(grid, ml, ngpus):
    if WORKLOAD["name"] == "cfg2":
        return {"workload": f"gallery.poisson({tuple(grid)[:2]}) 5-pt fp64 CSR, smoothed_aggregation_solver hierarchy "
                            f"({len(ml.levels)} levels, op-cx {ml.operator_complexity():.3f}), weighted Jacobi omega=4/3 "
                            "pre+post, pinv coarse solve, V(1,1)-cycle + per-cycle residual check",
                "n": int(ml.levels[0].A.shape[0]), "nnz": int(ml.levels[0].A.nnz),
                "sum_nnz_A": int(sum(lv.A.nnz for lv in ml.levels)),
                "parallelism": "1 GPU" if ngpus == 1 else f"{ngpus} GPUs", "l2": "inputs larger than L2"}
    if WORKLOAD["name"] == "cfg4":
        return {"workload": f"gallery.stencil_grid(diffusion_stencil_2d(eps=0.001, theta=pi/6, 'FE'), {tuple(grid)[:2]}) "
                            f"9-pt fp64 CSR, smoothed_aggregation_solver hierarchy (symmetric strength; {len(ml.levels)} "
                            f"levels, op-cx {ml.operator_complexity():.3f}), weighted Jacobi omega=4/3 pre+post, pinv "
                            "coarse solve, V(1,1)-cycle + per-cycle residual check",
                "n": int(ml.levels[0].A.shape[0]), "nnz": int(ml.levels[0].A.nnz),
                "sum_nnz_A": int(sum(lv.A.nnz for lv in ml.levels)),
                "parallelism": "1 GPU" if ngpus == 1 else f"{ngpus} GPUs", "l2": "inputs larger than L2"}
    if WORKLOAD["name"] == "cfg5":
        return {"workload": f"gallery.linear_elasticity({tuple(grid)[:2]}) Q1 fp64 BSR(2,2)->(3,3), "
                            f"smoothed_aggregation_solver(B = rigid-body modes) hierarchy ({len(ml.levels)} levels, "
                            f"op-cx {ml.operator_complexity():.3f}), block-Jacobi pre+post, pinv coarse solve, "
                            "V(1,1)-cycle + per-cycle residual check",
                "n": int(ml.levels[0].A.shape[0]), "nnz": int(ml.levels[0].A.nnz),
                "sum_nnz_A": int(sum(lv.A.nnz for lv in ml.levels)),
                "parallelism": "1 GPU" if ngpus == 1 else f"{ngpus} GPUs", "l2": "L2-resident problem"}
    return {"workload": f"gallery.poisson({tuple(grid)}) 7-pt fp64 CSR, ruge_stuben_solver hierarchy "
                        f"({len(ml.levels)} levels, op-cx {ml.operator_complexity():.3f}), symmetric multi-colour "
                        "Gauss-Seidel pre+post (gauss_seidel_indexed over colour-sorted rows), pinv coarse solve, "
                        "V(1,1)-cycle + per-cycle residual check",
            "n": int(ml.levels[0].A.shape[0]), "nnz": int(ml.levels[0].A.nnz),
            "sum_nnz_A": int(sum(lv.A.nnz for lv in ml.levels)),
            "parallelism": "1 GPU" if ngpus == 1 else f"{ngpus} independent replicas (one per GPU)",
            "l2": "inputs larger than L2 (level-0 operator 1.4 GB); no flush needed"}


def dist_measure(name, grid, args, local, rank, world, steps, warmup, dist_nnz):
    """One workload on `world` GPUs (strong scaling of the SAME problem): the levels with more than `dist_nnz` stored
    entries row-partitioned in contiguous slabs, the rest replicated (pyamg_b200/dist.py).  Halo exchange: one kernel
    per exchange that stores the boundary entries straight into the neighbours' memory over NVLink
    (csrc/abi_comm.cuh; AMGB_DIST_HALO=allgather|p2p selects the NCCL paths of round 1); restriction onto the
    replicated part and the stop-test norm are NCCL all-reduces; the whole cycle is ONE CUDA graph per rank.
    Returns rank 0's result dict (None on the other ranks)."""
    import torch
    import torch.distributed as dist
    from pyamg_b200.dist import DistributedSolver, GpuBackend, OP_GS, OP_JACOBI
    WORKLOAD["name"] = name
    dev = torch.device("cuda", local)
    tstream = torch.cuda.current_stream(dev)
    t0 = time.time()
    ml = build_hierarchy(grid, stream=tstream.cuda_stream, device=local)
    t_setup = time.time() - t0
    n = ml.levels[0].A.shape[0]
    t0 = time.time()
    be = GpuBackend(device=local, rank=rank, world=world)
    halo = os.environ.get("AMGB_DIST_HALO", "peer")
    ds = DistributedSolver(ml, be, halo=halo, dist_nnz=dist_nnz)
    log(f"[{name}] halo exchange: {halo}; partitioned levels {ds.n_dist} of {len(ml.levels)}; halo entries received/rank "
        f"{[int(L.sp.recv_off[-1]) if halo != 'allgather' else int(L.sp.maxB) for L in ds.lv]}; plan + upload {time.time() - t0:.1f}s")
    b_host = np.random.default_rng(SEED).random(n)
    ds.load(b_host)
    norms = be.vector(steps + warmup + 2)
    ds.cycles(max(warmup, 2))
    torch.cuda.synchronize()
    graphed = False
    if os.environ.get("AMGB_DIST_GRAPH", "1") == "1":            # the whole distributed cycle as one graph per rank
        try:
            ds.capture_graph()
            ds.cycles(1)
            torch.cuda.synchronize()
            graphed = True
        except Exception as exc:                                # noqa: BLE001 - fall back to host-driven launches
            ds._graph = None
            log(f"[{name}] graph capture unavailable ({type(exc).__name__}: {exc}); running host-driven")
    ok = torch.tensor([1 if graphed else 0], device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)                   # every rank replays a graph, or none does
    if int(ok.item()) == 0:
        ds._graph, graphed = None, False
    ds.load(b_host)
    dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = be.kernel_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    ds.cycles(steps, norms=norms)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    launches = be.kernel_launches - l0
    if graphed:
        launches += steps * getattr(ds, "graph_launches", 0)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    dist.barrier()
    # end to end: host rhs slice in, one cycle + stop-test norm, owned part of x back to the host
    L0 = ds.lv[0]
    own_b = b_host[L0.sp.order]
    pin_b = torch.from_numpy(own_b).pin_memory()
    pin_x = torch.empty(L0.sp.n_own, dtype=torch.float64).pin_memory()

    def e2e_step():
        L0.b[:L0.sp.n_own].copy_(pin_b, non_blocking=True)
        ds.cycles(1)
        ds.residual_norm()
        pin_x.copy_(L0.x[:L0.sp.n_own], non_blocking=True)
        torch.cuda.current_stream().synchronize()

    for _ in range(2):
        e2e_step()
    dist.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        e2e_step()
    e2e_dt = time.perf_counter() - t0
    t = torch.tensor([e2e_dt], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_dt = float(t.item())
    clocks = sampler.summary()
    # roofline of the local level-0 smoother kernel (same kernel as N=1, on this rank's slab)
    peak, peak_src = peak_hbm()
    D0 = L0.D
    if D0.wave_ptr is not None:
        w = int(np.argmax(np.diff(D0.wave_ptr)))
        rows_w = int(D0.wave_ptr[w + 1] - D0.wave_ptr[w])
        nnz_w = int(D0.A.indptr[D0.wave_ptr[w + 1]] - D0.A.indptr[D0.wave_ptr[w]])
        fn = lambda: be.apply(L0.A, OP_GS, L0.x, L0.b, L0.x, omega=1.0, wave=w)
        kbytes, kname = 12.0 * nnz_w + 36.0 * rows_w, "level 0 gs_wave on this rank's slab (csr_tile_kernel)"
    else:
        fn = lambda: be.apply(L0.A, OP_JACOBI, L0.x, L0.b, L0.xalt, omega=1.0)
        kbytes = 12.0 * D0.A.nnz + 4.0 * (D0.A.shape[0] + 1) + 24.0 * D0.A.shape[0]
        kname = "level 0 jacobi on this rank's slab (csr_tile_kernel)"
    for _ in range(3):
        fn()
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record()
    for _ in range(10):
        fn()
    a1.record()
    torch.cuda.synchronize()
    kms = a0.elapsed_time(a1) / 10
    res = np.sqrt(norms[:steps + 1].cpu().numpy())

    # ---- where the cycle's time goes: exchanges, local wave kernels, the replicated coarse part, the all-reduce ----
    def timed(fn, reps):
        for _ in range(2):
            fn()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dist.barrier()
        c0.record()
        for _ in range(reps):
            fn()
        c1.record()
        torch.cuda.synchronize()
        tt = torch.tensor([c0.elapsed_time(c1) / reps * 1e3], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return round(float(tt.item()), 2)

    parts = {"exchange_us": [timed(lambda L=L: ds.halo(L, L.x), 30) for L in ds.lv],
             "allreduce_restriction_us": timed(lambda: be.allreduce(ds.bc_rep), 20),
             "replicated_coarse_cycle_us": timed(lambda: ds.sub.cycle_device(ds.bc_rep, ds.xc_rep), 10),
             "largest_local_wave_us": []}
    for L in ds.lv:
        D = L.D
        if D.wave_ptr is not None:
            wl = int(np.argmax(np.diff(D.wave_ptr)))
            parts["largest_local_wave_us"].append(
                timed(lambda L=L, wl=wl: be.apply(L.A, OP_GS, L.x, L.b, L.x, omega=1.0, wave=wl), 20))
        else:
            parts["largest_local_wave_us"].append(
                timed(lambda L=L: be.apply(L.A, OP_JACOBI, L.x, L.b, L.xalt, omega=1.0), 20))
    log(f"[{name}] time model (us, host-driven launches, max over ranks): {parts}")
    # parity against the single-GPU engine on the same hierarchy and rhs: two cycles from zero on both
    ncyc = 2
    ds.load(b_host)
    ds.cycles(ncyc)
    x_dist = ds.gather_x()
    parity = None
    if rank == 0:
        x_one = ml.solve(b_host, tol=0, maxiter=ncyc)
        parity = float(np.linalg.norm(x_dist - x_one) / np.linalg.norm(x_one))
        ml._invalidate()
        log(f"[{name}] {world} GPUs: {steps / (ms * 1e-3):.1f} V-cycles/s ({ms / steps:.3f} ms/cycle, "
            f"{'one CUDA graph per rank' if graphed else 'host-driven launches'}), e2e {steps / e2e_dt:.1f}; "
            f"|x_{world}gpu - x_1gpu|/|x_1gpu| after {ncyc} cycles = {parity:.2e}")
    dist.barrier()
    out = None
    if rank == 0:
        cfg = workload_config(grid, ml, world)
        cfg["parallelism"] = (f"{world} GPUs: levels 0..{ds.n_dist - 1} row-partitioned (contiguous slabs), halo x entries "
                              + ("stored into the neighbours' memory over NVLink by one kernel per exchange"
                                 if halo == "peer" else f"exchanged with NCCL ({halo})")
                              + " before every operator application, NCCL all-reduce for the restriction onto the "
                              "replicated coarser levels (run redundantly on every rank)")
        out = {"value": steps / (ms * 1e-3), "unit": "V-cycles/s", "ms_per_step": ms / steps, "config": cfg,
               "roofline": {"bound": "hbm", "achieved": kbytes / kms / 1e6, "peak": peak, "unit": "GB/s",
                            "frac": kbytes / kms / 1e6 / peak, "traffic": None, "kernel": kname,
                            "peak_source": peak_src + " (MEASURED_PEAKS.json hbm_gbs)"},
               "e2e": {"value": steps / e2e_dt, "unit": "V-cycles/s", "h2d_bytes_per_step": 8 * n,
                       "d2h_bytes_per_step": 8 * n + 8 * world,
                       "path": "per rank: pinned rhs slab H2D, one distributed V-cycle + stop-test norm, owned x D2H"},
               "gpu_launches": int(launches), "clocks": clocks, "cuda_graph": graphed, "halo": halo,
               "residual_reduction_per_cycle": float((res[-1] / res[0]) ** (1.0 / max(len(res) - 1, 1))),
               "halo_entries_per_rank": [int(L.sp.recv_off[-1]) if halo != "allgather" else int(L.sp.maxB) for L in ds.lv],
               "exchanges_per_cycle": int(getattr(ds, "exchanges_per_cycle", 0)), "time_model_us": parts,
               "parity_vs_n1": {"rel_err": parity, "cycles": ncyc, "bar": 1e-12,
                                "against": "the single-GPU engine on rank 0, same hierarchy and rhs"},
               "host_setup_s": round(t_setup, 1)}
    be.close()
    del ds, be
    torch.cuda.empty_cache()
    return out


def run_distributed(args, grid, local, rank, world):
    """N > 1: the headline workload partitioned over the ranks, then (inside the same line, under `configs`) BASELINE
    configs[3] -- the multi-GPU configuration north_star names: anisotropic diffusion 4096^2, SA + Jacobi, one halo
    exchange per sweep."""
    import torch.distributed as dist
    head = dist_measure(args.workload, grid, args, local, rank, world, args.steps, args.warmup, 20_000_000)
    extra = {}
    for name in [c for c in args.configs.split(",") if c == "cfg4" and c != args.workload]:
        try:
            r = dist_measure(name, (DEFAULT_GRID[name],) * 3, args, local, rank, world, max(args.steps, 20), 3, 2_000_000)
            if r is not None:
                extra[name] = r
        except Exception as exc:                                   # noqa: BLE001 - the headline must still be printed
            if rank == 0:
                extra[name] = {"error": f"{type(exc).__name__}: {exc}"}
            log(f"[{name}] failed: {exc}")
    if rank == 0:
        out = {"metric": "V-cycles/sec", "value": head["value"], "unit": "V-cycles/s", "n_gpus": world,
               "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
               "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "cpu_baseline": None}
        for k, v in head.items():
            if k not in out:
                out[k] = v
        if extra:
            out["configs"] = extra
        out["so_sha16"] = so_sha()
        WORKLOAD["name"] = args.workload
        print(json.dumps(out), flush=True)
    dist.barrier()


OPS = {0: "spmv(restrict)", 1: "residual", 2: "prolong+add", 3: "jacobi", 4: "gs_wave", 5: "block_jacobi",
       6: "coarse_tail(cluster kernel)", 7: "resident_gs(cluster, DSMEM)", 8: "jacobi_indexed", 9: "block_gs_wave",
       10: "coarse_part(persistent grid kernel)"}
DEFAULT_GRID = {"cfg3": 256, "cfg2": 2000, "cfg4": 4096, "cfg5": 300}


def so_sha():
    try:
        return open(os.path.join(ROOT, "pyamg_b200", "libpyamg_b200.so.sha256")).read().split()[0][:16]
    except Exception:
        return None


def ncu_traffic(kernel_key):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of kernel `kernel_key` from the committed
    `ncu --set full` capture profiles/r02_ncu_traffic.json -- used only when that capture was taken from THIS build
    of the library (the capture records the .so's sha256); None otherwise."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")))
        if d.get("so_sha16") != so_sha():
            return None
        return d["kernels"].get(kernel_key, {}).get("dram_bytes_per_launch")
    except Exception:
        return None


DUMP_MAX_ENTRIES = 1 << 22       # 32 MB of float64: what --dump-outputs writes stays under 64 MB


def dump_outputs(out_dir, x, norms2):
    """--dump-outputs: what the timed amgb_solve_device call hands its caller, so that two builds run with the same
    arguments (hence the same inputs) can be compared output for output.  x.npy is the iterate after the last timed
    cycle (float64; above DUMP_MAX_ENTRIES entries a fixed sample at seeded positions, in index order) and
    residual_norms_sq.npy the call's steps + 1 squared residual norms."""
    os.makedirs(out_dir, exist_ok=True)
    x = x.cpu().numpy()
    if x.size > DUMP_MAX_ENTRIES:
        x = x[np.sort(np.random.default_rng(SEED).choice(x.size, DUMP_MAX_ENTRIES, replace=False))]
    np.save(os.path.join(out_dir, "x.npy"), x)
    np.save(os.path.join(out_dir, "residual_norms_sq.npy"), norms2.cpu().numpy())


def measure_config(name, grid, args, local, tstream, steps, warmup, cpu_sample, headline):
    """Everything bench.py reports for ONE workload on one GPU: device-resident V-cycles/s, e2e through the C ABI
    with host buffers, per-kernel roofline table, the reference's CPU path beside it and full-size parity."""
    import torch
    from pyamg_b200 import _engine as E
    WORKLOAD["name"] = name
    stream = tstream.cuda_stream
    t_setup = time.time()
    ml = build_hierarchy(grid, stream=stream, device=local)
    t_setup = time.time() - t_setup
    n = ml.levels[0].A.shape[0]
    t0 = time.time()
    dev_bytes = ml.upload()
    t_upload = time.time() - t0
    log(f"[{name}] upload + wave scheduling {t_upload:.1f}s, {dev_bytes / 1e9:.2f} GB in HBM")
    L, h = E.lib(), ml.handle
    b_host = E.pinned_empty(n)
    x_host = E.pinned_empty(n)
    b_host[:] = np.random.default_rng(SEED).random(n)
    dev = torch.device("cuda", local)
    b = torch.from_numpy(b_host).to(dev)
    x = torch.zeros(n, dtype=torch.float64, device=dev)
    norms = torch.zeros(steps + warmup + 2, dtype=torch.float64, device=dev)
    P = lambda t: ctypes.c_void_p(t.data_ptr())

    def cycles(k):
        E.check(L.amgb_solve_device(h, P(b), P(x), k, 0, 1, P(norms)))

    # ---- device-resident throughput -------------------------------------------------------
    cycles(warmup)
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    cycles(steps)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    launches = ml.last_launches()
    res = np.sqrt(norms[:steps + 1].cpu().numpy())
    if headline and args.dump_outputs:
        dump_outputs(args.dump_outputs, x, norms[:steps + 1])

    # ---- end to end through the C ABI with host buffers (one cycle per call) ---------------
    nres, info = ctypes.c_int32(0), ctypes.c_int32(0)
    rbuf = np.empty(4)
    x_host[:] = 0.0

    def e2e_step():      # what aspreconditioner() does per Krylov iteration: one cycle from x0 = 0
        E.check(L.amgb_solve_ex(h, b_host.ctypes.data, x_host.ctypes.data, 0.0, 1, 0, 1, E.FLAG_X0_ZERO,
                                E.f64p(rbuf), ctypes.byref(nres), ctypes.byref(info)))

    for _ in range(3):
        e2e_step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_dt = time.perf_counter() - t0
    clocks = sampler.summary()

    # ---- per-kernel roofline: CUDA events around every launch of one cycle ----------------
    peak, peak_src = peak_hbm()
    ml.profile_cycle()                                   # warm
    recs = np.concatenate([ml.profile_cycle() for _ in range(3)])
    groups = {}
    for lvl, op, rows, nnz, nbytes, t in recs:
        g = groups.setdefault((int(lvl), int(op)), [0.0, 0.0, 0])
        g[0] += nbytes; g[1] += t; g[2] += 1
    total_ms = sum(g[1] for g in groups.values())
    table = sorted(((k, g) for k, g in groups.items()), key=lambda kv: -kv[1][1])
    kernels = [{"level": k[0], "op": OPS.get(k[1], str(k[1])), "launches_per_cycle": g[2] // 3,
                "ms_per_cycle": round(g[1] / 3, 4), "share": round(g[1] / total_ms, 3),
                "GBps": round(g[0] / g[1] / 1e6, 1), "frac": round(g[0] / g[1] / 1e6 / peak, 3)} for k, g in table[:10]]
    (dk, dg) = table[0]
    key = f"{name}:L{dk[0]}:{OPS.get(dk[1], str(dk[1])).split('(')[0]}"
    roofline = {"bound": "hbm", "achieved": dg[0] / dg[1] / 1e6, "peak": peak, "unit": "GB/s",
                "frac": dg[0] / dg[1] / 1e6 / peak, "traffic": ncu_traffic(key),
                "kernel": f"level {dk[0]} {OPS.get(dk[1], str(dk[1]))}", "kernel_key": key,
                "peak_source": peak_src + " (MEASURED_PEAKS.json hbm_gbs)",
                "bytes_per_launch": dg[0] / dg[2], "ms_per_launch": dg[1] / dg[2], "share_of_cycle": dg[1] / total_ms}
    # whole-cycle figure: algorithmic bytes of every launch of the cycle / graphed cycle time
    cyc_bytes = sum(g[0] for g in groups.values()) / 3
    cycle_roof = {"algorithmic_GB_per_cycle": cyc_bytes / 1e9, "GBps": cyc_bytes / (ms / steps) / 1e6,
                  "frac": cyc_bytes / (ms / steps) / 1e6 / peak}
    small_ms = sum(g[1] for k, g in groups.items() if k[0] >= 3) / 3

    out = {"value": steps / (ms * 1e-3), "unit": "V-cycles/s", "ms_per_step": ms / steps, "steps": steps,
           "config": workload_config(grid, ml, 1), "roofline": roofline, "cycle_roofline": cycle_roof,
           "e2e": {"value": steps / e2e_dt, "unit": "V-cycles/s", "h2d_bytes_per_step": 8 * n,
                   "d2h_bytes_per_step": 8 * n + 16,
                   "path": "C ABI amgb_solve_ex(b_host, x_host, maxiter=1, X0_ZERO) per step (the aspreconditioner "
                           "pattern: rhs in, one cycle from zero + stop-test norms, iterate out), pinned host buffers"},
           "gpu_launches": int(launches), "clocks": clocks, "kernels": kernels,
           "levels_ge3_profiled_ms": round(small_ms, 4),     # un-graphed, event-timed launches: ~2.8x what they cost inside the graph
           "residual_reduction_per_cycle": float((res[-1] / res[0]) ** (1.0 / max(len(res) - 1, 1))),
           "hbm_bytes": int(dev_bytes), "host_setup_s": round(t_setup, 1), "upload_s": round(t_upload, 1)}

    # ---- fine-level kernels in isolation (metric: fine-level SpMV GB/s vs roofline), checked at size ----
    import oracle
    A0 = ml.levels[0].A
    if getattr(A0, "format", "csr") == "csr":
        keep = []
        A0c = E.as_matrix(A0, keep)
        op0 = ctypes.c_void_p()
        E.check(L.amgb_operator_create(local, ctypes.byref(A0c), None, 0, ctypes.c_void_p(stream), ctypes.byref(op0)))
        xin = torch.zeros(n + 2, dtype=torch.float64, device=dev)
        xin[:n] = b
        bb = torch.zeros(n + 2, dtype=torch.float64, device=dev)
        bb[:n] = torch.flip(b, dims=[0])
        y, r = torch.empty(n + 2, dtype=torch.float64, device=dev), torch.empty(n + 2, dtype=torch.float64, device=dev)

        def tkern(fn, reps=10):
            for _ in range(3):
                fn()
            a, c = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                fn()
            c.record()
            torch.cuda.synchronize()
            return a.elapsed_time(c) / reps

        nnz0 = A0.nnz
        omega = 0.8
        t_spmv = tkern(lambda: E.check(L.amgb_operator_apply(op0, 0, P(xin), None, P(y), None, 0.0, None, -1)))
        y_spmv = y[:n].cpu().numpy()
        t_jac = tkern(lambda: E.check(L.amgb_operator_apply(op0, 3, P(xin), P(bb), P(y), P(r), omega, None, -1)))
        y_jac, r_jac = y[:n].cpu().numpy(), r[:n].cpu().numpy()
        L.amgb_operator_destroy(op0)
        # parity of these launches AT SIZE against the reference's own kernels (amg_core.jacobi relaxation.h:309-346
        # compiled in place, SciPy csr_matvec): one Jacobi sweep, the residual by-product, the SpMV
        kern = "ref" if oracle.have_ref() else "oracle"
        xh, bh = b_host.copy(), b_host[::-1].copy()
        y_ref = oracle.matvec(A0, xh, kernels=kern)
        r_ref = bh - y_ref
        xj = xh.copy()
        oracle.jacobi(A0, xj, bh, iterations=1, omega=omega, kernels=kern)
        rel = lambda a_, b_: float(np.linalg.norm(a_ - b_) / np.linalg.norm(b_))
        by_spmv = 12 * nnz0 + 4 * (n + 1) + 16 * n
        by_jac = 12 * nnz0 + 4 * (n + 1) + 32 * n
        out["fine_level"] = {
            "kernel": "csr_tile_kernel (TMA-staged), level-0 operator, natural order",
            "spmv_ms": t_spmv, "spmv_GBps": by_spmv / t_spmv / 1e6, "spmv_frac": by_spmv / t_spmv / 1e6 / peak,
            "jacobi_residual_fused_ms": t_jac, "jacobi_residual_fused_GBps": by_jac / t_jac / 1e6,
            "jacobi_residual_fused_frac": by_jac / t_jac / 1e6 / peak, "jacobi_residual_fused_alg_bytes": by_jac,
            "parity": {"spmv": rel(y_spmv, y_ref), "jacobi_x": rel(y_jac, xj), "jacobi_residual": rel(r_jac, r_ref),
                       "against": "amg_core.jacobi (reference relaxation.h compiled in place) + SciPy csr_matvec"
                                  if kern == "ref" else "oracle C port", "bar": 1e-12}}
        log(f"[{name}] fine level: SpMV {out['fine_level']['spmv_frac']:.3f}, fused Jacobi+residual "
            f"{out['fine_level']['jacobi_residual_fused_frac']:.3f} of peak; parity {out['fine_level']['parity']}")
        del xin, bb, y, r

    # ---- CPU baseline: the reference's path on this box's host cores (bounded sample) + full-size parity ------
    cpu_v, cpu_dt, x_cpu, kind, desc = cpu_cycles_per_s(ml, b_host.copy(), cpu_sample)
    x_gpu = ml.solve(b_host, tol=0, maxiter=cpu_sample)
    parity = float(np.linalg.norm(x_gpu - x_cpu) / np.linalg.norm(x_cpu))
    log(f"[{name}] full-size parity after {cpu_sample} V-cycles: |x_gpu - x_cpu|/|x_cpu| = {parity:.3e}; "
        f"{out['value']:.1f} V-cycles/s, e2e {out['e2e']['value']:.1f}, cpu {cpu_v:.3f}")
    out["cpu_baseline"] = {"value": cpu_v, "unit": "V-cycles/s", "cores": 1, "kind": kind,
                           "sample": f"one solve(b, tol=0, maxiter={cpu_sample}) on the same hierarchy and rhs, "
                                     f"{cpu_dt:.1f}s; {desc}; single-threaded by construction; host has "
                                     f"{os.cpu_count()} cores"}
    out["parity_full_size"] = {"rel_err_vs_cpu_reference": parity, "cycles": cpu_sample, "bar": 1e-12}
    E.free_pinned(b_host)
    E.free_pinned(x_host)
    ml._invalidate()
    del b, x, norms
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--grid", type=int, default=None, help="grid points per dimension (default: the BASELINE size "
                    "of the workload: cfg3 256, cfg2 2000, cfg4 4096, cfg5 300)")
    ap.add_argument("--cpu-sample", type=int, default=2, help="V-cycles timed for cpu_baseline")
    ap.add_argument("--workload", default="cfg3", choices=["cfg3", "cfg2", "cfg4", "cfg5"],
                    help="cfg3 = BASELINE configs[2] (headline, default); cfg2 = configs[1]: 2-D Poisson 2000^2, SA + "
                         "Jacobi; cfg4 = configs[3]: anisotropic diffusion 4096^2, SA + Jacobi, the multi-GPU "
                         "configuration; cfg5 = configs[4]: 2-D elasticity 300^2, SA + block Jacobi")
    ap.add_argument("--configs", default="cfg2,cfg5,cfg4",
                    help="N=1 only: the other BASELINE GPU configurations measured after the headline and reported "
                         "under 'configs' (value, e2e, roofline, cpu_baseline, parity_full_size each); '' = none")
    ap.add_argument("--configs-budget-s", type=float, default=480.0,
                    help="a configuration of --configs is skipped once this much wall time has been spent on them")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the headline workload's timed solve returned as "
                         "DIR/<name>.npy (single GPU, --impl ours)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs is implemented for --impl ours on one GPU")
    WORKLOAD["name"] = args.workload
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    g = args.grid if args.grid is not None else DEFAULT_GRID[args.workload]
    grid = (g,) * 3

    if args.impl == "reference":
        run_reference(args, grid)
        return

    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1 and os.environ.get("OMP_NUM_THREADS", "1") == "1":
        # torchrun pins every rank to one OpenMP thread; the host-side setup (colouring, wave schedules, strength /
        # interpolation passes of csrc/host_setup.cpp) is multi-threaded: give each rank its share of the cores
        os.environ["OMP_NUM_THREADS"] = str(max(1, (os.cpu_count() or 1) // world))
    import torch
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        # NCCL's INFO lines would land on stdout, which carries exactly one JSON line: send them to stderr instead
        # (the driver's rank check reads the NCCL log; nothing is suppressed)
        if os.environ.get("NCCL_DEBUG") and not os.environ.get("NCCL_DEBUG_FILE"):
            os.environ["NCCL_DEBUG_FILE"] = "/dev/stderr"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    # a non-default torch stream: the engine launches on it, torch CUDA events time it
    tstream = torch.cuda.Stream(device=local)
    torch.cuda.set_stream(tstream)
    assert tstream.cuda_stream != 0
    if world > 1:
        run_distributed(args, grid, local, rank, world)
        return

    head = measure_config(args.workload, grid, args, local, tstream, args.steps, args.warmup, args.cpu_sample, True)
    out = {"metric": "V-cycles/sec", "value": head["value"], "unit": "V-cycles/s", "n_gpus": 1, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "strong",
           "vs_baseline": None, "dtype": "f64", "data": "synthetic"}
    for k in ("config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks", "fine_level", "kernels",
              "cycle_roofline", "levels_ge3_profiled_ms", "residual_reduction_per_cycle", "hbm_bytes",
              "parity_full_size", "host_setup_s", "upload_s"):
        if k in head:
            out[k] = head[k]
    out["so_sha16"] = so_sha()

    # ---- the other BASELINE GPU configurations, same measurements, bounded wall time ----------------------
    extra, t_extra = {}, time.time()
    for name in [c for c in args.configs.split(",") if c and c != args.workload]:
        if time.time() - t_extra > args.configs_budget_s:
            extra[name] = {"skipped": f"--configs-budget-s {args.configs_budget_s:.0f} s spent on the earlier ones"}
            continue
        try:
            gg = (DEFAULT_GRID[name],) * 3
            r = measure_config(name, gg, args, local, tstream, max(args.steps, 20), 3,
                               1 if name == "cfg4" else 2, False)
            r.pop("steps", None)
            extra[name] = r
        except Exception as exc:                                   # noqa: BLE001 - the headline must still be printed
            extra[name] = {"error": f"{type(exc).__name__}: {exc}"}
            log(f"[{name}] failed: {exc}")
    if extra:
        out["configs"] = extra
    WORKLOAD["name"] = args.workload
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()

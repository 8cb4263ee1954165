#!/usr/bin/env python
"""bench.py — headline benchmark of the B200 Newton iteration core.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--N 100] [--dump-outputs DIR]

Workload (BASELINE.json configs[2], the configuration the metric is quoted on): 3D Brusselator N=100 (10^6 cells, 2*10^6
unknowns), NewtonRaphson(linsolve = KrylovJL_GMRES()) with the matrix-free exact JVP, abstol = 1e-8 (the reference
test's value, sparsity_tests__item1.jl:54), GMRES tolerances inherited from the nonlinear solve (solve.jl:203), Krylov.jl's
default orthogonalisation (modified Gram-Schmidt, no reorthogonalisation, no restart) — `--orth cgs2` times the
reorthogonalised variant (Krylov's `reorthogonalization = true`), which is the library's own default because it is the
robust one on stiffer grids.
One "step" = one complete Newton solve from the synthetic initial condition (3 Newton iterations, ~2000 Arnoldi
iterations): a fixed, deterministic amount of hot-path work.  `value` = GMRES JVPs (Arnoldi iterations) per second with
inputs resident in HBM; `e2e` = the same through the host-buffer call (H2D of u0, solve, D2H of u and resid inside the
timed region).  N > 1: the single large system does not shard (SURVEY.md §8e, "replicas only"): every rank solves its own
replica, value = total JVPs of all ranks / max-over-ranks time ("weak").

The JSON line also carries `roofline` (dominant kernel family, live CUDA-event timing inside the timed region),
`cpu_baseline` (the CPU oracle timed on the host cores on a bounded sample) and `clocks`, and one object per remaining
BASELINE configuration, each with its own CPU baseline (rank 0 only, after the timed region of the headline):
  `n80`        the literal 10^6-DOF case (3D N=80, 1.02*10^6 unknowns), same algorithm as the headline;
  `lu`         config 2: 2D N=128 dense Jacobian fill + b200_getrf at n = 32768 (s, TFLOP/s), the same matrix through cuSOLVER
               (torch.linalg.lu_factor) as the stated comparison, and the whole NewtonRaphson() solve;
  `sparse_tr`  config 4: 3D N=100, coloured sparse Jacobian + TrustRegion + GMRES on the assembled matrix (s/solve, fill GB/s);
  `precond`    config 3 with the multigrid `precs` + EisenstatWalkerForcing2 (Arnoldi iterations, Newton steps/s);
  `ensemble`   config 5: 8192 x (2D N=32), sharded over the ranks, gathered through the library's C-ABI collective.
`--impl reference` times the CPU restatement of the reference (oracle/, "port": the Julia reference cannot run here).
`--dump-outputs DIR` writes what the last timed headline step returned (see `dump_outputs`), so that two builds can be compared
output for output on the same deterministic inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "gmres_jvps_per_s"
UNIT = "JVP/s"
MEAN_BASIS = {100: 345, 64: 217, 32: 107}  # mean Krylov basis size over one solve (measured; DESIGN.md §measurement)


def workload_name(N):
    return "bruss3d_N%d_newtonraphson_gmres_jfnk_abstol1e-8" % N


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
            "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for nm, val in zip(names, r[4:8]):
                    if val.lower().startswith("active"):
                        reasons.add(nm)
            except (ValueError, IndexError):
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def host_cpus():
    """Usable host cores: scheduler affinity capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(p))))
    except (OSError, ValueError):
        pass
    return n


_CPU_THREADS = {}


def cpu_sample(N, steps, count, orth="mgs"):
    """Time the CPU oracle on a bounded sample of the workload: `count` Arnoldi iterations (exact JVP + Gram-Schmidt
    orthogonalisation, the same arithmetic as the GPU arm) at the workload's mean Krylov basis size, using the thread
    count (all usable cores, or half / a quarter of them when SMT or memory-bandwidth saturation makes that faster)
    that a one-iteration calibration finds best."""
    os.environ.setdefault("OMP_WAIT_POLICY", "passive")
    os.environ.setdefault("OMP_PROC_BIND", "false")
    from oracle import pyoracle as po
    po.build()
    P = po.OracleProblem.bruss3d(N)
    u = P.u0(1)
    k0 = MEAN_BASIS.get(N, max(8, int(3.45 * N)))
    ocode = po.ORTH_MGS if orth == "mgs" else po.ORTH_CGS2
    if N not in _CPU_THREADS:
        T = host_cpus()
        best = None
        for cand in sorted({T, max(1, T // 2), max(1, T // 4)}, reverse=True):
            po.set_threads(cand)
            t = po.arnoldi_sample(P, u, k0, 1, ocode)
            if best is None or t < best[0]:
                best = (t, cand)
        _CPU_THREADS[N] = best[1]
    po.set_threads(_CPU_THREADS[N])
    times = []
    for _ in range(steps):
        # best of three: the first touches of a 5 GB basis and co-tenants on the host make single samples vary by +-50 %
        times.append(min(po.arnoldi_sample(P, u, k0, count, ocode) for _ in range(3)))
    cores = _CPU_THREADS[N]
    sample = "%d Arnoldi iterations (exact JVP + %s Gram-Schmidt + normalise) at the solve's mean basis size k=%d, N=%d, %d OpenMP threads" % (
        count, orth.upper(), k0, N, cores)
    return times, cores, sample, k0


def cpu_single_thread(N, orth="mgs"):
    """SURVEY §8(d): the CPU restatement single-threaded as well (the reference's Brusselator loop and Krylov.jl's BLAS-1 calls on
    `Array`s are effectively serial): ONE Arnoldi iteration at the mean basis size, best of two."""
    from oracle import pyoracle as po
    P = po.OracleProblem.bruss3d(N)
    u = P.u0(1)
    k0 = MEAN_BASIS.get(N, max(8, int(3.45 * N)))
    nthreads = po.get_threads()
    po.set_threads(1)
    try:
        t = min(po.arnoldi_sample(P, u, k0, 1, po.ORTH_MGS if orth == "mgs" else po.ORTH_CGS2) for _ in range(2))
    finally:
        po.set_threads(nthreads)
    return 1.0 / t


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port), bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    count = 4
    for _ in range(min(args.warmup, 1)):
        cpu_sample(args.N, 1, 1, args.orth)
    times, cores, sample, k0 = cpu_sample(args.N, args.steps, count, args.orth)
    total = sum(times)
    val = args.steps * count / total
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": {"workload": workload_name(args.N), "unknowns": 2 * args.N ** 3},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "CPU restatement of the reference NewtonRaphson+GMRES inner loop (oracle/oracle.c); the Julia reference cannot run in this image"}
    emit(line)


def ensemble_params(K):
    """BASELINE config 5 / SURVEY.md §8d: trajectory m is the 2D N=32 Brusselator with its own (A_m, B_m)."""
    import numpy as np
    m = np.arange(K)
    return 3.4 + 0.1 * (m % 64) / 64.0, 1.0 + 0.05 * (m // 64) / 128.0


def run_ensemble(nls, torch, dist, ctx, rank, world, K_total=8192, N=32, reps=2, orth="mgs"):
    """Config 5: ensemble of K_total independent 2D Brusselator problems, contiguous blocks sharded over the ranks
    (strong scaling, no data-path collective during the solve); after the solve one all-gather of the solutions and one
    all-reduce of the status counters (SURVEY.md §8e), both inside the timed region and both issued through the library's own
    C-ABI collective entry points (b200_nccl_init / b200_ens_allgather / b200_ens_allreduce_stats: NCCL over NVLink on the
    context's stream) — torch.distributed only ships the 128-byte NCCL id and collects the timing numbers."""
    import numpy as np
    n = 2 * N * N
    lo, hi = nls.shard_range(K_total, rank, world)
    K = hi - lo
    A, B = ensemble_params(K_total)
    dp = nls._DeviceProblem(ctx, nls.NonlinearProblem(nls.Brusselator2D(N), None, (3.4, 1.0, 10.0), ctx=ctx))
    u0 = np.tile(dp.u0().to_host(), K)
    d_u0, d_A, d_B = ctx.to_device(u0), ctx.to_device(A[lo:hi]), ctx.to_device(B[lo:hi])
    alg = nls.NewtonRaphson(linsolve=nls.KrylovJL_GMRES(orth=orth))
    cache = nls.EnsembleCache(ctx, N, K, 10.0, alg, abstol=1e-8)
    comm, gathered = None, None
    equal_blocks = K_total % world == 0
    if dist is not None:
        ids = [nls.Communicator.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        comm = nls.Communicator(ctx, world, rank, ids[0])
        gathered = ctx.empty(K_total * n) if equal_blocks else None
    stream = torch.cuda.current_stream()
    times, solve_ms, coll_ms = [], [], []
    res = glob = None
    for it in range(1 + reps):
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        e0, es, e1 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record(stream)
        res = cache.solve(d_u0, d_A, d_B)
        es.record(stream)
        glob = res
        if comm is not None:
            if gathered is not None:
                comm.allgather(cache.u_out, gathered)
            glob = comm.allreduce_stats(res)
        e1.record(stream)
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1), e0.elapsed_time(es), es.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        per_rank = [t.clone() for _ in range(world)]
        if dist is not None:
            dist.all_gather(per_rank, t)
        if it > 0:
            times.append(max(float(x[0]) for x in per_rank))
            solve_ms.append([float(x[1]) for x in per_rank])
            coll_ms.append(max(float(x[2]) for x in per_rank))
    ms = sum(times) / len(times)
    sm = np.mean(np.array(solve_ms), axis=0)
    return {"workload": "ensemble_%d_x_bruss2d_N%d_newtonraphson_gmres" % (K_total, N), "n_problems": K_total, "scaling": "strong", "orth": orth,
            "problems_per_s": K_total / (ms * 1e-3), "ms": ms, "n_success": int(glob.nsuccess), "newton_steps": int(glob.total_nsteps),
            "gmres_jvps": int(glob.total_njvp), "jvps_per_s": glob.total_njvp / (ms * 1e-3), "worst_resid_inf": glob.worst_resid_inf,
            "solve_ms_per_rank": [round(float(x), 2) for x in sm], "tail_imbalance": float(sm.max() / sm.mean()),
            "collective_ms": float(np.mean(coll_ms)),
            "collectives": ("b200_ens_allgather(u: %d x %d doubles per rank) + b200_ens_allreduce_stats through the C ABI (NCCL %s)" % (K, n, nls.Communicator.nccl_version()))
            if comm is not None else "none (1 rank)"}


def _events(torch, stream):
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def _timed(torch, stream, fn, reps=1, warm=0):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = _events(torch, stream)
    e0.record(stream)
    out = None
    for _ in range(reps):
        out = fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


def leg_n80(nls, torch, ctx, orth, peak):
    """The literal 10^6-DOF case: 3D N = 80 (1 024 000 unknowns), same algorithm as the headline."""
    N = 80
    f = nls.Brusselator3D(N)
    dp = nls._DeviceProblem(ctx, nls.NonlinearProblem(f, None, (3.4, 1.0, 10.0), ctx=ctx))
    u0 = dp.u0(nls.abi.U0_PERTURBED_Z)
    cache = nls.init(nls.NonlinearProblem(f, u0, (3.4, 1.0, 10.0), ctx=ctx), nls.NewtonRaphson(linsolve=nls.KrylovJL_GMRES(orth=orth)), abstol=1e-8)

    def step():
        cache.reinit(u0)
        return cache.solve(to_host=False)
    step()
    ctx.profile(True)
    ms, sol = _timed(torch, torch.cuda.current_stream(), step, reps=2)
    prof = ctx.profile_report()
    ctx.profile(False, reset=False)
    r = prof.get("resident", {"ms": 0.0, "bytes": 0.0, "launches": 0})
    ach = r["bytes"] / (r["ms"] * 1e-3) / 1e9 if r["ms"] > 0 else 0.0
    times, cores, sample, _ = cpu_sample(N, 1, 4, orth)
    return {"workload": workload_name(N), "unknowns": f.n(), "ms_per_solve": ms, "gmres_jvps_per_s": sol.stats.njvp / (ms * 1e-3),
            "newton_steps_per_s": sol.stats.nsteps / (ms * 1e-3), "lin_iters": [t.lin_iters for t in sol.trace], "resid_inf": sol.resid_inf,
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "share_of_step": r["ms"] * 0.5 / ms if ms > 0 else None},
            "cpu_baseline": {"value": 4 / sum(times), "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}}


def leg_lu(nls, torch, ctx):
    """Config 2: 2D Brusselator N = 128 (n = 32768): dense Jacobian fill, b200_getrf (FP64 tensor-core trailing update), the
    same matrix through cuSOLVER getrf (torch.linalg.lu_factor) on the same box, and the whole NewtonRaphson() solve."""
    import ctypes as C
    import numpy as np
    N = 128
    f = nls.Brusselator2D(N)
    dp = nls._DeviceProblem(ctx, nls.NonlinearProblem(f, None, (3.4, 1.0, 10.0), ctx=ctx))
    n = dp.n
    u = dp.u0()
    stream = torch.cuda.current_stream()
    L = nls.abi.lib()
    fill_ms, J = _timed(torch, stream, lambda: dp.dense_jacobian(u), reps=1, warm=0)
    A_t = torch.empty(n * n, dtype=torch.float64, device="cuda")
    nls.abi.check(ctx.handle, L.b200_memcpy_d2d(ctx.handle, C.c_void_p(A_t.data_ptr()), J.ptr, 8 * n * n))
    keep = ctx.empty(n * n)
    nls.abi.check(ctx.handle, L.b200_memcpy_d2d(ctx.handle, keep.ptr, J.ptr, 8 * n * n))
    ipiv = ctx.empty(n, np.int64)
    info = C.c_int32(-1)
    flops = 2.0 / 3.0 * float(n) ** 3

    def getrf():
        nls.abi.check(ctx.handle, L.b200_getrf(ctx.handle, n, J.ptr, n, ipiv.ptr, C.byref(info)))
    t1, _ = _timed(torch, stream, getrf)                      # first call: also sizes the workspaces
    nls.abi.check(ctx.handle, L.b200_memcpy_d2d(ctx.handle, J.ptr, keep.ptr, 8 * n * n))
    ctx.profile(True)
    t2, _ = _timed(torch, stream, getrf)
    prof = ctx.profile_report()
    ctx.profile(False, reset=False)
    assert info.value == 0
    piv_ours = ipiv.to_host()
    # getrs + residual of J x = f(u) as the correctness check of this very factorisation
    b = dp.residual(u)
    x = b.copy()
    solve_ms, _ = _timed(torch, stream, lambda: nls.abi.check(ctx.handle, L.b200_getrs(ctx.handle, n, 1, J.ptr, n, ipiv.ptr, x.ptr, n)))
    rel = dp.jvp(u, x).axpy(-1.0, b).norm(np.inf) / b.norm(np.inf)
    del keep
    # cuSOLVER on the same matrix (column-major view), same box, same stream
    A2 = A_t.view(n, n).T                                       # Fortran-contiguous n x n view of the same column-major data
    torch.linalg.lu_factor(A2[:1024, :1024].contiguous())       # warm up the handle
    cs_ms, (LU_t, piv_t) = _timed(torch, stream, lambda: torch.linalg.lu_factor(A2))
    same_pivots = bool(np.array_equal(piv_t.cpu().numpy().astype(np.int64), piv_ours))
    del LU_t, A_t, A2, J
    # whole config-2 solve
    u0 = dp.u0().to_host()
    prob = nls.NonlinearProblem(f, u0, (3.4, 1.0, 10.0), ctx=ctx)
    t0 = time.time()
    sol = nls.solve(prob, nls.NewtonRaphson(), abstol=1e-8)
    solve_s = time.time() - t0
    # CPU baseline: LAPACK getrf (scipy, all host threads) at n = 8192, extrapolated with n^3 and said so
    import scipy.linalg as sla
    nc = 8192
    M = np.random.default_rng(0).standard_normal((nc, nc))
    tc = time.time()
    sla.lu_factor(M, overwrite_a=True, check_finite=False)
    tc = time.time() - tc
    return {"workload": "bruss2d_N128_newtonraphson_dense_lu", "n": n, "jacobian_GB": 8.0 * n * n / 1e9, "fill_ms": fill_ms, "fill_gbs": 8.0 * n * n / (fill_ms * 1e-3) / 1e9,
            "getrf_s": t2 * 1e-3, "getrf_first_call_s": t1 * 1e-3, "lu_tflops": flops / (t2 * 1e-3) / 1e12, "getrs_ms": solve_ms, "solve_rel_residual": rel,
            "families_ms": {k: round(v["ms"], 2) for k, v in prof.items() if k.startswith("lu")},
            "tensor_pipe": "trailing update on the FP64 tensor cores (DMMA); pipe utilisation from ncu: see profiles/README.md",
            "cusolver_getrf_s": cs_ms * 1e-3, "cusolver_tflops": flops / (cs_ms * 1e-3) / 1e12, "vs_cusolver": cs_ms / t2, "pivots_equal_cusolver": same_pivots,
            "newton_solve_s": solve_s, "newton_nsteps": sol.stats.nsteps, "newton_nfactors": sol.stats.nfactors, "newton_resid_inf": sol.resid_inf,
            "newton_retcode": nls.ReturnCode.name(sol.retcode),
            "cpu_baseline": {"value": tc * (n / nc) ** 3, "unit": "s per getrf (n = 32768)", "cores": host_cpus(), "kind": "port",
                             "sample": "LAPACK getrf (scipy.linalg.lu_factor, OpenBLAS threads) at n = %d in %.2f s, extrapolated with n^3" % (nc, tc)}}


def leg_sparse_tr(nls, torch, ctx, orth, peak):
    """Config 4: 3D N = 100 with the coloured sparse Jacobian, TrustRegion, GMRES on the assembled matrix (resident engine with
    the CSR gather) — the direct sparse factorisation the reference would pick is infeasible at this size on any hardware."""
    import numpy as np
    N = 100
    f = nls.Brusselator3D(N)
    dp = nls._DeviceProblem(ctx, nls.NonlinearProblem(f, None, (3.4, 1.0, 10.0), ctx=ctx))
    u0 = dp.u0(nls.abi.U0_PERTURBED_Z)
    stream = torch.cuda.current_stream()
    sj = nls.SparseJacobian(dp)
    fill_ms, nz = _timed(torch, stream, lambda: sj.fill(u0), reps=3, warm=1)
    Bv = 8.0 * dp.n
    fill_bytes = sj.ncolors * 4.0 * Bv + sj.nnz * 16.0
    x = ctx.to_device(np.random.default_rng(0).standard_normal(dp.n))
    spmv_ms, _ = _timed(torch, stream, lambda: sj.mul(nz, x), reps=5, warm=1)
    spmv_bytes = sj.nnz * 24.0 + 2.0 * Bv
    ncolors, nnz = sj.ncolors, sj.nnz
    del sj, nz
    fs = nls.NonlinearFunction(f, sparsity=nls.TracerSparsityDetector())
    cache = nls.init(nls.NonlinearProblem(fs, u0, (3.4, 1.0, 10.0), ctx=ctx), nls.TrustRegion(linsolve=nls.KrylovJL_GMRES(orth=orth)), abstol=1e-8)

    def step():
        cache.reinit(u0)
        return cache.solve(to_host=False)
    step()
    ms, sol = _timed(torch, stream, step)
    # CPU baseline: the oracle's coloured fill of the same Jacobian (OpenMP), once
    from oracle import pyoracle as po
    P = po.OracleProblem.bruss3d(N)
    uh = P.u0(1)
    colptr, rowval = P.pattern(1)
    colors, nc = po.coloring_column(P.n, colptr, rowval, 1)
    tc = time.time()
    P.sparse_jac(uh, colptr, rowval, colors, nc, 1)
    tc = time.time() - tc
    return {"workload": "bruss3d_N100_trustregion_sparse_jacobian_gmres", "unknowns": dp.n, "ncolors": int(ncolors), "nnz": int(nnz),
            "s_per_solve": ms * 1e-3, "newton_steps": sol.stats.nsteps, "njacs": sol.stats.njacs, "gmres_jvps": sol.stats.njvp, "lin_iters": [t.lin_iters for t in sol.trace],
            "gmres_jvps_per_s": sol.stats.njvp / (ms * 1e-3), "resid_inf": sol.resid_inf, "retcode": nls.ReturnCode.name(sol.retcode),
            "jac_fill_ms": fill_ms, "jac_fill": {"bound": "hbm", "achieved": fill_bytes / (fill_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                                 "frac": fill_bytes / (fill_ms * 1e-3) / 1e9 / peak, "bytes": "ncolors*4*Bv + nnz*16"},
            "spmv": {"bound": "hbm", "achieved": spmv_bytes / (spmv_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": spmv_bytes / (spmv_ms * 1e-3) / 1e9 / peak,
                     "bytes": "nnz*24 + 2*Bv"},
            "cpu_baseline": {"value": fill_bytes / tc / 1e9, "unit": "GB/s (coloured Jacobian fill)", "cores": po.get_threads(), "kind": "port",
                             "sample": "one coloured sparse-Jacobian fill at N=100 (%d seeded JVP sweeps + scatter) in %.2f s" % (nc, tc)}}


def leg_precond(nls, torch, ctx):
    """Config 3 with what SURVEY.md §8f ranks next: EisenstatWalkerForcing2 + a preconditioner that cuts the iteration count
    (multigrid V-cycle through `precs`), beside the unpreconditioned headline."""
    N = 100
    f = nls.Brusselator3D(N)
    dp = nls._DeviceProblem(ctx, nls.NonlinearProblem(f, None, (3.4, 1.0, 10.0), ctx=ctx))
    u0 = dp.u0(nls.abi.U0_PERTURBED_Z)
    stream = torch.cuda.current_stream()
    out = {"workload": "bruss3d_N100_newtonraphson_gmres_multigrid_precs"}
    for name, alg in (("multigrid_right", nls.NewtonRaphson(linsolve=nls.KrylovJL_GMRES(orth="mgs", precs=nls.Multigrid("right")))),
                      ("multigrid_right_ew2", nls.NewtonRaphson(linsolve=nls.KrylovJL_GMRES(orth="mgs", precs=nls.Multigrid("right")), forcing=nls.EisenstatWalkerForcing2())),
                      ("ew2_only", nls.NewtonRaphson(linsolve=nls.KrylovJL_GMRES(orth="mgs"), forcing=nls.EisenstatWalkerForcing2()))):
        cache = nls.init(nls.NonlinearProblem(f, u0, (3.4, 1.0, 10.0), ctx=ctx), alg, abstol=1e-8)

        def step():
            cache.reinit(u0)
            return cache.solve(to_host=False)
        step()
        ms, sol = _timed(torch, stream, step, reps=1 if name == "ew2_only" else 3)
        out[name] = {"s_per_solve": ms * 1e-3, "newton_steps": sol.stats.nsteps, "newton_steps_per_s": sol.stats.nsteps / (ms * 1e-3), "arnoldi_iterations": sol.stats.njvp,
                     "lin_iters": [t.lin_iters for t in sol.trace], "resid_inf": sol.resid_inf, "retcode": nls.ReturnCode.name(sol.retcode)}
        del cache
    op = nls.Multigrid("right").linop(dp, u0)
    x = dp.residual(u0)
    y = ctx.zeros(dp.n)
    apply = lambda: nls.abi.check(ctx.handle, nls.abi.lib().b200_linop_apply(op, x.ptr, y.ptr))  # noqa: E731
    apply()
    ctx.sync()
    t0 = time.perf_counter()   # wall clock around 20 back-to-back applications, context drained on both sides (asynchronous calls:
    for _ in range(20):        # an event pair on another stream would time the host's enqueueing, not the V-cycle)
        apply()
    ctx.sync()
    out["vcycle_ms"] = (time.perf_counter() - t0) * 1e3 / 20
    nls.abi.lib().b200_linop_destroy(op)
    # CPU baseline: the NumPy restatement of the same V-cycle, one application
    from oracle import mg_numpy as mgn
    mg = mgn.Multigrid(N, 3, u0.to_host())
    xh = x.to_host()
    tc = time.time()
    mg.vcycle(xh)
    tc = time.time() - tc
    out["cpu_baseline"] = {"value": tc * 1e3, "unit": "ms per V-cycle", "cores": 1, "kind": "port", "sample": "one application of oracle/mg_numpy.py at N=100 (levels %s)" % mg.sizes()}
    return out


DUMP_LIMIT = 64 * 10 ** 6  # bytes, all files of --dump-outputs together


def dump_outputs(out_dir, sol, trace_fields):
    """What a caller of the timed path receives from its last step, as float64 arrays in out_dir/<name>.npy:
      u, resid      the root and the residual there (length n; when both no longer fit DUMP_LIMIT, the same seeded sample of
                    their entries, whose indices go to sample_index.npy);
      stats         retcode, nsteps, nf, njacs, nfactors, nsolve, njvp, resid_inf;
      trace         one row per Newton iteration, one column per trace field in `trace_fields` order."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    s = sol.stats
    out = {"u": sol.u.to_host(), "resid": sol.resid.to_host(),
           "stats": [sol.retcode, s.nsteps, s.nf, s.njacs, s.nfactors, s.nsolve, s.njvp, sol.resid_inf],
           "trace": np.array([[getattr(t, k) for k in trace_fields] for t in sol.trace], dtype=np.float64).reshape(-1, len(trace_fields))}
    n = out["u"].size
    keep = (DUMP_LIMIT - 10 ** 6) // (3 * 8)  # u, resid and the sample index; 1 MB left for stats and trace
    if n > keep:
        idx = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        out["u"], out["resid"], out["sample_index"] = out["u"][idx], out["resid"][idx], idx
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def traffic_from_profile(bytes_per_launch, resident):
    p = os.path.join(ROOT, "profiles", "r2_resident_traffic.json")
    if resident and os.path.exists(p):
        d = json.load(open(p))
        ratio = d["dram_bytes"] / d["algorithmic_bytes"]
        return {"traffic": bytes_per_launch * ratio,
                "traffic_source": "ncu --set full, one launch: dram read+write %.4f GB vs %.4f GB algorithmic (ratio %.4f, %s) applied to this run's mean bytes per launch" % (
                    d["dram_bytes"] / 1e9, d["algorithmic_bytes"] / 1e9, ratio, d["source"])}
    return {"traffic": None, "traffic_source": "no ncu summary for this kernel under profiles/"}


def run_b200(args):
    import numpy as np
    import torch
    import nonlinearsolve_jl_b200 as nls

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"  # keep NCCL's version banner off stdout: rank 0 prints exactly one JSON line
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    stream = torch.cuda.current_stream()
    ctx = nls.Context(local_rank, stream=stream.cuda_stream)
    N = args.N
    f = nls.Brusselator3D(N)
    n = f.n()
    dp = nls._DeviceProblem(ctx, nls.NonlinearProblem(f, None, (3.4, 1.0, 10.0), ctx=ctx))
    u0_dev = dp.u0(nls.abi.U0_PERTURBED_Z)  # synthetic, deterministic (SURVEY.md §8d)
    u0_pinned = ctx.pinned_empty(n)
    u0_pinned[:] = u0_dev.to_host()
    u_out, r_out = ctx.pinned_empty(n), ctx.pinned_empty(n)
    prob = nls.NonlinearProblem(f, u0_dev, (3.4, 1.0, 10.0), ctx=ctx)
    alg = nls.NewtonRaphson(linsolve=nls.KrylovJL_GMRES(orth=args.orth))
    cache = nls.init(prob, alg, abstol=1e-8, store_trace=True)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def one_step():
        cache.reinit(u0_dev)
        return cache.solve(to_host=False)

    for _ in range(args.warmup):
        sol = one_step()
    # ---- device-resident timed region
    clocks = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        clocks.start()
    ctx.profile(True)
    l0 = ctx.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    njvp = nsteps = 0
    bytes_moved = 0.0
    for _ in range(args.steps):
        sol = one_step()
        njvp += sol.stats.njvp
        nsteps += sol.stats.nsteps
        bytes_moved += sol.bytes_moved
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    ms_local = ms
    launches = ctx.kernel_launches() - l0
    prof = ctx.profile_report()
    ctx.profile(False, reset=False)
    clk = clocks.stop() if rank == 0 else None
    assert sol.retcode == nls.ReturnCode.Success and sol.resid_inf < 1e-8, (sol.retcode, sol.resid_inf)
    if args.dump_outputs and rank == 0:  # before the e2e region reuses the cache's buffers that sol.u and sol.resid point into
        dump_outputs(args.dump_outputs, sol, [k for k, _ in nls.abi.TraceRec._fields_])
    # ---- end-to-end timed region: host buffers, H2D + D2H inside
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record(stream)
    njvp_e2e = 0
    for _ in range(args.steps):
        s2 = cache.solve_host(u0_pinned, u_out, r_out)
        njvp_e2e += s2.stats.njvp
    e3.record(stream)
    barrier()
    ms_e2e = e2.elapsed_time(e3)
    assert np.abs(r_out).max() < 1e-8
    # ---- max over ranks, totals over ranks
    t = torch.tensor([ms, ms_e2e], dtype=torch.float64, device="cuda")
    c = torch.tensor([njvp, nsteps, njvp_e2e, launches], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
    ms, ms_e2e = t.tolist()
    njvp_all, nsteps_all, njvp_e2e_all, launches_all = c.tolist()
    ens = None
    if not args.no_ensemble:
        del cache  # release the Krylov basis before the ensemble workspaces are allocated
        ens = run_ensemble(nls, torch, dist, ctx, rank, world, orth=args.orth)
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    peak, peak_src = peaks()
    # dominant kernel family = the Gram-Schmidt streaming pair (multi-dot + update), timed live with CUDA events
    if prof.get("resident", {}).get("ms", 0.0) > prof.get("multidot", {}).get("ms", 0.0):
        dom, dom_name = ("resident",), ("resident3g_arnoldi_kernel (one cooperative kernel per Arnoldi step: JVP in registers + lag-1 modified Gram-Schmidt with the "
                                        "stored Gram sub-diagonal, the basis streamed once per pass through two TMA-fed shared-memory stages and a register stage, "
                                        "+ norm + Givens); algorithmic bytes (passes*k+3)*Bv per step, passes = %d" % (1 if args.orth == "mgs" else 2))
    else:
        dom, dom_name = ("multidot", "update"), "gmres orthogonalisation kernels of the multi-kernel engine (multidot_kernel + update_kernel)"
    dom_ms = sum(prof[k]["ms"] for k in dom if k in prof)
    dom_bytes = sum(prof[k]["bytes"] for k in dom if k in prof)
    dom_launches = sum(prof[k]["launches"] for k in dom if k in prof)
    achieved = dom_bytes / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
    roofline = {"bound": "hbm", "kernel": dom_name, "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                # DRAM traffic cannot be counted from inside a plain run; it comes from the committed `ncu --set full` capture of this
                # kernel (profiles/r2_resident_traffic.json, written by tools/ncu_traffic.py from the raw CSV): dram read + write
                # bytes of ONE launch and the algorithmic bytes of that same launch.  Null when the summary is absent.
                **traffic_from_profile(dom_bytes / max(dom_launches, 1), "resident" in dom),
                "bytes_per_launch": dom_bytes / max(dom_launches, 1), "ms_per_launch": dom_ms / max(dom_launches, 1),
                "share_of_step": dom_ms / (ms_local if ms_local > 0 else 1.0),
                "whole_step_gbs": bytes_moved / (ms * 1e-3) / 1e9,
                "families": {k: {"gbs": round(v["gbs"], 1), "ms": round(v["ms"], 2), "launches": v["launches"]} for k, v in prof.items()}}
    count = 4
    times, cores, sample, k0 = cpu_sample(N, 1, count, args.orth)
    cpu_val = count / sum(times)
    value = njvp_all / (ms * 1e-3)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": workload_name(N), "unknowns": n, "cells": N ** 3, "step": "one full Newton solve (%d Newton iterations, %d Arnoldi iterations)" % (
                nsteps // args.steps, njvp // args.steps), "orth": args.orth + (" (Krylov.jl default: modified Gram-Schmidt, no reorthogonalisation)" if args.orth == "mgs" else " (reorthogonalised)"), "gmres_engine": "resident" if "resident" in dom else "multikernel", "parallelism": "replicas x%d (single system does not shard)" % world,
                "l2": "inputs_exceed_l2 (Krylov basis %.1f GB per solve)" % (max(t_.lin_iters for t_ in sol.trace) * 8.0 * n / 1e9)},
            "newton_steps_per_s": nsteps_all / (ms * 1e-3),
            "e2e": {"value": njvp_e2e_all / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": 8 * n, "d2h_bytes_per_step": 16 * n,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches_all),
            "roofline": roofline,
            "cpu_baseline": {"value": cpu_val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                             "single_thread_value": cpu_single_thread(N, args.orth) if world == 1 else None},
            "clocks": clk,
            "ensemble": ens,
            "resid_inf": sol.resid_inf, "retcode": nls.ReturnCode.name(sol.retcode)}
    if not args.no_legs and world == 1:  # the other BASELINE configurations, each in a few seconds (N = 1 only, after the headline's timed regions)
        for key, fn in (("n80", lambda: leg_n80(nls, torch, ctx, args.orth, peak)), ("lu", lambda: leg_lu(nls, torch, ctx)),
                        ("sparse_tr", lambda: leg_sparse_tr(nls, torch, ctx, args.orth, peak)), ("precond", lambda: leg_precond(nls, torch, ctx))):
            try:
                line[key] = fn()
            except Exception as e:  # noqa: BLE001 — a failing extra leg must not take the headline line down with it
                line[key] = {"error": "%s: %s" % (type(e).__name__, e)}
            ctx.sync()
            torch.cuda.empty_cache()
    emit(line)
    if dist is not None:
        dist.destroy_process_group()


class _OneLineStdout:
    """The driver parses ONE JSON line from stdout.  Libraries print there behind our back (NCCL's version banner on the first
    communicator, whatever NCCL_DEBUG says): route file descriptor 1 to stderr for the whole run and write the line to the
    real stdout at the end."""

    def __enter__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)
        return self

    def emit(self, text):
        sys.stdout.flush()
        os.write(self.real, (text + "\n").encode())

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.real, 1)
        os.close(self.real)
        return False


_OUT = None


def emit(line):
    (_OUT.emit if _OUT is not None else print)(json.dumps(line))


def main():
    global _OUT
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--N", type=int, default=100)
    ap.add_argument("--orth", default="mgs", choices=["mgs", "cgs2"], help="GMRES orthogonalisation: mgs = Krylov.jl default (reference), cgs2 = reorthogonalised")
    ap.add_argument("--no-ensemble", dest="no_ensemble", action="store_true", help="skip the config-5 ensemble leg")
    ap.add_argument("--no-legs", dest="no_legs", action="store_true", help="skip the n80 / lu / sparse_tr / precond legs (configs 2, 4 and the §8f variants)")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", help="write the last timed step's outputs (u, resid, stats, trace) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl b200: the reference arm times a sample of the solve, not the whole path")
    with _OneLineStdout() as out:
        _OUT = out
        if args.impl == "reference":
            run_reference(args)
        else:
            run_b200(args)
        _OUT = None


if __name__ == "__main__":
    main()

#!/usr/bin/env python3
"""bench.py — headline benchmark of the Module A Krylov hot path (contract: see the task statement / DESIGN.md §6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--n 256] [--dump-outputs DIR]

Metric (BASELINE.json): CG iterations/s, fp64, 7-point Poisson n^3 (n=256 on one GPU), b = ones, tol = 1e-8.
A "step" is ONE full CG solve of that system (611 iterations) made through the reference-facing API
`pytorch_sparse_solver.module_a.cg(A, b, tol=1e-8)`:

  value         iterations done in the K timed solves / their device time (CUDA events), A and b resident in HBM
                (torch CSR tensor on the GPU; its registration with the library is cached and validated by content
                on every call, as for any user).  Inputs (1.4 GB touched per iteration) exceed L2: no flush needed.
  e2e           the same call with HOST tensors: module_a.cg(A_cpu, b_cpu, tol=1e-8) with A's arrays and b in pinned
                host memory — H2D of the CSR arrays and b, registration, solve and D2H of x inside the timed region.
  roofline      the GENERAL CSR SpMV kernel that SURVEY 8d's byte formula describes (kernel 2: int32 columns + fp64
                values streamed by TMA; option use_compress=0) on the same matrix in the same run, timed alone:
                achieved = algorithmic bytes per launch / mean launch time; frac = achieved / measured copy peak.
  roofline_coded  the kernel the solve actually uses for this constant-coefficient stencil (kernel 7, the stencil fast
                path over kernel 6's row-bitmask plan; lossless, bit-identical): achieved = ACTUAL bytes per launch — the matrix-side
                bytes counted by the library at registration (bk_csr_info.bytes_stream) + one read of x + one write of
                y — / mean launch time.
  iteration     the whole CG iteration both ways: algorithmic bytes (SURVEY 8d: nnz*12 + 4(n+1) + 11n*8) and actual
                bytes (bytes_stream + 10n*8: K1 reads p writes Ap, K2 reads Ap,r writes r, K3 reads x,p,r writes x,p; 9.5n*8 with
                the lagged-x cut).
  cpu_baseline  the oracle port of the reference (torch CPU, all host threads) on a bounded fixed-iteration window.
  extra         the other BASELINE configs through the same API: config 3 (BiCGStab, CD3D-256), config 4 (GMRES(30) on
                the LDC-100 pressure system, forward and forward+backward), config 1 (CG, 2-D Poisson 256^2) and the
                1-GPU anchor of the strong-scaling curve (CG on P3D-512).
With --impl reference the oracle port itself is the thing timed (rank 0 only): the SAME workload (config identical
to this arm's), each step a bounded sample of it — a fixed window of CG iterations of the same system.
For N > 1 (torchrun, one rank per GPU) the matrix is row-partitioned into N slabs of n^3 rows each (weak scaling;
BASELINE configs[4] geometry: 2n x 2n planes, n/4 planes per GPU, so N = 8 is exactly the (2n)^3 system); value =
N * global iterations/s.  Every N > 1 line carries a `parity` object (a full tol=1e-8 solve of the global system
checked by an independent residual computed with torch from the all-gathered x; mismatch => exit code 3) and
`extra.strong` (the SAME (2n)^3 system split over the N GPUs).

--dump-outputs DIR (one process: N = 1 or --impl reference) writes what the last timed step returned to its caller as
float64 .npy files, so that two builds can be compared output for output on identical inputs: x.npy and info.npy.  An x
of more than DUMP_MAX_ENTRIES entries is replaced by a fixed sample of its rows (seed 0), x.npy then holds x at the rows
listed in x_index.npy.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
PKG_DIR = ROOT / "pytorch-sparse-linalg-torch-amgx.cg.bicg.gmres_b200"
for p in (str(PKG_DIR), str(ROOT)):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

KERNEL_NAMES = {0: "bk_spmv_stream_kernel", 1: "bk_spmv_vector_kernel", 2: "bk_spmv_tma_kernel<int32 columns>",
                3: "bk_spmv_tma_kernel<8-bit dictionary-coded columns>", 4: "row-split view + bk_vrow_reduce_kernel",
                5: "bk_spmv_pair_kernel<8-bit (offset,value) pair codes, SELL-32-4>",
                6: "bk_spmv_mask_kernel<row bitmasks over chunk patterns>",
                7: "bk_spmv_mask2_kernel<stencil fast path: two rows per lane, 128-bit gathers, one summary per 64 rows>"}

METRIC = "cg_iterations_per_second"
UNIT = "it/s"
FALLBACK_HBM_GBS = 6650.0
DUMP_MAX_ENTRIES = 1 << 21      # 16 MB of sampled x + 16 MB of its row indices: at most 32 MB per dump


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback"


def dump_outputs(out_dir, x, info):
    """Write the solve's result (x, info) as float64 .npy files under out_dir (see the module docstring)."""
    import numpy as np
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    x = x.detach().to("cpu", torch.float64).reshape(-1)
    if x.numel() > DUMP_MAX_ENTRIES:
        idx = torch.randperm(x.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ENTRIES].sort().values
        np.save(out / "x_index.npy", idx.to(torch.float64).numpy())
        x = x[idx]
    else:
        (out / "x_index.npy").unlink(missing_ok=True)     # left by an earlier, sampled dump into the same directory
    np.save(out / "x.npy", x.numpy())
    np.save(out / "info.npy", np.array(info, dtype=np.float64))


def workload_config(n, tol):
    """The `config` object — identical for this arm and for --impl reference (same workload)."""
    N = n ** 3
    return {"workload": f"CG fp64, 7-pt Poisson {n}^3 CSR, b=ones, tol={tol:g} (BASELINE configs[1])",
            "n": N, "nnz": 7 * N - 6 * n * n, "tol": tol}


def dist_workload(n, world, window):
    """The N>1 workload string (both arms print the same one): n^3 rows per GPU, slabs stacked along the first axis."""
    npl, ppg = 2 * n, max(n // 4, 1)          # same slab geometry as _dist_problem
    if ppg * npl * npl != n ** 3:
        npl, ppg = n, n
    return (f"CG fp64, 7-pt Poisson {world * ppg}x{npl}x{npl} CSR row-partitioned over {world} GPUs "
            f"({n}^3 rows per GPU; 8 GPUs = BASELINE configs[4] 512^3 at n=256), b=ones, fixed window of "
            f"{window} iterations per step")


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 200 ms while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.lines = []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def __exit__(self, *a):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def oracle_window(A_cpu, b_cpu, target_s=15.0):
    """Time the oracle port (torch CPU, all threads) on a fixed-iteration CG window of the same system."""
    from oracle import krylov_oracle as orc
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    t0 = time.perf_counter()
    orc.cg(A_cpu, b_cpu, tol=0.0, atol=0.0, maxiter=2)
    t2 = time.perf_counter() - t0          # 2 iterations + 2 extra matvecs
    per_it = max(t2 / 4.0, 1e-6)
    iters = int(min(max(target_s / per_it, 5), 200))
    t0 = time.perf_counter()
    _x, _info, st = orc.cg(A_cpu, b_cpu, tol=0.0, atol=0.0, maxiter=iters)
    dt = time.perf_counter() - t0
    return st["iterations"] / dt, cores, iters, dt


def run_reference(args, rank, world):
    """`--impl reference`: the reference's CPU path (its oracle port: same torch-CPU primitives in the same order,
    pinned bit-exact to the reference in oracle/pin_reference.py), all host threads, rank 0 only.  Same workload as
    this repo's arm; each step is a bounded sample of it (a fixed window of CG iterations of the same system, long
    enough that the two matvecs outside the loop — r0 and the final residual check — weigh ~1 %)."""
    if rank != 0:
        return
    from pytorch_sparse_solver import problems
    n = args.n
    if world > 1:   # one slab of this repo's N-GPU workload (same geometry as _dist_problem), as a system of its own
        npl, ppg = 2 * n, max(n // 4, 1)
        if ppg * npl * npl != n ** 3:
            npl, ppg = n, n
        crow, col, val = problems.stencil3d_rows(npl, ppg, 0, ppg)
        A = torch.sparse_csr_tensor(crow, col, val, size=(n ** 3, n ** 3))
    else:
        A = problems.poisson3d_csr(n)
    b = torch.ones(A.shape[0], dtype=torch.float64)
    from oracle import krylov_oracle as orc
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    window = args.ref_window
    for _ in range(args.warmup):           # warm-up: thread pool, page faults (short windows)
        orc.cg(A, b, tol=0.0, atol=0.0, maxiter=min(window, 3))
    t0 = time.perf_counter()
    its = 0
    for _ in range(args.steps):
        x, info, st = orc.cg(A, b, tol=0.0, atol=0.0, maxiter=window)
        its += st["iterations"]
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, x, info)
    value = its / dt
    sample = (f"{args.steps} x fixed window of {window} CG iterations (tol=0, same recurrences as the tol={args.tol:g} "
              f"solve, which takes 611) on P3D-{n}, torch CPU, {cores} threads, {dt:.0f} s")
    cfg = workload_config(n, args.tol)
    if world > 1:
        # N > 1: this repo's arm runs the weak-scaled system (n^3 rows per GPU) and counts n^3-row CG iterations per
        # second over all ranks.  The reference is single-process: one n^3-row slab is its bounded sample, and its rate
        # on the slab IS its rate in those units (N times the rows take it N times as long per iteration).
        cfg = {"workload": dist_workload(n, world, args.dist_window),
               "value_definition": f"{n}^3-row CG iterations per second"}
        sample += (f"; the sample is ONE {ppg}x{npl}x{npl} slab of {n}^3 rows (1/{world} of the system) — the metric counts {n}^3-row "
                   f"iterations, which a single process performs at this rate whatever the number of slabs")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(args.steps, 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def time_events(fn, reps, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def extra_configs(args, dev, peak):
    """The other BASELINE configs, each through the public module_a API (device-resident inputs)."""
    from pytorch_sparse_solver import module_a, problems
    from pytorch_sparse_solver.module_a import krylov
    out = {}
    n = args.n
    try:   # config 3: BiCGStab fp64 on the upwind convection-diffusion n^3 system, manufactured RHS
        C = problems.convdiff3d_csr(n, device=dev)
        bc, _xt = problems.manufactured_rhs(C, 0)
        module_a.bicgstab(C, bc, tol=1e-8)
        its = 0
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        reps = 3
        for _ in range(reps):
            module_a.bicgstab(C, bc, tol=1e-8)
            its += krylov.last_result["iterations"]
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        r = krylov.last_result
        nnz = C.values().numel()
        balg = problems.bicgstab_bytes_per_iteration(C.shape[0], nnz)
        out["config3_bicgstab_cd3d"] = {
            "workload": f"BiCGStab fp64, upwind convection-diffusion {n}^3, b = A randn(seed 0), tol=1e-8 (BASELINE configs[2])",
            "iterations_per_solve": r["iterations"], "info": r["info"], "relres": r["final_residual"] / r["b_norm"],
            "us_per_iteration": 1e3 * ms / its, "iterations_per_second": its / (ms * 1e-3),
            "algorithmic_gbs": balg * its / ms / 1e6, "frac_of_8tbs_algorithmic": balg * its / ms / 1e6 / 8000.0}
        del C, bc
    except Exception as e:  # pragma: no cover
        out["config3_bicgstab_cd3d"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    try:   # config 4: GMRES(30) on the LDC-100 pressure system (RHS of time step 1 of the reference driver), + backward
        import numpy as np
        L = problems.ldc_pressure_csr(100, device=dev)
        gold = ROOT / "tests" / "golden" / "gmres_ldc100_step1_batched.npz"
        if gold.exists():
            with np.load(gold) as z:
                bl = torch.from_numpy(z["b"].copy()).to(dev)
            rhs = "RHS of time step 1 of the reference LDC driver (tests/golden)"
        else:
            bl = torch.sin(torch.arange(L.shape[0], dtype=torch.float64, device=dev))
            bl -= bl.mean()
            rhs = "synthetic zero-mean RHS"
        kw = dict(tol=1e-10, maxiter=1000, restart=30)
        module_a.gmres(L, bl, **kw)
        ms_f = time_events(lambda: module_a.gmres(L, bl, **kw), reps=5, warm=1)
        r = dict(krylov.last_result)

        def fwd_bwd():
            b1 = bl.clone().requires_grad_(True)
            x, _ = module_a.gmres(L, b1, **kw)
            (x ** 2).sum().backward()
            return b1.grad
        ms_fb = time_events(fwd_bwd, reps=3, warm=1)
        out["config4_gmres_ldc100"] = {
            "workload": f"GMRES(30) fp64, LDC 100x100 pressure system (CSR), tol=1e-10, maxiter=1000 (BASELINE configs[3]); {rhs}",
            "restart_cycles": r["iterations"], "matvecs": r["matvecs"], "info": r["info"],
            "ms_per_solve": ms_f, "matvecs_per_second": r["matvecs"] / (ms_f * 1e-3),
            "ms_per_solve_with_backward": ms_fb, "loop_mode_used": r.get("loop_mode_used")}
    except Exception as e:  # pragma: no cover
        out["config4_gmres_ldc100"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    try:   # config 1: CG on the 2-D Poisson 256 x 256 system (the reference's own CPU-runnable case), launch-bound
        P = problems.poisson2d_csr(256, 256, device=dev)
        bp = torch.ones(P.shape[0], dtype=torch.float64, device=dev)
        module_a.cg(P, bp, tol=1e-8)
        ms = time_events(lambda: module_a.cg(P, bp, tol=1e-8), reps=10, warm=2)
        r = krylov.last_result
        out["config1_cg_p2d256"] = {
            "workload": "CG fp64, 2-D 5-pt Poisson 256x256, b=ones, tol=1e-8 (BASELINE configs[0], on the GPU)",
            "iterations_per_solve": r["iterations"], "info": r["info"], "ms_per_solve": ms,
            "iterations_per_second": r["iterations"] / (ms * 1e-3), "loop_mode_used": r.get("loop_mode_used")}
    except Exception as e:  # pragma: no cover
        out["config1_cg_p2d256"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    if not args.no_strong:
        try:   # 1-GPU anchor of the strong-scaling curve: the (2n)^3 system of BASELINE configs[4] on ONE GPU
            n2 = 2 * n
            S = problems.poisson3d_csr(n2, device=dev)
            bs_ = torch.ones(S.shape[0], dtype=torch.float64, device=dev)
            W = args.dist_window
            module_a.cg(S, bs_, tol=0.0, atol=0.0, maxiter=10)
            torch.cuda.synchronize()
            ms = time_events(lambda: module_a.cg(S, bs_, tol=0.0, atol=0.0, maxiter=W), reps=2, warm=1)
            out["strong"] = {"workload": f"CG fp64, 7-pt Poisson {n2}^3 on 1 GPU, fixed window of {W} iterations "
                                         f"(anchor of the strong-scaling curve, BASELINE configs[4])",
                             "n_gpus": 1, "iterations_per_second": W / (ms * 1e-3), "us_per_iteration": 1e3 * ms / W}
            del S, bs_
        except Exception as e:  # pragma: no cover
            out["strong"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    return out


def run_single(args):
    from pytorch_sparse_solver import _native, module_a, problems
    from pytorch_sparse_solver.module_a import krylov
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    n = args.n
    N = n ** 3
    A = problems.poisson3d_csr(n, device=dev)                      # torch CSR, int64 indices, fp64 values
    nnz = A.values().numel()
    b = torch.ones(N, dtype=torch.float64, device=dev)
    bytes_iter = problems.cg_bytes_per_iteration(N, nnz)
    bytes_k1 = nnz * 12 + (N + 1) * 4 + 2 * N * 8                  # matrix + read p + write Ap
    peak, peak_kind = measured_peak()
    h = _native.Handle.get(dev)

    # ---- value: K full solves through the reference-facing API, device-resident inputs ---------------------------
    for _ in range(max(args.warmup, 3)):
        module_a.cg(A, b, tol=args.tol)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    its = launches = 0
    dev_ms = 0.0
    with ClockSampler(0) as clk:
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(args.steps):
            x, info = module_a.cg(A, b, tol=args.tol)
            res = krylov.last_result
            its += res["iterations"]
            launches += res["kernel_launches"] + 3                 # + the cache validation's checksum kernels
            dev_ms += res["device_ms"]
        ev1.record()
        torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, x, info)
    value = its / (ms * 1e-3)
    last = dict(res)
    m = _native.register_matrix(A)
    minfo = m.info()

    # ---- rooflines: the SpMV kernels timed alone (back-to-back launches, CUDA events on the launching stream) -----
    p = torch.randn(N, dtype=torch.float64, device=dev)
    reps = 20
    k_ms = time_events(lambda: m.spmv_dot(p, p), reps)
    actual_k1 = minfo["bytes_stream"] + 2 * N * 8
    roofline_coded = {
        "bound": "hbm", "kernel": KERNEL_NAMES.get(minfo["kernel"], "?") + " (SpMV fused with p.Ap; the kernel the solve uses)",
        "achieved": actual_k1 / (k_ms * 1e-3) / 1e9, "peak": peak, "peak_kind": peak_kind, "unit": "GB/s",
        "frac": actual_k1 / (k_ms * 1e-3) / 1e9 / peak, "traffic": None, "bytes_per_launch": actual_k1,
        "bytes_matrix_stream": minfo["bytes_stream"], "ms_per_launch": k_ms,
        "note": "ACTUAL bytes per launch: matrix-side bytes counted by the library at registration (bk_csr_info."
                "bytes_stream) + one read of x + one write of y; DRAM traffic measured by ncu is in profiles/"}
    saved = h.get_option("use_compress")
    try:
        h.set_option("use_compress", 0)
        _native.clear_cache()
        m2 = _native.register_matrix(A)
        i2 = m2.info()
        k2_ms = time_events(lambda: m2.spmv_dot(p, p), reps)
        W = 60
        cg2_ms = time_events(lambda: m2.cg(b, None, 0.0, 0.0, W), reps=2, warm=1)
        del m2
    finally:
        h.set_option("use_compress", saved)
        _native.clear_cache()
    roofline = {
        "bound": "hbm", "kernel": KERNEL_NAMES.get(i2["kernel"], "?") + " (general CSR SpMV fused with p.Ap; use_compress=0)",
        "achieved": bytes_k1 / (k2_ms * 1e-3) / 1e9, "peak": peak, "peak_kind": peak_kind, "unit": "GB/s",
        "frac": bytes_k1 / (k2_ms * 1e-3) / 1e9 / peak, "traffic": None, "bytes_per_launch": bytes_k1,
        "ms_per_launch": k2_ms,
        "cg_iteration_general_csr": {"us_per_iteration": 1e3 * cg2_ms / W, "iterations_per_second": W / (cg2_ms * 1e-3),
                                     "achieved_gbs": bytes_iter * W / cg2_ms / 1e6,
                                     "frac_of_peak": bytes_iter * W / cg2_ms / 1e6 / peak,
                                     "frac_of_8tbs": bytes_iter * W / cg2_ms / 1e6 / 8000.0},
        "note": "the kernel SURVEY 8d's algorithmic byte count (nnz*12 + (n+1)*4 + 2n*8) describes: every CSR byte is "
                "streamed; read-dominated, so it can sit slightly above the measured COPY peak. traffic: see profiles/ "
                "(ncu DRAM bytes are not measurable inside this run)"}
    # vector passes per iteration: K1 reads p writes Ap (2), K2 reads Ap,r writes r (3), K3 reads x,p,r writes x,p (5) —
    # or, with the lagged-x cut (cg_lag_x, large systems), K3 alternates 3 and 6 passes: 9.5 per iteration
    lagged = bool(h.get_option("cg_lag_x")) and N > 300000
    vec_passes = 9.5 if lagged else 10.0
    actual_iter = int(minfo["bytes_stream"] + vec_passes * N * 8)
    iteration = {
        "us_per_iteration": 1e3 * ms / its,
        "algorithmic": {"bytes_per_iteration": bytes_iter, "achieved_gbs": bytes_iter * value / 1e9,
                        "frac_of_8tbs": bytes_iter * value / 8e12,
                        "note": "SURVEY 8d yardstick (reference-equivalent CSR plan); above 1 because the coded SpMV and "
                                "the re-cut iteration move fewer bytes than that plan"},
        "actual": {"bytes_per_iteration": actual_iter, "achieved_gbs": actual_iter * value / 1e9,
                   "frac_of_peak": actual_iter * value / 1e9 / peak,
                   "note": f"bytes the three kernels of an iteration really stream: matrix stream + {vec_passes:g} vector passes"
                           + (" (lagged-x cut: x is updated every second iteration)" if lagged else "")}}

    # ---- e2e: the same API call with HOST tensors (pinned): H2D + registration + solve + D2H inside -----------------
    e2e = None
    if not args.no_e2e:
        crow_h = A.crow_indices().cpu().pin_memory()
        col_h = A.col_indices().cpu().pin_memory()
        val_h = A.values().cpu().pin_memory()
        b_h = b.cpu().pin_memory()
        A_h = torch.sparse_csr_tensor(crow_h, col_h, val_h, size=A.shape)
        pinned = bool(A_h.values().is_pinned() and A_h.col_indices().is_pinned() and b_h.is_pinned())
        h2d = sum(t.numel() * t.element_size() for t in (crow_h, col_h, val_h, b_h))
        d2h = N * 8
        # warm-up in the same pattern as the timed loop (the result of the previous solve stays referenced while the
        # next one runs, so the pinned result buffers alternate: both must exist before the clock starts — the first
        # round-2 runs timed one 50 ms cudaHostAlloc in three steps)
        for _ in range(3):
            xh, _info = module_a.cg(A_h, b_h, tol=args.tol)
        torch.cuda.synchronize()
        k_e2e = max(1, min(args.steps, 3))
        t0 = time.perf_counter()
        its_e = 0
        for _ in range(k_e2e):
            xh, _info = module_a.cg(A_h, b_h, tol=args.tol)
            its_e += krylov.last_result["iterations"]
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        e2e = {"value": its_e / dt, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "ms_per_step": 1e3 * dt / k_e2e, "steps": k_e2e, "api": "pytorch_sparse_solver.module_a.cg(A_cpu, b_cpu)",
               "host_buffers_pinned": pinned, "x_on_host": (not xh.is_cuda)}
        del crow_h, col_h, val_h, A_h

    cpu = None
    if not args.no_cpu:
        A_cpu = torch.sparse_csr_tensor(A.crow_indices().cpu(), A.col_indices().cpu(), A.values().cpu(), size=A.shape)
        v, cores, iters, dt = oracle_window(A_cpu, b.cpu(), args.cpu_seconds)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"fixed window of {iters} CG iterations (tol=0) of the same P3D-{n} system, torch CPU, "
                         f"{cores} threads, {dt:.1f} s"}
        del A_cpu
    del A, p
    extra = {} if args.no_extra else extra_configs(args, dev, peak)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": workload_config(n, args.tol),
        "details": {"api": "pytorch_sparse_solver.module_a.cg(A, b, tol)", "iterations_per_solve": last["iterations"],
                    "info": last["info"], "relres": last["final_residual"] / last["b_norm"],
                    "loop_mode_used": last["loop_mode_used"], "device_ms_per_solve": dev_ms / args.steps,
                    "l2_policy": "inputs (1.4 GB streamed per iteration) exceed L2; no flush needed",
                    "spmv_kernel": minfo["kernel"],
                    "options": {k: h.get_option(k) for k in ("use_tma", "use_compress", "tma_ctas", "pair_ctas", "mask_ctas",
                                                             "mask_group", "mask_const", "mask_cctas", "cg_lag_x", "tma_stages",
                                                             "grid_mult_spmv", "grid_mult_vec", "fuse_xpay", "snake", "loop_mode",
                                                             "chunk")}},
        "roofline": roofline, "roofline_coded": roofline_coded, "iteration": iteration,
        "e2e": e2e, "cpu_baseline": cpu, "extra": extra, "gpu_launches": int(launches), "clocks": clk.summary(),
    }
    print(json.dumps(line))


# ---- N > 1: weak scaling on the row-partitioned system, with a parity object and the strong-scaling arm -------------
def _dist_problem(problems, n, world, rank, dev, strong):
    npl, ppg = 2 * n, max(n // 4, 1)
    rows = n ** 3
    if ppg * npl * npl != rows:
        npl, ppg = n, n
    if strong:   # BASELINE configs[4] as written: the SAME (2n)^3 system split over N GPUs (N must divide 2n)
        ppg = npl // world
        rows = ppg * npl * npl
    offsets = [q * rows for q in range(world + 1)]
    crow, col, val = problems.stencil3d_rows(npl, world * ppg, rank * ppg, (rank + 1) * ppg, device=dev)
    return npl, ppg, rows, offsets, crow, col, val


def _dist_parity(D, crow, col, val, rows, world, rank, dev, tol):
    """Full tol solve of the global system through the reference API on the DistMatrix + an INDEPENDENT residual:
    all-gather x, multiply this rank's slab rows (GLOBAL columns) with torch's own CSR SpMV (checker only, never on
    the product path), reduce ||b - A x||^2 over the ranks."""
    import torch.distributed as dist
    from pytorch_sparse_solver import module_a
    from pytorch_sparse_solver.module_a import krylov
    b = torch.ones(rows, dtype=torch.float64, device=dev)
    x, info = module_a.cg(D, b, tol=tol)
    r1 = dict(krylov.last_result)
    x2, _ = module_a.cg(D, b, tol=tol)
    xs = [torch.empty_like(x) for _ in range(world)]
    dist.all_gather(xs, x.contiguous())
    xg = torch.cat(xs)
    A_slab = torch.sparse_csr_tensor(crow, col, val, size=(rows, rows * world))
    r = b - torch.mv(A_slab, xg)
    acc = torch.stack([(r * r).sum(), (b * b).sum(), (x * x).sum()])
    dist.all_reduce(acc)
    rel_ind = float(torch.sqrt(acc[0] / acc[1]))
    rel_lib = r1["final_residual"] / r1["b_norm"]
    ok = (info == 0 and rel_ind <= tol * 1.0000001 and abs(rel_ind - rel_lib) <= 1e-3 * rel_lib + 1e-14
          and bool(torch.equal(x, x2)))
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    return {"ok": bool(int(flag)), "check": "full tol solve via module_a.cg(DistMatrix, b_local); independent residual "
            "||b - A x|| / ||b|| from the all-gathered x with torch's CSR SpMV on this rank's rows (global columns), "
            "all-reduced; library's own final residual must agree; two solves bitwise equal",
            "tol": tol, "iterations": int(r1["iterations"]), "info": int(info), "relres_independent": rel_ind,
            "relres_library": rel_lib, "x_norm": float(torch.sqrt(acc[2])), "bitwise_repeatable": bool(torch.equal(x, x2))}


def _dist_window(D, b, window, steps, warm, ClockSamplerCls, local):
    import torch.distributed as dist
    for _ in range(warm):
        D.cg(b, None, 0.0, 0.0, min(window, 50))
    torch.cuda.synchronize()
    dist.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    its = launches = 0
    with ClockSamplerCls(local) as clk:
        torch.cuda.synchronize()
        dist.barrier()
        ev0.record()
        for _ in range(steps):
            x, res = D.cg(b, None, 0.0, 0.0, window)
            its += res["iterations"]
            launches += res["kernel_launches"]
        ev1.record()
        torch.cuda.synchronize()
        dist.barrier()
    ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=b.device)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms), its, launches, clk


def run_dist(args, rank, world):
    import torch.distributed as dist
    from pytorch_sparse_solver import distributed as bkd
    from pytorch_sparse_solver import problems
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    n = args.n
    peak, peak_kind = measured_peak()
    strong_main = bool(args.strong)
    npl, ppg, rows, offsets, crow, col, val = _dist_problem(problems, n, world, rank, dev, strong_main)
    nnz_local = val.numel()
    D = bkd.DistMatrix(crow, col, val, offsets, rank, world)
    b = torch.ones(rows, dtype=torch.float64, device=dev)
    window = args.dist_window
    ms, its, launches, clk = _dist_window(D, b, window, args.steps, max(args.warmup, 3), ClockSampler, local)
    it_s = its / (ms * 1e-3)
    value = it_s * (rows * world) / float(n ** 3)   # n^3-row CG iterations per second over all ranks
    bytes_iter = problems.cg_bytes_per_iteration(rows, nnz_local)
    parity = _dist_parity(D, crow, col, val, rows, world, rank, dev, args.tol)
    comm = ("peer-memory (CUDA IPC over NVLink): kernel halo push + one-shot all-reduce" if D.p2p
            else "NCCL send/recv + allreduce")
    peers0 = list(D.plan.peers)
    info_loc = D.local_info() if hasattr(D, "local_info") else {}
    # end to end: host slab -> device, partition set-up, IPC mapping, solve window, x back to host
    D.close()
    crow_h, col_h, val_h = (t.cpu().pin_memory() for t in (crow, col, val))
    b_h = b.cpu().pin_memory()
    h2d = sum(t.numel() * t.element_size() for t in (crow_h, col_h, val_h, b_h))
    del crow, col, val
    from pytorch_sparse_solver import module_a
    from pytorch_sparse_solver.module_a import krylov
    xh = torch.empty(rows, dtype=torch.float64).pin_memory()        # the result lands in pinned host memory
    for rep in range(2):                                            # first pass = warm-up of this code path
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        D2 = bkd.DistMatrix(crow_h.to(dev, non_blocking=True), col_h.to(dev, non_blocking=True),
                            val_h.to(dev, non_blocking=True), offsets, rank, world)
        xe, info_e = module_a.cg(D2, b_h.to(dev, non_blocking=True), tol=args.tol)   # the call a user makes: a full solve
        xh.copy_(xe)
        torch.cuda.synchronize()
        dist.barrier()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        its_e = int(krylov.last_result["iterations"])
        if rep == 0:
            D2.close()
            del D2, xe
    e2e = {"value": world * its_e / float(dt), "unit": UNIT, "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": rows * 8, "ms_per_step": 1e3 * float(dt), "steps": 1,
           "iterations": its_e, "info": int(info_e),
           "api": "DistMatrix(slab from pinned host buffers) + pytorch_sparse_solver.module_a.cg(D, b_local, tol) + x to host",
           "note": "one full tol solve per step; includes H2D of the slab, partition set-up, halo-plan exchange, IPC "
                   "window mapping, registration (the NCCL communicator of the process is reused)"}
    D2.close()
    del crow_h, col_h, val_h, xh, xe
    # strong-scaling arm: the SAME (2n)^3 system split over the N GPUs
    strong = None
    if not strong_main and not args.no_strong and (2 * n) % world == 0:
        npl_s, ppg_s, rows_s, off_s, crow, col, val = _dist_problem(problems, n, world, rank, dev, True)
        Ds = bkd.DistMatrix(crow, col, val, off_s, rank, world)
        bs_ = torch.ones(rows_s, dtype=torch.float64, device=dev)
        ms_s, its_s, _l, _c = _dist_window(Ds, bs_, window, max(1, min(args.steps, 3)), 2, ClockSampler, local)
        strong = {"workload": f"CG fp64, 7-pt Poisson {2 * n}^3 split over {world} GPUs, fixed window of {window} iterations",
                  "n_gpus": world, "iterations_per_second": its_s / (ms_s * 1e-3), "us_per_iteration": 1e3 * ms_s / its_s,
                  "note": "strong-scaling efficiency = this / (N x extra.strong.iterations_per_second of the N=1 line)"}
        Ds.close()
        del crow, col, val
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong" if strong_main else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": (dist_workload(n, world, window) if not strong_main else
                                    f"CG fp64, 7-pt Poisson {2 * n}^3 CSR split over {world} GPUs (strong scaling), b=ones, "
                                    f"fixed window of {window} iterations per step"),
                       "comm": comm,
                       "value_definition": f"{world} x global iterations/s = {n}^3-row CG iterations per second over all ranks",
                       "global_iterations_per_second": it_s, "n_local": rows, "nnz_local": nnz_local,
                       "halo_bytes_per_neighbour": npl * npl * 8, "peers_rank0": peers0, "local_matrix": info_loc,
                       "l2_policy": "inputs exceed L2; no flush needed"},
            "roofline": {"bound": "hbm", "kernel": "whole distributed CG iteration (per GPU), ALGORITHMIC bytes",
                         "achieved": bytes_iter * it_s / 1e9, "peak": peak, "peak_kind": peak_kind, "unit": "GB/s",
                         "frac": bytes_iter * it_s / 1e9 / peak, "traffic": None,
                         "note": "algorithmic (CSR-plan) bytes; the coded SpMV moves fewer — see the N=1 line's "
                                 "roofline_coded / iteration.actual"},
            "iteration": {"bytes_per_iteration_per_gpu": bytes_iter, "us_per_iteration": 1e3 * ms / its,
                          "frac_of_8tbs": bytes_iter * it_s / 8e12},
            "parity": parity, "extra": {"strong": strong},
            "e2e": e2e, "cpu_baseline": None, "gpu_launches": int(launches), "clocks": clk.summary(),
        }
        print(json.dumps(line))
    dist.barrier()
    dist.destroy_process_group()
    if not parity["ok"]:
        sys.exit(3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=256, help="grid edge (n^3 rows per GPU)")
    ap.add_argument("--tol", type=float, default=1e-8)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra BASELINE configs (3, 4, 1, strong anchor)")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling arm / anchor")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--dist-window", type=int, default=200, help="N>1: CG iterations per timed step")
    ap.add_argument("--strong", action="store_true", help="N>1: make the strong-scaling split the headline value")
    ap.add_argument("--ref-window", type=int, default=100, help="--impl reference: CG iterations per step")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's solution x and info as float64 .npy files to DIR (one process)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1 or args.gpus > 1 or args.strong or os.environ.get("BK_BENCH_FORCE_DIST"):  # env: 1-rank run of the multi-GPU path
        if "RANK" not in os.environ:
            raise SystemExit("launch multi-GPU runs with torch.distributed.run (one rank per GPU)")
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes the result of one process: use it with --gpus 1 or --impl reference")
        run_dist(args, rank, world)
    else:
        run_single(args)


if __name__ == "__main__":
    main()

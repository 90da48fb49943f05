#!/usr/bin/env python
"""bench.py — AMG-PCG solve of 3D 7-point Poisson 256^3 (BASELINE.json configs[2]) on N B200s.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the reference's own CPU path on the host cores
    python bench.py --steps K --dump-outputs DIR              # also write the last step's outputs to DIR (see --help)

One "step" = one complete AMG-preconditioned CG solve (HEM hierarchy as shipped, V(7,7) Jacobi, omega = 0.66667) of the
16.8M-row system to a RELATIVE residual of 1e-8 (north_star; the reference's absolute 1e-8 is unreachable at this size,
SURVEY F6), x0 = 0, b = 1.  The hierarchy is built once by the host setup and uploaded once (outside the timed region,
as north_star specifies); every step re-solves from x0 = 0.

  value  solve seconds, device-timed (CUDA events on the library's stream), b and x resident in HBM
  e2e    the same solve through the reference-facing host-buffer call (sparsh_hierarchy_solve_host, the twin of
         AMG_GPU1_solver::helper / Solver_PCG_4's cudaMemcpy prologue+epilogue): pinned host b, x -> H2D, solve, D2H of x
  roofline      the dominant kernel (fused Jacobi sweep on the finest level: 14 of the 17 matrix passes per level),
                timed alone with CUDA events on the same stream right after the timed steps; algorithmic bytes from
                SURVEY §8d; peak = MEASURED_PEAKS.json hbm_gbs (burst figure)
  cpu_baseline  the reference's own host code (oracle/_ref: its sources compiled unmodified against the OpenMP MKL shim)
                on all host cores, a bounded sample of the same workload

Inputs are far larger than L2 (the finest matrix alone is 1.4 GB against 126 MB), so no explicit L2 flush is needed.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# PCG iterations to rel 1e-8 on 3D Poisson n^3, b = 1, HEM hierarchy, V(7,7): the count the REFERENCE ITSELF needs (its
# stock Solver_PCG_1 run to convergence by tools/pin_reference_pcg.py, frozen under tests/golden/); the GPU path's count
# is gated against it by tests/test_gpu_host_api.py.  Used only when the reference arm is asked to skip its own
# converged solve (--warmup 0).
def reference_iterations(grid):
    f = os.path.join(ROOT, "tests", "golden", f"pcg_poisson3d_{grid}_ref.json")
    return int(json.load(open(f))["iterations"]) if os.path.exists(f) else None


METRIC = "amg_pcg_solve_seconds_poisson3d_256"
UNIT = "s"


def measured_peak():
    from sparsh_amg_b200 import benchutil

    return benchutil.measured_peak()


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 200 ms during the timed region"""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower() == "active"})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def problem_rhs(n):
    return np.ones(n)


# --dump-outputs: solution vectors longer than this are written at one fixed, seeded sample of rows (2^21 doubles = 16 MB
# per vector), so that the outputs of two builds at 256^3 can be compared entry for entry in well under 64 MB
DUMP_ROWS = 1 << 21


def dump_outputs(path, vectors, residual_history):
    """write each vector of `vectors` (all of one length n) at the rows listed in x_index.npy, plus the residual history,
    as float64 <path>/<name>.npy"""
    n = len(next(iter(vectors.values())))
    idx = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "x_index.npy"), idx.astype(np.float64))
    for name, v in vectors.items():
        np.save(os.path.join(path, f"{name}.npy"), np.ascontiguousarray(v[idx], dtype=np.float64))
    np.save(os.path.join(path, "residual_history.npy"), np.asarray(residual_history, dtype=np.float64))


# ----------------------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation on the host cores
# ----------------------------------------------------------------------------------------------------------------
class CpuReference:
    """the reference's own host code (oracle/_ref: its sources compiled unmodified against the OpenMP MKL shim) on one
    n^3 Poisson system: its setup (AMG_solver::AMG_solver_setup_jacobi, HEM as shipped) runs once in the constructor"""

    def __init__(self, grid, threads):
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from oracle_bindings import Oracle, Ref, RefAmg, have_ref

        if not have_ref():
            raise RuntimeError("oracle/_ref/libsparsh_ref.so missing (built where /root/reference exists)")
        o = Oracle.get()
        o.set_threads(threads)
        Ref.get().set_threads(threads)
        self.A = o.gen_poisson3d(grid, grid, grid)
        self.ref = RefAmg(self.A)
        self.b = problem_rhs(self.A.nrow)
        self.threads = threads

    def sample(self, iters):
        """seconds per iteration of a bounded sample: `iters` iterations of Solver_PCG_1's loop"""
        t, _, _ = self.ref.pcg_sample(self.b, np.zeros(self.A.nrow), iters)
        return t / iters

    def converged(self, max_iter=500):
        """one solve to rel 1e-8 with the reference's own stopping rule -> (seconds, iterations, history)"""
        t, _, hist = self.ref.pcg_solve(self.b, np.zeros(self.A.nrow), 1e-8 * float(np.linalg.norm(self.b)), max_iter)
        return t, len(hist) - 1, hist


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # under torchrun only rank 0 runs the CPU arm
    from sparsh_amg_b200 import benchutil

    threads = os.cpu_count() or 1
    grid = args.grid
    cpu = CpuReference(grid, threads)
    nlev = cpu.ref.nlevels
    conv = None
    iters = reference_iterations(grid)
    if args.warmup >= 1:  # warm-up = ONE solve run to convergence: measured iteration count and measured solve seconds
        t_full, iters, hist = cpu.converged()
        conv = {"seconds": t_full, "iterations": iters, "final_rel_residual": float(hist[-1] / hist[0])}
    per_iter = float(np.mean([cpu.sample(args.ref_iters) for _ in range(args.steps)]))
    sample = (f"{args.steps} steps, each a bounded sample of {args.ref_iters} PCG iterations of the full {grid}^3 system "
              f"(the loop body of the reference's Solver_PCG_1, src/AMG_main_solvers.cpp:136-152, around its own "
              f"AMG_solve_jacobi V(7,7) cycle; unmodified sources + OpenMP MKL shim), {threads} threads")
    if iters:
        value = per_iter * iters
        sample += (f"; value = mean seconds/iteration x {iters} iterations"
                   + (" (the count the converged warm-up solve of this run needed)" if conv else
                      " (the count the reference's stock Solver_PCG_1 needs, tests/golden)"))
    else:
        value = per_iter
        sample += "; iteration count to rel 1e-8 unknown here: value is seconds per PCG ITERATION"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": value * 1e3, "higher_is_better": False,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": benchutil.workload(grid, nlev), "grid": grid, "rows": int(cpu.A.nrow),
                       "nnz": int(cpu.A.nnz)},
            "details": {"seconds_per_pcg_iteration": per_iter, "reference_setup_seconds": cpu.ref.setup_seconds,
                        "converged_solve": conv, "extrapolated": True,
                        "driver": "oracle/ref_harness.cpp: ref_pcg_sample / ref_pcg_solve (Solver_PCG_1's loop on a "
                                  "hierarchy built once by the reference's AMG_solver_setup_jacobi)"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "reference", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
# this repo's arm
# ----------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch

    import sparsh_amg_b200 as sp
    from sparsh_amg_b200 import host

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        from sparsh_amg_b200 import distributed as dist_mod

        return dist_mod.bench_main(args, METRIC, UNIT, ClockSampler)

    torch.cuda.set_device(local_rank)
    sp.init(local_rank)
    stream = torch.cuda.Stream()
    sp.set_stream(stream.cuda_stream)
    lib = sp.capi.load()
    grid = args.grid
    threads = os.cpu_count() or 1
    host.set_options(threads=threads, max_levels=32, print_setup=0, print_solve=0, coarsening=0, sweeps=7,
                     use_graph=1, gpu_rap=int(args.gpu_rap))
    t0 = time.time()
    A = host.HostMatrix.poisson3d(grid, grid, grid)
    t_gen = time.time() - t0
    amg = host.HostAmg(A)  # native host setup: HEM + Galerkin, bit-identical integers to the reference's
    rep = host.report()
    dH = amg.upload()       # AMG_GPU1_solver::GPU_Allocations: once
    rep2 = host.report()
    n = A.nrow

    # pinned host buffers for the e2e leg, device-resident vectors for the device-timed leg
    hb, hx = C.c_void_p(), C.c_void_p()
    sp.capi.check(lib.sparsh_host_alloc(n * 8, C.byref(hb)))
    sp.capi.check(lib.sparsh_host_alloc(n * 8, C.byref(hx)))
    b_host = np.ctypeslib.as_array(C.cast(hb, C.POINTER(C.c_double)), shape=(n,))
    x_host = np.ctypeslib.as_array(C.cast(hx, C.POINTER(C.c_double)), shape=(n,))
    b_host[:] = problem_rhs(n)
    tol = 1e-8 * float(np.linalg.norm(b_host))
    db, dx = sp.DeviceVector(data=b_host), sp.DeviceVector(n)
    max_iter = args.max_iter

    def solve_device():
        dx.fill(0.0)
        return dH.pcg(db, dx, tol, max_iter)

    def solve_host():
        return dH.solve_host("pcg", b_host, x_host, tol, max_iter)

    n_warm = args.warmup if args.profile else max(args.warmup, 3)
    for _ in range(n_warm):
        it, hist, ok = solve_device()
    if not ok and not args.profile:
        raise RuntimeError(f"PCG did not converge in {max_iter} iterations (last residual {hist[-1]:.3e})")

    sampler = ClockSampler(local_rank)
    sampler.start()
    sp.launch_count(reset=True)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    sp.sync()
    ev[0].record(stream)
    for _ in range(args.steps):
        it, hist, ok = solve_device()
    ev[1].record(stream)
    ev[1].synchronize()
    launches = sp.launch_count()
    solve_s = ev[0].elapsed_time(ev[1]) * 1e-3 / args.steps
    x_device = dx.download() if args.dump_outputs else None  # before the e2e leg and the kernel timings reuse dx

    # e2e: host buffers in, host buffer out, copies inside the timed region
    # (each step is timed by itself: writing the initial guess x0 = 0 into the caller's buffer between two steps is the
    # caller preparing its input, like filling b, and stays outside; both copies of it and of b are inside)
    for _ in range(2):
        x_host[:] = 0.0
        solve_host()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2e_dev = e2e_wall = 0.0
    for _ in range(args.steps):
        x_host[:] = 0.0
        sp.sync()
        w0 = time.perf_counter()
        e0.record(stream)
        it_h, hist_h, ok_h = solve_host()
        e1.record(stream)
        e1.synchronize()
        e2e_wall += time.perf_counter() - w0
        e2e_dev += e0.elapsed_time(e1) * 1e-3
    e2e_s = max(e2e_dev, e2e_wall) / args.steps  # wall clock covers the host-side orchestration too
    clocks = sampler.stop()
    x_final = x_host.copy()
    if args.dump_hist:  # residual history of the solve, for the pin against the reference's own history (tools/)
        json.dump({"grid": grid, "iterations": int(it), "tol": tol, "history": [float(v) for v in hist]},
                  open(args.dump_hist, "w"))
    if args.dump_outputs:  # what the caller of each timed path receives from its last step
        dump_outputs(args.dump_outputs, {"x": x_device, "x_e2e": x_final}, hist)

    # roofline of the dominant kernel (fused Jacobi sweep on the finest level), timed alone on the same stream: the
    # kernel the solve really runs, then the same matrix forced to plain CSR (the kernel north_star's ">= 70 % of HBM
    # peak" is written for), then every other kernel of the iteration
    from sparsh_amg_b200 import benchutil

    A0, _, _ = dH.level(0)
    z = A0.nnz
    kind, tl, _ = A0.kernel()
    tb = sp.DeviceVector(n)
    roof, roof_csr, kernels = {"bound": "hbm"}, None, None
    try:
        roof = benchutil.roofline_jacobi(torch, stream, lib, A0, db, dx, tb, grid)
        kernels = benchutil.kernel_table(torch, stream, lib, dH, db, dx, grid)
        A0.force_kernel(sp.capi.KIND_STREAM, 256)
        roof_csr = benchutil.roofline_jacobi(torch, stream, lib, A0, db, dx, tb, grid)
        csr_spmv = benchutil.timed(torch, stream, lambda: sp.capi.check(lib.sparsh_spmv(A0.h, dx.ptr, tb.ptr)), 20)
        nb = benchutil.csr_bytes("spmv", n, n, z)
        roof_csr["spmv"] = {"kernel": "csr_stream_kernel<256,EPI_SPMV>", "ms_per_launch": csr_spmv * 1e3, "bytes_per_launch": nb,
                            "achieved": nb / csr_spmv / 1e9, "frac": nb / csr_spmv / 1e9 / roof_csr["peak"],
                            "frac_of_8TBs_nominal": nb / csr_spmv / 1e9 / 8000.0}
        A0.force_kernel(kind, tl)
    except Exception as e:  # the solve timing above must survive a failure of the reporting extras
        roof["error"] = f"{type(e).__name__}: {e}"
    vbytes = dH.vcycle_bytes(True)
    iter_bytes = vbytes + (12 * z + 4 * (n + 1) + 16 * n) + 48 * n + 16 * n + 24 * n  # + SpMV, x/r update, dot, p update

    # true residual of the returned solution (host check of the device result, outside any timed region)
    r_true = float(np.linalg.norm(b_host - A.times(x_final)))

    cpu = None
    if not args.no_cpu_baseline:
        try:
            ref = CpuReference(grid, threads)
            per_iter = ref.sample(args.ref_iters)
            cpu = {"value": per_iter * it, "unit": UNIT, "cores": threads, "kind": "reference",
                   "sample": f"{args.ref_iters} PCG iterations of the full {grid}^3 system by the reference's own host "
                             f"code (oracle/_ref: unmodified sources + OpenMP MKL shim), seconds/iteration x {it} "
                             f"iterations (the reference needs the same {reference_iterations(grid)}: tests/golden); "
                             f"reference setup {ref.ref.setup_seconds:.1f}s not included",
                   "seconds_per_pcg_iteration": per_iter}
        except Exception as e:  # the checker is optional for the measurement itself
            cpu = {"value": None, "unit": UNIT, "cores": threads, "kind": "reference", "sample": f"unavailable: {e}"}

    line = {"metric": METRIC, "value": solve_s, "unit": UNIT, "n_gpus": 1, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": solve_s * 1e3, "higher_is_better": False,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": benchutil.workload(grid, amg.nlevels), "grid": grid, "rows": n, "nnz": z},
            "details": {"pcg_iterations": it, "reference_pcg_iterations": reference_iterations(grid),
                        "final_rel_residual": float(hist[-1] / hist[0]),
                        "true_rel_residual": r_true / float(np.linalg.norm(b_host)),
                        "ms_per_pcg_iteration": solve_s * 1e3 / max(it, 1),
                        "iteration_algorithmic_gb": iter_bytes / 1e9,
                        "solve_effective_gbs": iter_bytes * it / solve_s / 1e9,
                        "l2": "inputs larger than L2 (finest matrix 1.4 GB vs 126 MB): no flush needed", "cuda_graph": True,
                        "host_setup_seconds": rep["setup_seconds"], "upload_seconds": rep2["upload_seconds"],
                        "galerkin_products": "device (csrc/rap.cu)" if args.gpu_rap else "host (host/setup.cpp)",
                        "matrix_generation_seconds": t_gen},
            "e2e": {"value": e2e_s, "unit": UNIT, "h2d_bytes_per_step": 2 * n * 8, "d2h_bytes_per_step": n * 8,
                    "pcg_iterations": it_h},
            "gpu_launches": int(launches),
            "roofline": roof, "roofline_csr": roof_csr, "kernels": kernels,
            "cpu_baseline": cpu, "clocks": clocks}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--grid", type=int, default=256, help="grid side n of the n^3 Poisson problem")
    ap.add_argument("--max-iter", type=int, default=1000)
    ap.add_argument("--ref-iters", type=int, default=2, help="PCG iterations per bounded CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--tail-threshold", type=int, default=1100000,
                    help="N>1: levels with at most this many rows are replicated on every GPU instead of partitioned")
    ap.add_argument("--share-hierarchy", action="store_true",
                    help="N>1: rank 0 builds the host hierarchy once, the other ranks map it (needed beyond 256^3)")
    ap.add_argument("--halo-mode", type=int, default=1, help="N>1: 1 NVLink peer-memory pushes, 0 ncclSend/ncclRecv")
    ap.add_argument("--gpu-rap", action="store_true",
                    help="N=1: the Galerkin products of the (untimed) host setup run on the device (same hierarchy, bit for bit)")
    ap.add_argument("--dump-hist", default=None, help="N=1: write the PCG residual history of the solve to this JSON file")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="N=1: after the timed steps write the solution x of the last device-timed solve (x.npy), of the "
                         "last e2e solve (x_e2e.npy) and the residual history (residual_history.npy) as float64 .npy "
                         f"files to DIR; above {DUMP_ROWS} rows x is sampled at the fixed rows of x_index.npy")
    ap.add_argument("--profile", action="store_true",
                    help="for ncu: honour --warmup/--max-iter literally, do not insist on convergence")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.gpus > 1 or args.impl != "ours"):
        ap.error("--dump-outputs is implemented for this repository's path on one GPU")
    if args.grid != 256:  # the headline metric is quoted at 256^3; other grids are named for what they are
        global METRIC
        METRIC = f"amg_pcg_solve_seconds_poisson3d_{args.grid}"
    if args.impl == "reference":
        run_reference(args)
        return
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # started without the launcher: become `torchrun --nproc-per-node N bench.py ...` (one process per GPU)
        port = str(29500 + os.getpid() % 400)
        os.execv(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                                  f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1", "--master-port", port,
                                  os.path.abspath(__file__)] + sys.argv[1:])
    run_ours(args)


if __name__ == "__main__":
    main()

"""Kernel-level timing probe (developer tool; run under gpurun).

Times the SpMV-family kernels and BLAS-1 on synthetic Poisson matrices with CUDA events on the library's stream and
prints achieved algorithmic GB/s (SURVEY §8d byte model) per kernel family.  Usage:
    python tools/perf_probe.py [--n 256] [--dim 3] [--reps 20] [--families all|default]
The csr-pattern8 kernels are probed when the twin exists (default: the lean kernel where it applies, the table kernel
elsewhere).  The dict families need SPARSH_DICT=2 (the dict twin is not built where csr-pattern8 is selected).
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import sparsh_amg_b200 as sp  # noqa: E402
from sparsh_amg_b200 import generators  # noqa: E402


def timed(stream, fn, reps, warm=3):
    for _ in range(warm):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1) / reps * 1e-3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--dim", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--families", default="all")
    ap.add_argument("--matrix", default="poisson", choices=["poisson", "diffusion27", "sa_coarse"],
                    help="poisson: 7-/5-point Poisson n^dim; diffusion27: the 27-point variable-coefficient operator of "
                         "BASELINE config 4 (plain CSR: nothing repeats); sa_coarse: level 1 of its smoothed-aggregation "
                         "hierarchy (50-60 nnz/row)")
    args = ap.parse_args()
    sp.init(0)
    stream = torch.cuda.Stream()
    sp.set_stream(stream.cuda_stream)
    peak = 6537.3
    try:
        peak = json.load(open(os.path.join(os.path.dirname(__file__), "..", "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        pass
    t0 = time.time()
    if args.matrix == "poisson":
        A = generators.poisson_7pt(args.n, args.n, args.n) if args.dim == 3 else generators.poisson_5pt(args.n, args.n)
    else:
        from sparsh_amg_b200 import host

        host.set_options(threads=os.cpu_count() or 1, max_levels=32, print_setup=0, print_solve=0, coarsening=2)
        D = host.HostMatrix.diffusion27(args.n, args.n, args.n)
        if args.matrix == "diffusion27":
            A = generators.HostCSR(D.nrow, D.nrow, D.rowptr.copy(), D.colindex.copy(), D.val.copy())
        else:
            L1 = host.HostAmg(D).levels()[1]["A"]
            A = generators.HostCSR(L1.nrow, L1.ncol, L1.rowptr.copy(), L1.colindex.copy(), L1.val.copy())
    print(f"# matrix {args.matrix} {args.dim}D n={A.nrow} nnz={A.nnz} ({A.nnz / A.nrow:.1f} per row) generated in "
          f"{time.time()-t0:.1f}s", flush=True)
    m, z = A.nrow, A.nnz
    dA = sp.DeviceMatrix.from_csr(A)
    print("# default kernel:", dA.kernel())
    rng = np.random.default_rng(0)
    x, b, y, t = (sp.DeviceVector(data=rng.standard_normal(m)) for _ in range(4))
    bytes_spmv = 12 * z + 4 * (m + 1) + 8 * m + 8 * m
    bytes_res = 12 * z + 4 * (m + 1) + 8 * m + 16 * m
    bytes_jac = 12 * z + 4 * (m + 1) + 32 * m
    lib = sp.capi.load()
    ck = sp.capi.check  # a failed launch must not be timed as a success
    fams = [("default", None, None)]
    if args.families == "pattern":
        fams += [("pattern128", 4, 128), ("pattern256", 4, 256)]
    if args.families == "all":
        fams += [("dict256", 3, 256), ("dict128", 3, 128), ("stream256", 1, 256), ("stream128", 1, 128),
                 ("vector4", 2, 4), ("scalar", 0, 256)]
        if os.environ.get("SPARSH_PATTERN", "1") in ("1", "2"):
            fams[1:1] = [("pattern128", 4, 128), ("pattern256", 4, 256)]
    for name, kind, tl in fams:
        if kind is not None:
            dA.force_kernel(kind, tl)
        ops = [("spmv", bytes_spmv, 1, lambda: ck(lib.sparsh_spmv(dA.h, x.ptr, y.ptr))),
               ("residual", bytes_res, 1, lambda: ck(lib.sparsh_residual(dA.h, b.ptr, x.ptr, y.ptr))),
               ("jacobi_sweep", bytes_jac, 2, lambda: ck(lib.sparsh_jacobi(dA.h, b.ptr, x.ptr, t.ptr, 0.66667, 2))),
               ("spmv_dot", bytes_spmv, 1, lambda: ck(lib.sparsh_spmv_dot(dA.h, x.ptr, y.ptr, t.ptr)))]
        for op, nb, div, fn in ops:
            try:
                dt = timed(stream, fn, args.reps) / div
                ck(lib.sparsh_sync())
            except sp.SparshError as e:  # a launch the library refused is reported, never timed
                print(f"{name:10s} {op:13s} not run: {e}", flush=True)
                continue
            gbs = nb / dt / 1e9
            print(f"{name:10s} {op:13s} {dt*1e3:8.4f} ms  {gbs:8.1f} GB/s  {gbs/peak:6.3f} of measured copy "
                  f"({gbs/8000:5.3f} of 8 TB/s)", flush=True)
    # BLAS-1
    dt = timed(stream, lambda: ck(lib.sparsh_axpy(m, 0.5, x.ptr, y.ptr)), args.reps)
    print(f"blas1      axpy          {dt*1e3:8.4f} ms  {24*m/dt/1e9:8.1f} GB/s")
    dt = timed(stream, lambda: ck(lib.sparsh_axpby(m, 0.5, x.ptr, 0.25, y.ptr)), args.reps)
    print(f"blas1      axpby         {dt*1e3:8.4f} ms  {24*m/dt/1e9:8.1f} GB/s")
    dt = timed(stream, lambda: ck(lib.sparsh_fill(y.ptr, m, 0.0)), args.reps)
    print(f"blas1      fill          {dt*1e3:8.4f} ms  {8*m/dt/1e9:8.1f} GB/s")
    hv = np.zeros(1)
    import ctypes as C
    dt = timed(stream, lambda: ck(lib.sparsh_dot(m, x.ptr, b.ptr, hv.ctypes.data_as(C.POINTER(C.c_double)))), args.reps)
    print(f"blas1      dot(+sync)    {dt*1e3:8.4f} ms  {16*m/dt/1e9:8.1f} GB/s")
    # torch copy on the same stream as a sanity reference for the peak
    with torch.cuda.stream(stream):
        a = torch.empty(1 << 28, dtype=torch.float64, device="cuda")
        c = torch.empty_like(a)
        dt = timed(stream, lambda: c.copy_(a), 10)
    print(f"torch      copy 2GiB     {dt*1e3:8.4f} ms  {2*a.numel()*8/dt/1e9:8.1f} GB/s")


if __name__ == "__main__":
    main()

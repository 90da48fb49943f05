"""Per-level kernel probe of the bench hierarchy (developer tool; needs a GPU).

bench.py times the row-sum kernels of level 0 only.  This builds and uploads the hierarchy exactly as bench.py does (3D
7-point Poisson n^3, native HEM setup, V(7,7) Jacobi) and times, on EVERY level, the kernel the library selects for the
fused Jacobi sweep, the residual, the SpMV and the SpMV+dot, with CUDA events on the library's stream over enough launches
to fill about 20 ms (at least --min-reps).  It prints rows, kernel, ms per launch and GB/s of the bytes the kernel has to
move in its storage format (benchutil.stored_bytes), and writes everything, with the GPU's name and power limit, as JSON.
Launches are issued one by one from the host, not from a graph as in the solve: on the small levels a kernel can end
before the host has enqueued the next one, and the events then time the enqueue rate, not the kernel.  The probe times
that floor (a one-element fill per call) and marks every row within 1.5x of it `launch_bound`: its ms and GB/s are
upper / lower bounds, not kernel figures.
    python tools/level_probe.py [--grid 256] [--out level_probe.json] [--census]
On every level but the coarsest it also times the grid transfers of the V-cycle against the kernels they replace:
resid_restrict (fused residual + restriction, sparsh_residual_restrict) against resid+restrict (sparsh_residual into a
vector, then sparsh_restrict), prolong (the default: the aggregation kernel for HEM's P) against prolong_scalar (P forced
to KIND_SCALAR), and zero_sweep (x = (omega*b)/d, sparsh_jacobi_zero: d through the pattern twin) against
zero_sweep_diag (the same with A forced to the stream kernel, which reads the diagonal array; timed last on a level, as
the forcing is not undone).  Their stored bytes count each array once: pattern byte 1, b / x / vectors 8, R / P column
4, rowptr 4 per row, values 8 unless the operator passes its one value by value.
--census adds, per level, what the csr-pattern8 encoder makes of the level (host encoder, no GPU time): patterns, rows
of pattern 0, patterns the lean kernel runs as masked pattern 0, and the share of 32-row warps that mix pattern-0 rows with
rows of other patterns.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import sparsh_amg_b200 as sp  # noqa: E402
from sparsh_amg_b200 import benchutil, host  # noqa: E402


def gpu_info():
    """name and power limit of the card (a read-only query)"""
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in out.split(",")]
    except Exception as e:  # the timings do not depend on it; the report says it is missing
        info["power_limit"] = f"unavailable: {e}"
    return info


def census(lib, levels):
    """per level: the host encoder's table and masks, and the share of 32-row warps mixing pattern 0 with other rows"""
    out = []
    for k, L in enumerate(levels):
        M, n = L["A"], L["A"].nrow
        pat = np.empty(n, dtype=np.uint8)
        ev, eo, st = np.zeros(2048), np.zeros(2048, dtype=np.int32), np.zeros(257, dtype=np.int32)
        npat, nesc = C.c_int(), C.c_int()
        sp.capi.check(lib.sparsh_pattern_encode(n, M.ncol, M.nnz, sp.capi.ip(M.rowptr), sp.capi.ip(M.colindex), sp.capi.dp(M.val),
                                                sp.capi.dp(np.ascontiguousarray(L["diag"])), pat.ctypes.data_as(C.c_void_p),
                                                sp.capi.dp(ev), sp.capi.ip(eo), sp.capi.ip(st), C.byref(npat), C.byref(nesc)))
        mask = np.zeros(256, dtype=np.uint8)
        sp.capi.check(lib.sparsh_pattern_masks(npat.value, sp.capi.ip(st), sp.capi.dp(ev), sp.capi.ip(eo), mask.ctypes.data_as(C.c_void_p)))
        warps = np.concatenate([pat, np.zeros((-n) % 32, dtype=np.uint8)]).reshape(-1, 32)
        zero = warps == 0
        mixed = zero.any(axis=1) & ~zero.all(axis=1)
        masked = (mask[pat] & 0x80) != 0
        out.append({"level": k, "rows": n, "patterns": npat.value, "escapes": nesc.value, "cover0": float(np.mean(pat == 0)),
                    "masked_patterns": int(np.count_nonzero(mask[1:npat.value] & 0x80)), "other_patterns": npat.value - 1,
                    "cover_masked": float(np.mean(masked)), "mixed_warps": float(np.mean(mixed))})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", type=int, default=256)
    ap.add_argument("--min-reps", type=int, default=20)
    ap.add_argument("--target-ms", type=float, default=20.0, help="launches per timing: enough to fill about this long")
    ap.add_argument("--out", default=None, help="JSON file to write")
    ap.add_argument("--census", action="store_true")
    args = ap.parse_args()

    sp.init(0)
    stream = torch.cuda.Stream()
    sp.set_stream(stream.cuda_stream)
    lib = sp.capi.load()
    host.set_options(threads=os.cpu_count() or 1, max_levels=32, print_setup=0, print_solve=0, coarsening=0, sweeps=7,
                     use_graph=1)
    t0 = time.time()
    A = host.HostMatrix.poisson3d(args.grid, args.grid, args.grid)
    amg = host.HostAmg(A)
    dH = amg.upload()
    host_levels = amg.levels()
    gpu = gpu_info()
    print(f"# {args.grid}^3 HEM hierarchy, {dH.nlevels} levels, built and uploaded in {time.time() - t0:.1f} s; {gpu}", flush=True)
    ck = sp.capi.check
    one = sp.DeviceVector(1)
    fill = lambda: ck(lib.sparsh_fill(one.ptr, 1, 0.0))  # noqa: E731
    benchutil.timed(torch, stream, fill, 100)
    floor = benchutil.timed(torch, stream, fill, 2000)
    print(f"# enqueue floor: {floor * 1e6:.2f} us per launch (rows within 1.5x of it are marked launch-bound)", flush=True)
    rows = []
    def timed_row(k, n, z, op, kernel, per_call, kernels, fn, nb):
        once = benchutil.timed(torch, stream, fn, 3)
        reps = max(args.min_reps, min(5000, int(args.target_ms * 1e-3 / max(once, 1e-7))))
        sec = benchutil.timed(torch, stream, fn, reps) / per_call
        row = {"level": k, "rows": n, "nnz": z, "op": op, "kernel": kernel, "launches": reps * per_call,
               "ms": sec * 1e3, "stored_bytes": nb, "gbs": nb / sec / 1e9, "launch_bound": sec * per_call <= 1.5 * floor * kernels}
        print(f"L{k:<2d} {n:>9d} rows  {op:15s} {row['kernel']:40s} {row['ms']:9.5f} ms  {row['gbs']:8.1f} GB/s  "
              f"({row['launches']} launches){'  launch-bound' if row['launch_bound'] else ''}", flush=True)
        return row

    for k in range(dH.nlevels):
        Ak, Pk, Rk = dH.level(k)
        n, m, z = Ak.nrow, Ak.ncol, Ak.nnz
        kind = Ak.kernel()[0]
        rng = np.random.default_rng(k)
        x, b, y, t = (sp.DeviceVector(data=rng.standard_normal(n)) for _ in range(4))
        dsc = sp.DeviceVector(8).fill(0.0)
        ops = [("jacobi", 2, 2, lambda: ck(lib.sparsh_jacobi(Ak.h, b.ptr, x.ptr, t.ptr, 0.66667, 2))),
               ("residual", 1, 1, lambda: ck(lib.sparsh_residual(Ak.h, b.ptr, x.ptr, y.ptr))),
               ("spmv", 1, 1, lambda: ck(lib.sparsh_spmv(Ak.h, x.ptr, y.ptr))),
               ("spmv_dot", 1, 2, lambda: ck(lib.sparsh_spmv_dot(Ak.h, x.ptr, y.ptr, dsc.ptr)))]
        for op, per_call, kernels, fn in ops:  # per_call: sweeps per call; kernels: launches per call (+ finalize)
            rows.append(timed_row(k, n, z, op, Ak.kernel_name(op), per_call, kernels, fn, benchutil.stored_bytes(kind, op, n, m, z)))
        if Pk is None:
            continue
        mc = Pk.ncol
        r, bc, xc = sp.DeviceVector(n), sp.DeviceVector(mc), sp.DeviceVector(data=rng.standard_normal(mc))
        one, uni, _ = Pk.transfer_info()
        hP = host_levels[k]["P"]  # a private copy of P on the plain scalar kernel
        Pf = sp.DeviceMatrix(hP.nrow, hP.ncol, hP.rowptr, hP.colindex, hP.val).force_kernel(sp.capi.KIND_SCALAR, 256)
        pair_nb = benchutil.stored_bytes(kind, "residual", n, m, z) + 4 * (mc + 1) + 12 * Pk.nnz + 8 * n + 8 * mc
        fused_nb = n + 16 * n + 4 * (mc + 1) + 4 * Pk.nnz + 8 * mc + (0 if Rk.transfer_info()[1] else 8 * Pk.nnz)
        xfer = [("resid+restrict", f"{Ak.kernel_name('residual')} + {Rk.kernel_name('spmv')}", 2,
                 lambda: (ck(lib.sparsh_residual(Ak.h, b.ptr, x.ptr, r.ptr)), ck(lib.sparsh_restrict(Rk.h, r.ptr, bc.ptr))), pair_nb),
                ("resid_restrict", "resid_restrict_kernel" if Ak.kernel_name("residual").startswith("csr_pat2") and Rk.transfer_info()[1]
                 else "(two launches)", 1, lambda: ck(lib.sparsh_residual_restrict(Ak.h, Rk.h, b.ptr, x.ptr, bc.ptr)), fused_nb),
                ("prolong_scalar", Pf.kernel_name("prolong"), 1, lambda: ck(lib.sparsh_prolong_add(Pf.h, xc.ptr, y.ptr)),
                 4 * (n + 1) + 12 * Pk.nnz + 8 * mc + 16 * n),
                ("prolong", Pk.kernel_name("prolong"), 1, lambda: ck(lib.sparsh_prolong_add(Pk.h, xc.ptr, y.ptr)),
                 (4 * n + (0 if uni else 8 * n) if one else 4 * (n + 1) + 12 * Pk.nnz) + 8 * mc + 16 * n),
                ("zero_sweep", "jacobi_zero_pat_kernel" if Ak.kernel_name("jacobi").startswith("csr_pat2") else "jacobi_zero_kernel", 1,
                 lambda: ck(lib.sparsh_jacobi_zero(Ak.h, b.ptr, 0.66667, t.ptr)),
                 17 * n if Ak.kernel_name("jacobi").startswith("csr_pat2") else 24 * n)]
        for op, kname, kernels, fn, nb in xfer:
            rows.append(timed_row(k, n, z, op, kname, 1, kernels, fn, nb))
        if Ak.kernel()[0] == sp.capi.KIND_PATTERN:
            Ak.force_kernel(sp.capi.KIND_STREAM, 128)  # not undone: nothing else runs on this level afterwards
            rows.append(timed_row(k, n, z, "zero_sweep_diag", "jacobi_zero_kernel", 1, 1,
                                  lambda: ck(lib.sparsh_jacobi_zero(Ak.h, b.ptr, 0.66667, t.ptr)), 24 * n))
        Pf.free()
    out = {"grid": args.grid, "levels": dH.nlevels, "gpu": gpu, "enqueue_floor_ms": floor * 1e3, "timings": rows}
    if args.census:
        out["census"] = census(lib, amg.levels())
        for c in out["census"]:
            print(f"census L{c['level']:<2d} {c['rows']:>9d} rows  cover0 {c['cover0']:.3f}  masked {c['masked_patterns']}/"
                  f"{c['other_patterns']}  cover0+masked {c['cover_masked']:.3f}  mixed warps {c['mixed_warps']:.3f}", flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()

"""What a coefficient refresh costs against a new setup (developer tool; needs a GPU).

Builds the bench hierarchy (3D 7-point Poisson n^3, native HEM setup, V(7,7) Jacobi) with the host setup and uploads it,
timing both.  Then, with new level-0 values A_0 + sigma I (the time-step case):
  refresh         sparsh_hierarchy_refresh with the values already on the device, host clock around the call (it ends
                  with a device synchronise).  The first call also builds the plan; the steady state is the median of
                  the calls after it.
  refresh_h2d     the same preceded by the host-to-device copy of the values.
  breakdown       one more refresh with SPARSH_REFRESH_TIMING set: per level the product, the twins and the coarse
                  inverse (each phase synchronised, so their sum exceeds the plain refresh), and the product's GB/s on
                  the bytes it has to move (A_l, P_l and R_l read once, A_{l+1}'s rowptr and columns read, its values
                  written).
A PCG solve runs before and after the refresh, and the refreshed result is compared bit for bit with a fresh hierarchy
built from the new A_0, the same P_l and the device Galerkin products.  Writes JSON (--out) with the GPU's name and
power limit.
    python tools/refresh_probe.py [--grid 256] [--reps 5] [--out refresh_probe.json]
"""
import argparse
import json
import os
import re
import statistics
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from level_probe import gpu_info  # noqa: E402  (also puts the repository on sys.path)

import sparsh_amg_b200 as sp  # noqa: E402
from sparsh_amg_b200 import host  # noqa: E402
from sparsh_amg_b200.generators import HostCSR  # noqa: E402


def csr_copy(A):
    return HostCSR(A.nrow, A.ncol, np.array(A.rowptr), np.array(A.colindex), np.array(A.val))


def extracted_diag(A):
    rows = np.repeat(np.arange(A.nrow), np.diff(A.rowptr))
    d = np.zeros(A.nrow)
    hit = np.flatnonzero(A.colindex == rows)
    first = np.unique(rows[hit], return_index=True)  # the first stored entry with col == row
    d[first[0]] = A.val[hit[first[1]]]
    return d


def timed_refresh(dH, dv):
    t = time.perf_counter()
    dH.refresh(dv)
    return time.perf_counter() - t


def refresh_breakdown(dH, dv):
    """one refresh with SPARSH_REFRESH_TIMING: its stderr lines, parsed"""
    os.environ["SPARSH_REFRESH_TIMING"] = "1"
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as f:
        os.dup2(f.fileno(), 2)
        try:
            dH.refresh(dv)
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["SPARSH_REFRESH_TIMING"]
        f.seek(0)
        text = f.read()
    out = {"levels": [], "coarse_inverse_s": None}
    for line in text.splitlines():
        if m := re.match(r"\[refresh\] level (\d+): product ([\d.]+) s \((\w+)\) twins ([\d.]+) s", line):
            out["levels"].append({"level": int(m[1]), "product_s": float(m[2]), "product": m[3], "twins_s": float(m[4])})
        elif m := re.match(r"\[refresh\] level 0: twins ([\d.]+) s", line):
            out["levels"].append({"level": 0, "product_s": 0.0, "product": None, "twins_s": float(m[1])})
        elif m := re.match(r"\[refresh\] coarse inverse \(n = (\d+)\): ([\d.]+) s", line):
            out["coarse_inverse_s"], out["coarse_n"] = float(m[2]), int(m[1])
    return out


def product_bytes(dH, k):
    """bytes the product of level k (k >= 1) has to move: A_{k-1}, P, R read once, A_k's rowptr and columns read and its
    values written"""
    A, P, R = dH.level(k - 1)
    C = dH.level(k)[0]
    csr = lambda M: 4 * (M.nrow + 1) + 12 * M.nnz  # noqa: E731
    return csr(A) + 12 * P.nnz + csr(R) + 4 * (C.nrow + 1) + 12 * C.nnz


def pcg(dH, b):
    x = sp.DeviceVector(dH.n).fill(0.0)
    t = time.perf_counter()
    it, hist, ok = dH.pcg(sp.DeviceVector(data=b), x, 1e-8, max_iter=500)
    return {"iterations": it, "converged": bool(ok), "seconds": time.perf_counter() - t}, hist, x.download()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", type=int, default=256)
    ap.add_argument("--sigma", type=float, default=0.05)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    n = args.grid
    sp.init(0)
    gpu = gpu_info()
    host.set_options(threads=os.cpu_count() or 1, max_levels=32, print_setup=0, print_solve=0, coarsening=0, sweeps=7,
                     use_graph=1)
    M = host.HostMatrix.poisson3d(n, n, n)
    t0 = time.perf_counter()
    amg = host.HostAmg(M)
    t1 = time.perf_counter()
    dH = amg.upload()
    t2 = time.perf_counter()
    levels = amg.levels()
    rep = {"grid": n, "gpu": gpu, "levels": dH.nlevels, "rows": dH.n, "setup_s": t1 - t0, "upload_s": t2 - t1}
    print(f"# {n}^3 HEM, {dH.nlevels} levels; {gpu}", flush=True)
    print(f"host setup {rep['setup_s']:.3f} s, upload {rep['upload_s']:.3f} s", flush=True)

    b = np.ones(dH.n)
    rep["pcg_before"], _, _ = pcg(dH, b)
    pcg(dH, b)  # the graphs of the solve are captured now: the refresh has to drop them
    A0 = csr_copy(levels[0]["A"])
    rows = np.repeat(np.arange(A0.nrow), np.diff(A0.rowptr))
    v_new = A0.val.copy()
    v_new[A0.colindex == rows] += args.sigma
    v_old = A0.val.copy()
    dv_new, dv_old = sp.DeviceVector(data=v_new), sp.DeviceVector(data=v_old)

    rep["refresh_first_s"] = timed_refresh(dH, dv_new)  # builds the plan
    steady = []
    for _ in range(args.reps):  # alternate values so every call really changes the coefficients
        steady.append(timed_refresh(dH, dv_old))
        steady.append(timed_refresh(dH, dv_new))
    rep["refresh_s"] = steady
    rep["refresh_median_s"] = statistics.median(steady)
    h2d = []
    for _ in range(args.reps):
        t = time.perf_counter()
        dv_new.upload(v_new)
        dH.refresh(dv_new)
        h2d.append(time.perf_counter() - t)
    rep["refresh_h2d_s"] = h2d
    rep["refresh_h2d_median_s"] = statistics.median(h2d)
    rep["setup_plus_upload_over_refresh"] = (rep["setup_s"] + rep["upload_s"]) / rep["refresh_median_s"]
    print(f"refresh (values on the device): first {rep['refresh_first_s']:.4f} s, median {rep['refresh_median_s']:.4f} s "
          f"(min {min(steady):.4f}, max {max(steady):.4f}); with the H2D copy: median {rep['refresh_h2d_median_s']:.4f} s; "
          f"setup + upload = {rep['setup_plus_upload_over_refresh']:.1f} x refresh", flush=True)

    bd = refresh_breakdown(dH, dv_new)
    for L in bd["levels"]:
        if L["level"] > 0:
            L["product_bytes"] = product_bytes(dH, L["level"])
            L["product_gbs"] = L["product_bytes"] / L["product_s"] / 1e9 if L["product_s"] > 0 else None
        print(f"L{L['level']:<2d} product {L['product_s'] * 1e3:9.3f} ms ({L['product'] or '-':11s}"
              f"{'' if L.get('product_gbs') is None else f', {L['product_gbs']:7.1f} GB/s'}) twins {L['twins_s'] * 1e3:9.3f} ms",
              flush=True)
    print(f"coarse inverse (n = {bd.get('coarse_n')}): {bd['coarse_inverse_s'] * 1e3:.3f} ms", flush=True)
    rep["breakdown"] = bd

    rep["pcg_after"], hist, x = pcg(dH, b)
    fresh_levels = []
    A = HostCSR(A0.nrow, A0.ncol, A0.rowptr, A0.colindex, v_new)
    for k, L in enumerate(levels):
        fresh_levels.append(dict(A=A, diag=extracted_diag(A), P=L["P"]))
        if L["P"] is not None:
            rp, ci, v = sp.galerkin_rap(A, L["P"])
            A = HostCSR(L["P"].ncol, L["P"].ncol, rp, ci, v)
    fresh = sp.DeviceHierarchy(fresh_levels)
    rep["pcg_fresh"], hist_f, x_f = pcg(fresh, b)
    rep["bit_identical_to_fresh"] = bool(len(hist) == len(hist_f) and np.array_equal(hist.view(np.uint64), hist_f.view(np.uint64))
                                         and np.array_equal(x.view(np.uint64), x_f.view(np.uint64)))
    print(f"PCG before: {rep['pcg_before']}; after the refresh: {rep['pcg_after']}; fresh hierarchy: {rep['pcg_fresh']}; "
          f"refreshed == fresh bit for bit: {rep['bit_identical_to_fresh']}", flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rep, f, indent=1)
    fresh.free()
    amg.free()
    if not rep["bit_identical_to_fresh"]:
        sys.exit(1)


if __name__ == "__main__":
    main()

"""What the host-driven solve loop costs against the device-driven one (developer tool; needs a GPU).

For the bench hierarchy (3D 7-point Poisson n^3, native HEM setup, V(7,7) Jacobi, graphs on) at --grid and at --small,
AMG-PCG from x0 = 0 to tol = 1e-8 ||b||, b = ones, on a torch stream adopted with sp.set_stream (as bench.py does):
  sync      DeviceHierarchy.pcg: one graph launch per iteration, then a copy of ||r||^2 to the host and a synchronise
  enqueue   DeviceHierarchy.pcg_enqueue: the loop is a conditional WHILE node on the device; nothing waits until
            PendingSolve.result()
  device time per solve   CUDA events on the stream around the solve (x0 = 0 fill included in both), after a warm-up
                          of both; A and B alternate --reps times
  enqueue host time       host clock around the pcg_enqueue call alone (median of --reps), the solve still running
  gap per iteration       (sync - enqueue) / iterations: what the host round trip of each iteration adds
Both paths must give the same x and history bit for bit; the report says whether they did.  The GPU's name, power limit
and max SM clock are read in the same run.
    python tools/enqueue_probe.py [--grid 256] [--small 64] [--reps 3] [--out enqueue_probe.json]
"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from level_probe import gpu_info  # noqa: E402  (also puts the repository on sys.path)

import torch  # noqa: E402

import sparsh_amg_b200 as sp  # noqa: E402
from sparsh_amg_b200 import host  # noqa: E402


def probe(grid, reps, stream):
    host.set_options(threads=os.cpu_count() or 1, max_levels=32, print_setup=0, print_solve=0, coarsening=0, sweeps=7,
                     use_graph=1)
    amg = host.HostAmg(host.HostMatrix.poisson3d(grid, grid, grid))
    dH = amg.upload()
    n = dH.n
    b = np.ones(n)
    tol, max_iter = 1e-8 * float(np.linalg.norm(b)), 500
    db, dx = sp.DeviceVector(data=b), sp.DeviceVector(n)
    pend = sp.PendingSolve(max_iter)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

    def sync_solve():
        ev[0].record(stream)
        dx.fill(0.0)
        it, hist, ok = dH.pcg(db, dx, tol, max_iter)
        ev[1].record(stream)
        ev[1].synchronize()
        return ev[0].elapsed_time(ev[1]) * 1e-3, (it, hist, ok)

    def enqueued_solve():
        ev[0].record(stream)
        dx.fill(0.0)
        t = time.perf_counter()
        dH.pcg_enqueue(db, dx, tol, max_iter, pending=pend)
        host_s = time.perf_counter() - t
        ev[1].record(stream)
        ev[1].synchronize()
        return ev[0].elapsed_time(ev[1]) * 1e-3, pend.result(), host_s

    for _ in range(2):  # warm-up of both paths (the first enqueue builds the solve graph)
        sync_solve()
        enqueued_solve()
    t_sync, t_enq, t_host = [], [], []
    for _ in range(reps):
        s, (it_s, hist_s, ok_s) = sync_solve()
        x_s = dx.download()
        e, (it_e, hist_e, ok_e), h = enqueued_solve()
        x_e = dx.download()
        t_sync.append(s)
        t_enq.append(e)
        t_host.append(h)
    same = bool(it_s == it_e and ok_s == ok_e and np.array_equal(hist_s.view(np.uint64), hist_e.view(np.uint64))
                and np.array_equal(x_s.view(np.uint64), x_e.view(np.uint64)))
    rep = {"grid": grid, "rows": n, "levels": dH.nlevels, "iterations": it_s, "converged": bool(ok_s),
           "sync_s": t_sync, "enqueue_s": t_enq, "enqueue_host_call_s": t_host,
           "sync_median_s": statistics.median(t_sync), "enqueue_median_s": statistics.median(t_enq),
           "enqueue_host_call_median_s": statistics.median(t_host), "bit_identical": same}
    rep["gap_per_iteration_s"] = (rep["sync_median_s"] - rep["enqueue_median_s"]) / max(it_s, 1)
    rep["sync_per_iteration_s"] = rep["sync_median_s"] / max(it_s, 1)
    print(f"{grid}^3 ({dH.nlevels} levels, {it_s} iterations): sync {rep['sync_median_s'] * 1e3:.3f} ms, "
          f"enqueue {rep['enqueue_median_s'] * 1e3:.3f} ms (device time per solve, median of {reps}); "
          f"gap per iteration {rep['gap_per_iteration_s'] * 1e6:.1f} us of {rep['sync_per_iteration_s'] * 1e6:.1f} us; "
          f"enqueue call on the host {rep['enqueue_host_call_median_s'] * 1e6:.1f} us; bit-identical: {same}", flush=True)
    amg.free()
    return rep


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", type=int, default=256)
    ap.add_argument("--small", type=int, default=64)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    sp.init(0)
    stream = torch.cuda.Stream()
    sp.set_stream(stream.cuda_stream)
    rep = {"gpu": gpu_info(), "cases": []}
    print(f"# {rep['gpu']}", flush=True)
    for grid in (args.grid, args.small):
        rep["cases"].append(probe(grid, args.reps, stream))
    sp.set_stream(None)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rep, f, indent=1)
    if not all(c["bit_identical"] for c in rep["cases"]):
        sys.exit(1)


if __name__ == "__main__":
    main()

"""Device-driven solves (sparsh_hierarchy_pcg_enqueue / _pbicgstab_enqueue / _amg_solve_enqueue).

The iteration loop runs on the device as a conditional WHILE node of a CUDA graph, the kernels are the synchronous
solvers' own: x, the residual history, the iteration count and the status are pinned bit for bit to the synchronous
call from the same b and x0, at the stopping edges too.  A solve recorded into a caller's torch.cuda.graph capture (which
fails on any synchronisation or allocation) replays to the same bits."""
import os

import numpy as np
import pytest
from oracle_bindings import CSR

pytestmark = pytest.mark.gpu

METHODS = ["pcg", "pbicgstab", "amg"]


@pytest.fixture(scope="module")
def sp():
    # torch first: the library links the system's libnccl, and a torch imported after it would resolve its NCCL symbols
    # there instead of in its own
    import torch  # noqa: F401

    import sparsh_amg_b200 as s

    s.init(0)
    return s


def same_bits(got, want, msg):
    """NaN where the other has NaN, the same bits everywhere else"""
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, (msg, got.shape, want.shape)
    nan = np.isnan(want)
    np.testing.assert_array_equal(np.isnan(got), nan, err_msg=msg)
    np.testing.assert_array_equal(np.ascontiguousarray(got[~nan]).view(np.uint64),
                                  np.ascontiguousarray(want[~nan]).view(np.uint64), err_msg=msg)


def host_levels(kind, n=32):
    """(levels as CSR copies, the HostAmg) for 'hem' | 'beck' | 'sa' | 'sor' (HEM, multicolour SOR) on 3D Poisson n^3"""
    from sparsh_amg_b200 import host

    host.set_options(threads=min(8, os.cpu_count() or 1), max_levels=32, print_setup=0, print_solve=0,
                     coarsening={"hem": 0, "beck": 1, "sa": 2, "sor": 0}[kind], relax=0.66667,
                     coarse_upper=500 if kind == "sa" else 4000, coarse_lower=100 if kind == "sa" else 2000)
    amg = host.HostAmg(host.HostMatrix.poisson3d(n, n, n), sor=kind == "sor")
    levels = []
    for L in amg.levels():
        A, P = L["A"], L["P"]
        levels.append(dict(A=CSR(A.nrow, A.ncol, A.rowptr.copy(), A.colindex.copy(), A.val.copy()), diag=np.array(L["diag"]),
                           P=None if P is None else CSR(P.nrow, P.ncol, P.rowptr.copy(), P.colindex.copy(), P.val.copy())))
    return levels, amg


def hierarchy(sp, kind, n=32):
    levels, amg = host_levels(kind, n)
    return (amg.upload() if kind == "sor" else sp.DeviceHierarchy(levels)), levels, amg


def sync_solve(sp, dH, method, b, x0, tol, max_iter):
    x = sp.DeviceVector(data=x0)
    fn = {"pcg": dH.pcg, "pbicgstab": dH.pbicgstab, "amg": dH.amg_solve}[method]
    it, hist, ok = fn(sp.DeviceVector(data=b), x, tol, max_iter)
    return it, hist, ok, x.download()


def enqueued_solve(sp, dH, method, b, x0, tol, max_iter, pending=None):
    x = sp.DeviceVector(data=x0)
    fn = {"pcg": dH.pcg_enqueue, "pbicgstab": dH.pbicgstab_enqueue, "amg": dH.amg_solve_enqueue}[method]
    it, hist, ok = fn(sp.DeviceVector(data=b), x, tol, max_iter, pending=pending).result()
    return it, hist, ok, x.download()


def assert_same_solve(got, want, msg):
    assert got[0] == want[0], (msg, got[0], want[0])
    assert got[2] == want[2], msg
    same_bits(got[1], want[1], f"{msg} history")
    same_bits(got[3], want[3], f"{msg} x")


@pytest.mark.parametrize("kind", ["hem", "beck", "sa", "sor"])
@pytest.mark.parametrize("method", METHODS)
def test_enqueued_solve_equals_the_synchronous_one(sp, kind, method):
    dH, levels, amg = hierarchy(sp, kind)
    rng = np.random.default_rng(11)
    b, x0 = rng.standard_normal(dH.n), rng.standard_normal(dH.n)
    tol = 1e-8 * np.linalg.norm(b)
    want = sync_solve(sp, dH, method, b, x0, tol, 300)
    assert want[0] > 2, want[0]
    bv, xv = sp.DeviceVector(data=b), sp.DeviceVector(dH.n)
    fn = {"pcg": dH.pcg_enqueue, "pbicgstab": dH.pbicgstab_enqueue, "amg": dH.amg_solve_enqueue}[method]
    for call in range(2):  # the same vectors: the first call builds the solve graph, the second replays it
        got = fn(bv, xv.upload(x0), tol, 300).result() + (xv.download(),)
        assert_same_solve(got, want, f"{kind} {method} call {call}")
    amg.free()


@pytest.mark.parametrize("method", METHODS)
def test_stopping_edges_match_the_synchronous_solve(sp, method):
    dH, levels, amg = hierarchy(sp, "hem")
    rng = np.random.default_rng(12)
    b, x0 = rng.standard_normal(dH.n), rng.standard_normal(dH.n)
    # tol above the initial residual: no iteration, x untouched, converged
    got = enqueued_solve(sp, dH, method, b, x0, 1e30, 50)
    assert got[0] == 0 and got[2]
    same_bits(got[3], x0, "x untouched")
    assert_same_solve(got, sync_solve(sp, dH, method, b, x0, 1e30, 50), f"{method} tol above r0")
    # the iteration limit: not converged after exactly max_iter iterations
    got = enqueued_solve(sp, dH, method, b, x0, 0.0, 3)
    assert got[0] == 3 and not got[2]
    assert_same_solve(got, sync_solve(sp, dH, method, b, x0, 0.0, 3), f"{method} max_iter")
    # max_iter = 0
    assert_same_solve(enqueued_solve(sp, dH, method, b, x0, 1e-8, 0), sync_solve(sp, dH, method, b, x0, 1e-8, 0),
                      f"{method} max_iter 0")
    # a NaN in b: the initial residual is NaN, which stops before the first iteration
    bn = b.copy()
    bn[77] = np.nan
    got = enqueued_solve(sp, dH, method, bn, x0, 1e-8, 20)
    assert got[0] == 0 and not got[2]
    assert_same_solve(got, sync_solve(sp, dH, method, bn, x0, 1e-8, 20), f"{method} NaN in b")
    # an inf in b: the initial residual +inf iterates, the first iteration's residual is not finite, which stops the loop
    bi = b.copy()
    bi[77] = np.inf
    got = enqueued_solve(sp, dH, method, bi, x0, 1e-8, 20)
    assert got[1][0] == np.inf and 1 <= got[0] < 20 and not np.isfinite(got[1][-1]) and not got[2], got[:2]
    assert_same_solve(got, sync_solve(sp, dH, method, bi, x0, 1e-8, 20), f"{method} inf in b")
    amg.free()


def test_repeated_calls_with_other_arguments(sp):
    dH, levels, amg = hierarchy(sp, "beck")
    rng = np.random.default_rng(13)
    pend = sp.PendingSolve(300)
    cases = [(rng.standard_normal(dH.n), rng.standard_normal(dH.n), tol, mi) for tol, mi in
             ((1e-6, 300), (1e-10, 300), (1e-10, 4), (1e-3, 100))]
    for method in METHODS:
        for k, (b, x0, tol, mi) in enumerate(cases):
            msg = f"{method} case {k}"
            assert_same_solve(enqueued_solve(sp, dH, method, b, x0, tol, mi, pending=pend),
                              sync_solve(sp, dH, method, b, x0, tol, mi), msg)
    # the same device vectors with new contents (the cached graph of (b, x) replays)
    bv, xv = sp.DeviceVector(dH.n), sp.DeviceVector(dH.n)
    for b, x0, tol, mi in cases:
        bv.upload(b)
        xv.upload(x0)
        got = dH.pcg_enqueue(bv, xv, tol, mi, pending=pend).result() + (xv.download(),)
        assert_same_solve(got, sync_solve(sp, dH, "pcg", b, x0, tol, mi), f"same vectors tol={tol} max_iter={mi}")
    amg.free()


def extracted_diag(A):
    d = np.zeros(A.nrow)
    for i in range(A.nrow):
        lo, hi = A.rowptr[i], A.rowptr[i + 1]
        hit = np.flatnonzero(A.colindex[lo:hi] == i)
        if hit.size:
            d[i] = A.val[lo + hit[0]]
    return d


def shifted(A, sigma):
    v = A.val.copy()
    rows = np.repeat(np.arange(A.nrow), np.diff(A.rowptr))
    v[A.colindex == rows] += sigma
    return CSR(A.nrow, A.ncol, A.rowptr, A.colindex, v)


def galerkin_levels(sp, A0, levels):
    """A_0, the same P_l, A_{l+1} = device Galerkin product, diagonals extracted"""
    out, A = [], A0
    for L in levels:
        out.append(dict(A=A, diag=extracted_diag(A), P=L["P"]))
        if L["P"] is not None:
            A = CSR(L["P"].ncol, L["P"].ncol, *sp.galerkin_rap(A, L["P"]))
    return out


def test_refresh_drops_the_solve_graphs(sp):
    dH, levels, amg = hierarchy(sp, "hem")
    rng = np.random.default_rng(14)
    b, x0 = rng.standard_normal(dH.n), np.zeros(dH.n)
    bv, xv = sp.DeviceVector(data=b), sp.DeviceVector(dH.n)
    for _ in range(2):
        dH.pcg_enqueue(bv, xv.fill(0.0), 1e-9, 200).result()
    A0 = shifted(levels[0]["A"], 2.0)
    dH.refresh(A0.val)
    fresh = sp.DeviceHierarchy(galerkin_levels(sp, A0, levels))
    want = sync_solve(sp, fresh, "pcg", b, x0, 1e-9, 200)
    for _ in range(2):
        got = dH.pcg_enqueue(bv, xv.fill(0.0), 1e-9, 200).result() + (xv.download(),)
        assert_same_solve(got, want, "after refresh")
    fresh.free()
    amg.free()


def test_result_waits_for_the_stream_the_solve_was_enqueued_on(sp):
    import torch

    dH, levels, amg = hierarchy(sp, "hem")
    rng = np.random.default_rng(17)
    b = rng.standard_normal(dH.n)
    want = sync_solve(sp, dH, "pcg", b, np.zeros(dH.n), 1e-9, 200)
    bv, xv = sp.DeviceVector(data=b), sp.DeviceVector(dH.n).fill(0.0)
    dH.pcg_enqueue(bv, xv, 1e-9, 200).result()  # warm: the solve graph exists
    side = torch.cuda.Stream()
    for _ in range(2):
        xv.fill(0.0)
        sp.sync()
        sp.set_stream(side.cuda_stream)
        pend = dH.pcg_enqueue(bv, xv, 1e-9, 200)
        sp.set_stream(None)  # the library's own stream is current again
        got = pend.result()  # waits for `side`, not for the current stream
        assert_same_solve(got + (xv.download(),), want, "enqueued on a side stream")
    amg.free()


def capture_pcg(sp, dH, b, x, tol, max_iter, pend):
    import torch

    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        sp.set_stream(torch.cuda.current_stream().cuda_stream)
        try:
            dH.pcg_enqueue(b, x, tol, max_iter, pending=pend)
        finally:
            sp.set_stream(None)
    return g


@pytest.mark.parametrize("grid", [32, 25])  # coarsest level 2048 rows (even) and 3907 rows (odd)
def test_a_solve_captured_again_after_a_refresh_equals_a_fresh_hierarchy(sp, grid):
    """The header's contract: a caller's graph holding an enqueued solve is captured again after a refresh (and the
    method is run once outside the capture first).  The coarse inverse keeps its address through refreshes (an odd
    coarsest size ends the elimination in the spare buffer), so a captured coarse solve keeps reading the current one."""
    import torch

    dH, levels, amg = hierarchy(sp, "hem", grid)
    assert levels[-1]["A"].nrow % 2 == (grid % 2)
    n, tol, max_iter = dH.n, 1e-9, 200
    b = torch.from_numpy(np.random.default_rng(18).standard_normal(n)).cuda()
    x = torch.zeros_like(b)
    nc = levels[-1]["A"].nrow
    bc = torch.from_numpy(np.random.default_rng(19).standard_normal(nc)).cuda()
    xc = torch.zeros_like(bc)
    pend = sp.PendingSolve(max_iter)
    torch.cuda.synchronize()  # torch's stream wrote the tensors; the library's own stream reads them
    dH.pcg_enqueue(b, x, tol, max_iter, pending=pend).result()
    gc = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gc):
        sp.set_stream(torch.cuda.current_stream().cuda_stream)
        try:
            sp.capi.check(dH.lib.sparsh_hierarchy_coarse_solve(dH.h, bc.data_ptr(), xc.data_ptr()))
        finally:
            sp.set_stream(None)
    for sigma in (2.0, 0.5, 1.0):  # three refreshes: the buffer roles alternate with an odd coarsest size
        A0 = shifted(levels[0]["A"], sigma)
        dH.refresh(A0.val)
        fresh = sp.DeviceHierarchy(galerkin_levels(sp, A0, levels))
        with pytest.raises(sp.SparshError, match="error 2"):  # the refresh asks for a warm call again
            capture_pcg(sp, dH, b, x, tol, max_iter, pend)
        x.zero_()
        torch.cuda.synchronize()
        dH.pcg_enqueue(b, x, tol, max_iter, pending=pend).result()  # the warm call
        g = capture_pcg(sp, dH, b, x, tol, max_iter, pend)
        x.zero_()
        g.replay()
        torch.cuda.synchronize()
        want = sync_solve(sp, fresh, "pcg", b.cpu().numpy(), np.zeros(n), tol, max_iter)
        assert_same_solve(pend.result() + (x.cpu().numpy(),), want, f"grid {grid} sigma {sigma}")
        gc.replay()
        torch.cuda.synchronize()
        same_bits(xc.cpu().numpy(), fresh.coarse_solve(sp.DeviceVector(data=bc.cpu().numpy())).download(),
                  f"grid {grid} sigma {sigma} captured coarse solve")
        del g
        fresh.free()
    del gc
    amg.free()


def test_a_stale_hierarchy_is_refused(sp):
    dH, levels, amg = hierarchy(sp, "hem")
    b = sp.DeviceVector(data=np.random.default_rng(15).standard_normal(dH.n))
    x = sp.DeviceVector(dH.n).fill(0.0)
    dH.pcg_enqueue(b, x, 1e-9, 100).result()
    with pytest.raises(sp.SparshError, match="error 2"):
        dH.refresh(np.zeros(levels[0]["A"].nnz))
    for fn in (dH.pcg_enqueue, dH.pbicgstab_enqueue, dH.amg_solve_enqueue):
        with pytest.raises(sp.SparshError, match="error 2"):
            fn(b, x, 1e-9, 100)
    amg.free()


def test_capture_into_a_torch_graph_replays_the_synchronous_bits(sp):
    import torch

    dH, levels, amg = hierarchy(sp, "hem")
    n, tol, max_iter = dH.n, 1e-9, 200
    dev = torch.device("cuda", 0)
    src = torch.zeros(n, dtype=torch.float64, device=dev)  # the graph's static input
    b = torch.zeros_like(src)
    x = torch.zeros_like(src)
    y = torch.zeros_like(src)
    pend = sp.PendingSolve(max_iter)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):  # the warm call, outside the capture
        sp.set_stream(side.cuda_stream)
        try:
            dH.pcg_enqueue(b, x, tol, max_iter, pending=pend).result()
        finally:
            sp.set_stream(None)
    torch.cuda.synchronize()

    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        torch.mul(src, 2.0, out=b)  # a torch op builds b
        x.zero_()
        sp.set_stream(torch.cuda.current_stream().cuda_stream)
        try:
            dH.pcg_enqueue(b, x, tol, max_iter, pending=pend)
        finally:
            sp.set_stream(None)
        torch.mul(x, 2.0, out=y)  # a torch op on the solution
    rng = np.random.default_rng(16)
    for k in range(2):
        bk = rng.standard_normal(n)
        src.copy_(torch.from_numpy(bk / 2.0).to(dev))
        g.replay()
        torch.cuda.synchronize()
        want = sync_solve(sp, dH, "pcg", bk, np.zeros(n), tol, max_iter)
        got = pend.result() + (x.cpu().numpy(),)
        assert want[2] and want[0] > 2
        assert_same_solve(got, want, f"replay {k}")
        same_bits(y.cpu().numpy(), 2.0 * want[3], f"replay {k} torch op after the solve")
    del g
    amg.free()


def test_capture_before_a_warm_call_is_refused(sp):
    import torch

    dH, levels, amg = hierarchy(sp, "hem")
    n = dH.n
    b = torch.ones(n, dtype=torch.float64, device="cuda")
    x = torch.zeros_like(b)
    pend = sp.PendingSolve(100)
    g = torch.cuda.CUDAGraph()
    with pytest.raises(sp.SparshError, match="error 2.*run it once before capturing"):
        with torch.cuda.graph(g):
            sp.set_stream(torch.cuda.current_stream().cuda_stream)
            try:
                dH.pcg_enqueue(b, x, 1e-9, 100, pending=pend)
            finally:
                sp.set_stream(None)
    del g
    torch.cuda.synchronize()
    # nothing was done behind the caller's back: the hierarchy works, and the first call outside capture is right
    bn = np.ones(n)
    xv = sp.DeviceVector(n).fill(0.0)
    got = dH.pcg_enqueue(sp.DeviceVector(data=bn), xv, 1e-9, 100, pending=pend).result()
    assert_same_solve(got + (xv.download(),), sync_solve(sp, dH, "pcg", bn, np.zeros(n), 1e-9, 100), "after refusal")
    amg.free()

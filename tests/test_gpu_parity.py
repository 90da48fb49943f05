"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C-ABI, against the CPU oracle on the
same seeded inputs and against the golden vectors produced by the reference itself.

Tolerances (north_star): per-kernel fp64 results within 1e-12 relative — the thread-per-row kernel families (stream,
scalar) accumulate in the reference's order and must in fact be BIT-IDENTICAL; V-cycle / PCG residual histories within
1e-10 relative with the same iteration count (+-1); integer data bit-exact.
"""
import os

import numpy as np
import pytest
from conftest import system_by_name
from oracle_bindings import CSR, OracleAmg

pytestmark = pytest.mark.gpu

OMEGA = 0.66667
KINDS = [("scalar", 0, 256), ("stream", 1, 256), ("stream", 1, 128), ("vector", 2, 2), ("vector", 2, 8),
         ("vector", 2, 32)]


@pytest.fixture(scope="module")
def sp():
    import sparsh_amg_b200 as s

    s.init(0)  # raises (no fallback) if the extension or the GPU is missing
    return s


@pytest.fixture(scope="module")
def fixture_hierarchies(oracle, fixture_system):
    A, b = fixture_system
    return {c: OracleAmg(A, coarsening=i) for i, c in enumerate(["hem", "beck"])}


def rel_close(got, want, rtol):
    np.testing.assert_allclose(got, want, rtol=rtol, atol=rtol * max(1e-300, float(np.max(np.abs(want)))))


def assert_hist(got, want, rtol=1e-10, r0=None):
    """north_star: histories within 1e-10 relative, same iteration count (+-1).  A residual norm that has dropped by
    eight orders is itself only evaluable to ~1e-16*||A||*||x|| in fp64 (different summation trees in the norm and the
    coarse solve), so entries are compared to rtol OR to 1e-13 of the initial residual, whichever is larger."""
    got, want = np.asarray(got), np.asarray(want)
    assert abs(len(got) - len(want)) <= 1, (len(got), len(want))
    m = min(len(got), len(want))
    floor = 1e-13 * (float(r0) if r0 is not None else float(max(want[0], got[0])))
    np.testing.assert_allclose(got[:m], want[:m], rtol=rtol, atol=floor)


# ---------------------------------------------------------------------------------------------------- per-op
@pytest.mark.parametrize("coarsening", ["hem", "beck"])
@pytest.mark.parametrize("kname,kind,tl", KINDS)
def test_level_ops_match_oracle(sp, oracle, fixture_hierarchies, coarsening, kname, kind, tl):
    """K1-K5, K9 on every level of the fixture hierarchy, every kernel family."""
    H = fixture_hierarchies[coarsening].hierarchy()
    rng = np.random.default_rng(5)
    exact = kname in ("scalar", "stream")
    for L in H.levels:
        A, diag = L["A"], L["diag"]
        dA = sp.DeviceMatrix.from_csr(A, diag=diag).force_kernel(kind, tl)
        x, b = rng.standard_normal(A.nrow), rng.standard_normal(A.nrow)
        dx, db = sp.DeviceVector(data=x), sp.DeviceVector(data=b)
        checks = [
            (dA.spmv(dx).download(), oracle.spmv(A, x)),
            (dA.residual(db, dx).download(), oracle.store_residual(A, b, x)),
            (dA.jacobi(db, sp.DeviceVector(data=x), OMEGA, 7).download(), oracle.jacobi(A, diag, b, x, OMEGA, 6)),
            (dA.jacobi(db, sp.DeviceVector(data=x), OMEGA, 2).download(), oracle.jacobi(A, diag, b, x, OMEGA, 1)),
        ]
        y, pdot = dA.spmv_dot(dx)
        checks.append((y.download(), oracle.spmv(A, x)))
        for got, want in checks:
            if exact:
                np.testing.assert_array_equal(got, want)
            else:
                rel_close(got, want, 1e-12)
        np.testing.assert_allclose(pdot, np.dot(x, oracle.spmv(A, x)), rtol=1e-12)
        np.testing.assert_allclose(dA.residual_norm(db, dx), oracle.residual(A, b, x), rtol=1e-12)
        if L["P"] is not None:
            P = L["P"]
            xc = rng.standard_normal(P.ncol)
            dP = sp.DeviceMatrix.from_csr(P).force_kernel(kind, tl)
            dR = sp.DeviceMatrix.from_csr(P, transpose=True).force_kernel(kind, tl)
            got_r = dR.restrict(dx).download()
            got_p = dP.prolong_add(sp.DeviceVector(data=xc), sp.DeviceVector(data=x)).download()
            if exact:
                np.testing.assert_array_equal(got_r, oracle.transfer_residual(P, x))
                np.testing.assert_array_equal(got_p, oracle.transfer_solution(P, xc, x))
            else:
                rel_close(got_r, oracle.transfer_residual(P, x), 1e-12)
                rel_close(got_p, oracle.transfer_solution(P, xc, x), 1e-12)


def test_default_kernel_selection(sp, oracle, monkeypatch):
    A = oracle.gen_poisson3d(20, 20, 20)
    dA = sp.DeviceMatrix.from_csr(A)
    assert dA.kernel()[0] == sp.capi.KIND_PATTERN  # rows repeat (27 patterns): csr-pattern8, lean kernel
    assert dA.kernel_name("jacobi") == "csr_pat2_kernel<256,1,7,EPI_JACOBI>"
    assert dA.kernel_name("spmv") == "csr_pat2_kernel<128,2,7,EPI_SPMV>"
    monkeypatch.setenv("SPARSH_PATTERN", "0")
    assert sp.DeviceMatrix.from_csr(A).kernel()[0] == sp.capi.KIND_DICT  # 2 distinct values, 7 distinct offsets
    monkeypatch.delenv("SPARSH_PATTERN")
    nc, agg = oracle.hem(A, 0)
    P = CSR(A.nrow, nc, np.arange(A.nrow + 1, dtype=np.int32), agg, np.ones(A.nrow))
    assert sp.DeviceMatrix.from_csr(P).kernel()[0] == sp.capi.KIND_SCALAR
    assert sp.DeviceMatrix.from_csr(P, transpose=True).kernel()[0] == sp.capi.KIND_SCALAR
    # one dense row among short ones -> irregular -> vector family
    n = 600
    rp = np.concatenate([[0], np.cumsum([n] + [1] * (n - 1))]).astype(np.int32)
    ci = np.concatenate([np.arange(n), np.arange(1, n)]).astype(np.int32)
    M = CSR(n, n, rp, ci, np.ones(len(ci)))
    dM = sp.DeviceMatrix.from_csr(M)
    assert dM.kernel()[0] == sp.capi.KIND_VECTOR
    x = np.random.default_rng(1).standard_normal(n)
    rel_close(dM.spmv(sp.DeviceVector(data=x)).download(), oracle.spmv(M, x), 1e-12)


def test_fixture_matrix_keeps_plain_csr(sp, fixture_system):
    """the bundled FE matrix has ~80k distinct values: no csr-dict16 twin, plain TMA-staged stream kernel"""
    A, _ = fixture_system
    dA = sp.DeviceMatrix.from_csr(A)
    assert dA.kernel()[0] == sp.capi.KIND_STREAM
    with pytest.raises(sp.SparshError):
        dA.force_kernel(sp.capi.KIND_DICT, 256)


def _host_pattern_encode(sp, M, diag):
    """the host statement of the csr-pattern8 encoder (sparsh_pattern_encode) -> (n_pat, n_ent, n_escape)"""
    import ctypes as C

    lib = sp.capi.load()
    pat = np.zeros(M.nrow + 16, dtype=np.uint8)
    ev, eo, st = np.zeros(2048), np.zeros(2048, dtype=np.int32), np.zeros(257, dtype=np.int32)
    npat, nesc = C.c_int(), C.c_int()
    dptr = sp.capi.dp(np.ascontiguousarray(diag, dtype=np.float64)) if diag is not None else None
    sp.capi.check(lib.sparsh_pattern_encode(M.nrow, M.ncol, M.nnz, sp.capi.ip(M.rowptr), sp.capi.ip(M.colindex), sp.capi.dp(M.val),
                                            dptr, pat.ctypes.data_as(C.c_void_p), sp.capi.dp(ev), sp.capi.ip(eo), sp.capi.ip(st),
                                            C.byref(npat), C.byref(nesc)))
    return npat.value, int(st[npat.value]), nesc.value, float(np.mean(pat[: M.nrow] == 0))


def test_device_pattern_encoder_matches_the_host_encoder(sp, oracle, fixture_system):
    """the upload encodes csr-pattern8 on the DEVICE (hash table + entry-by-entry verification); its table and its escape
    rows must be the host encoder's: Poisson hierarchy levels, a level whose smoothing diagonal differs on a few rows
    (those rows become escapes), and a matrix whose rows do not repeat (the bundled FE system: no twin)"""
    A = oracle.gen_poisson3d(24, 20, 18)
    H = OracleAmg(A, coarsening=0, limit_upper=300, limit_lower=150).hierarchy()
    cases = [(L["A"], L["diag"]) for L in H.levels]
    d2 = H.levels[0]["diag"].copy()
    d2[[3, 77, 4001]] *= 1.0 + 1e-9
    cases.append((A, d2))
    checked = 0
    for M, diag in cases:
        dA = sp.DeviceMatrix.from_csr(M, diag=diag)
        npat, nent, nesc, cover0 = dA.pattern_stats()
        want = _host_pattern_encode(sp, M, diag)
        if dA.kernel()[0] == sp.capi.KIND_PATTERN:
            assert (npat, nent, nesc) == want[:3] and abs(cover0 - want[3]) < 1e-12
            checked += 1
    assert checked >= 3
    F, _ = fixture_system
    assert sp.DeviceMatrix.from_csr(F).pattern_stats()[0] == 0 and sp.DeviceMatrix.from_csr(F).kernel()[0] == sp.capi.KIND_STREAM


@pytest.mark.parametrize("coarsening", [0, 1])
@pytest.mark.parametrize("threads", [128, 256])
def test_dict_format_is_bit_identical(sp, oracle, coarsening, threads, monkeypatch):
    """csr-dict16 (2 B/nnz) against the oracle AND against the plain stream kernel on every level of a Poisson
    hierarchy: lossless re-encoding, same summation order -> identical bits."""
    monkeypatch.setenv("SPARSH_DICT", "2")  # build the csr-dict16 twin even where csr-pattern8 is selected
    A = oracle.gen_poisson3d(24, 20, 18)
    H = OracleAmg(A, coarsening=coarsening, limit_upper=300, limit_lower=150).hierarchy()
    rng = np.random.default_rng(17)
    used = 0
    for L in H.levels:
        M, diag = L["A"], L["diag"]
        dA = sp.DeviceMatrix.from_csr(M, diag=diag)
        try:
            dA.force_kernel(sp.capi.KIND_DICT, threads)
        except sp.SparshError:
            continue  # no csr-dict16 twin on this level
        used += 1
        x, b = rng.standard_normal(M.nrow), rng.standard_normal(M.nrow)
        dx, db = sp.DeviceVector(data=x), sp.DeviceVector(data=b)
        res = {}
        for kind, tl in [(sp.capi.KIND_DICT, threads), (sp.capi.KIND_STREAM, threads)]:
            dA.force_kernel(kind, tl)
            y, pdot = dA.spmv_dot(dx)
            res[kind] = (dA.spmv(dx).download(), dA.residual(db, dx).download(),
                         dA.jacobi(db, sp.DeviceVector(data=x), OMEGA, 7).download(), y.download(), pdot,
                         dA.residual_norm(db, dx))
        want = (oracle.spmv(M, x), oracle.store_residual(M, b, x), oracle.jacobi(M, diag, b, x, OMEGA, 6),
                oracle.spmv(M, x))
        for got_d, got_s, w in zip(res[sp.capi.KIND_DICT][:4], res[sp.capi.KIND_STREAM][:4], want):
            np.testing.assert_array_equal(got_d, w)
            np.testing.assert_array_equal(got_d, got_s)
        # fused reductions: identical contributions, different (but fixed) summation trees in the two kernels
        np.testing.assert_allclose(res[sp.capi.KIND_DICT][4], res[sp.capi.KIND_STREAM][4], rtol=1e-12)
        np.testing.assert_allclose(res[sp.capi.KIND_DICT][5], res[sp.capi.KIND_STREAM][5], rtol=1e-12)
    assert used >= 2


@pytest.mark.parametrize("coarsening", [0, 1])
@pytest.mark.parametrize("threads", [128, 256])
def test_pattern_format_is_bit_identical(sp, oracle, coarsening, threads, monkeypatch):
    """csr-pattern8 (1 B/row) against the oracle AND against the plain stream kernel on every level of a Poisson
    hierarchy, plus a matrix with escape rows: same entries, same summation order -> identical bits."""
    monkeypatch.setenv("SPARSH_PATTERN", "2")  # build the twin, keep the default kernel; the test forces kinds
    A = oracle.gen_poisson3d(24, 20, 18)
    H = OracleAmg(A, coarsening=coarsening, limit_upper=300, limit_lower=150).hierarchy()
    rng = np.random.default_rng(23)
    mats = [(L["A"], L["diag"]) for L in H.levels]
    # perturb a handful of entries of level 0: those rows stop repeating and must take the escape path
    P0 = CSR(A.nrow, A.ncol, A.rowptr.copy(), A.colindex.copy(), A.val.copy())
    for r in (0, 17, 513, 4000, A.nrow - 1):
        P0.val[P0.rowptr[r]] *= 1.0 + 1e-3 * rng.standard_normal()
    d0 = np.array([P0.val[P0.rowptr[i]:P0.rowptr[i + 1]][P0.colindex[P0.rowptr[i]:P0.rowptr[i + 1]] == i][0]
                   for i in range(P0.nrow)])
    mats.append((P0, d0))
    used = 0
    for M, diag in mats:
        dA = sp.DeviceMatrix.from_csr(M, diag=diag)
        try:
            dA.force_kernel(sp.capi.KIND_PATTERN, threads)
        except sp.SparshError:
            continue  # rows do not repeat on this level
        used += 1
        x, b = rng.standard_normal(M.nrow), rng.standard_normal(M.nrow)
        dx, db = sp.DeviceVector(data=x), sp.DeviceVector(data=b)
        res = {}
        for kind, tl in [(sp.capi.KIND_PATTERN, threads), (sp.capi.KIND_STREAM, threads)]:
            dA.force_kernel(kind, tl)
            y, pdot = dA.spmv_dot(dx)
            res[kind] = (dA.spmv(dx).download(), dA.residual(db, dx).download(),
                         dA.jacobi(db, sp.DeviceVector(data=x), OMEGA, 7).download(), y.download(), pdot,
                         dA.residual_norm(db, dx))
        want = (oracle.spmv(M, x), oracle.store_residual(M, b, x), oracle.jacobi(M, diag, b, x, OMEGA, 6),
                oracle.spmv(M, x))
        for got_p, got_s, w in zip(res[sp.capi.KIND_PATTERN][:4], res[sp.capi.KIND_STREAM][:4], want):
            np.testing.assert_array_equal(got_p, w)
            np.testing.assert_array_equal(got_p, got_s)
        np.testing.assert_allclose(res[sp.capi.KIND_PATTERN][4], res[sp.capi.KIND_STREAM][4], rtol=1e-12)
        np.testing.assert_allclose(res[sp.capi.KIND_PATTERN][5], res[sp.capi.KIND_STREAM][5], rtol=1e-12)
    assert used >= 3


def test_pattern_format_solver_history(sp, oracle, monkeypatch):
    """whole AMG-PCG solve with the pattern kernel on every level that has the twin: same history as the oracle"""
    monkeypatch.setenv("SPARSH_PATTERN", "1")
    A = oracle.gen_poisson3d(32, 32, 32)
    amg = OracleAmg(A, limit_upper=500, limit_lower=250)
    dH = sp.DeviceHierarchy(amg.hierarchy().levels)
    assert dH.level(0)[0].kernel()[0] == sp.capi.KIND_PATTERN
    b = np.ones(A.nrow)
    _, hist_ref = amg.pcg(b, np.zeros(A.nrow), 1e-8)
    db, dx = sp.DeviceVector(data=b), sp.DeviceVector(A.nrow).fill(0.0)
    it, hist, ok = dH.pcg(db, dx, 1e-8)
    assert ok and it == len(hist_ref) - 1
    assert_hist(hist, hist_ref)
    monkeypatch.setenv("SPARSH_PATTERN", "0")
    dH0 = sp.DeviceHierarchy(amg.hierarchy().levels)
    assert dH0.level(0)[0].kernel()[0] == sp.capi.KIND_DICT
    dx0 = sp.DeviceVector(A.nrow).fill(0.0)
    it0, hist0, _ = dH0.pcg(db, dx0, 1e-8)
    # row sums are bit-identical; the fused dot products see another (fixed) tree because the kernels tile differently
    assert it0 == it
    np.testing.assert_allclose(hist, hist0, rtol=1e-10, atol=1e-13 * hist0[0])
    np.testing.assert_allclose(dx.download(), dx0.download(), rtol=1e-9, atol=1e-12 * np.abs(dx0.download()).max())
    # ... and the smoother alone (no reduction involved) leaves the same bits behind as the default kernels
    A0p, A0d = dH.level(0)[0], dH0.level(0)[0]
    xr = sp.DeviceVector(data=np.random.default_rng(3).standard_normal(A.nrow))
    np.testing.assert_array_equal(A0p.jacobi(db, sp.DeviceVector(data=xr.download()), OMEGA, 7).download(),
                                  A0d.jacobi(db, sp.DeviceVector(data=xr.download()), OMEGA, 7).download())


def test_smoothed_aggregation_hierarchy_on_gpu(sp, oracle):
    """SURVEY §8f.2: a smoothed-aggregation hierarchy (general P, 30-60 nnz/row coarse operators) through the same
    device path: V-cycle and AMG-PCG histories against the oracle running the same hierarchy."""
    from sparsh_amg_b200 import host

    host.set_options(coarsening=2, coarse_upper=500, coarse_lower=250, max_levels=32, print_setup=0)
    try:
        M = host.HostMatrix.poisson3d(32, 32, 32)
        amg = host.HostAmg(M)
        levels = []
        for L in amg.levels():
            A, P = L["A"], L["P"]
            levels.append(dict(A=CSR(A.nrow, A.ncol, A.rowptr.copy(), A.colindex.copy(), A.val.copy()),
                               diag=np.array(L["diag"]),
                               P=None if P is None else CSR(P.nrow, P.ncol, P.rowptr.copy(), P.colindex.copy(), P.val.copy())))
    finally:
        host.set_options(coarsening=0, coarse_upper=4000, coarse_lower=2000, max_levels=6, print_setup=1)
    from oracle_bindings import Hierarchy

    oa = OracleAmg(hierarchy=Hierarchy(levels))
    dH = sp.DeviceHierarchy(levels)
    n = levels[0]["A"].nrow
    b = np.ones(n)
    rng = np.random.default_rng(5)
    xr = rng.standard_normal(n)
    db = sp.DeviceVector(data=b)
    rel_close(dH.vcycle(db, sp.DeviceVector(data=xr), 1).download(), oa.vcycle(b, xr, 1), 1e-10)
    _, hist_ref = oa.pcg(b, np.zeros(n), 1e-8 * np.sqrt(n))
    it, hist, ok = dH.pcg(db, sp.DeviceVector(n).fill(0.0), 1e-8 * np.sqrt(n))
    assert ok and abs(it - (len(hist_ref) - 1)) <= 1
    m = min(len(hist), len(hist_ref))
    assert_hist(hist[:m], hist_ref[:m])


def test_gmres_matches_the_oracle_statement(sp, oracle, fixture_system):
    """SURVEY §8f.2: restarted GMRES (CGS2 + Givens) on the device against the oracle's statement of the same algorithm:
    plain on a nonsymmetric matrix (full and restarted), V-cycle-preconditioned on the bundled system."""
    import scipy.sparse as sps

    rng = np.random.default_rng(11)
    n = 3000
    S = (sps.diags([-1.3, 2.6, -0.7], [-1, 0, 1], shape=(n, n)) + sps.random(n, n, density=0.001, random_state=3) * 0.2).tocsr()
    S.sort_indices()
    A = CSR(n, n, S.indptr, S.indices, S.data)
    b = rng.standard_normal(n)
    tol = 1e-9 * np.linalg.norm(b)
    dA = sp.DeviceMatrix.from_csr(A)
    db = sp.DeviceVector(data=b)
    for restart in (200, 10):
        x_ref, h_ref = oracle.gmres(A, b, np.zeros(n), tol, restart=restart, max_iter=2000)
        dx = sp.DeviceVector(n).fill(0.0)
        it, hist, ok = dA.gmres(db, dx, tol, restart=restart, max_iter=2000)
        assert ok and abs(it - (len(h_ref) - 1)) <= 1
        m = min(len(hist), len(h_ref))
        np.testing.assert_allclose(hist[:m], h_ref[:m], rtol=1e-7, atol=1e-13 * h_ref[0])
        assert np.linalg.norm(b - S @ dx.download()) <= tol * (1 + 1e-6)
    F, fb = fixture_system
    amg = OracleAmg(F)
    _, hp_ref = amg.pgmres(fb, np.zeros(F.nrow), 1e-8, restart=30)
    dH = sp.DeviceHierarchy(amg.hierarchy().levels)
    dfx = sp.DeviceVector(F.nrow).fill(0.0)
    it, hist, ok = dH.pgmres(sp.DeviceVector(data=fb), dfx, 1e-8, restart=30)
    assert ok and abs(it - (len(hp_ref) - 1)) <= 1
    m = min(len(hist), len(hp_ref))
    np.testing.assert_allclose(hist[:m], hp_ref[:m], rtol=1e-7, atol=1e-13 * hp_ref[0])
    assert np.linalg.norm(fb - F.to_scipy() @ dfx.download()) <= 1e-8 * (1 + 1e-6)


def test_device_galerkin_product(sp, oracle, fixture_system):
    """SURVEY 8f.1: A_c = P^T (A P) on the device (csrc/rap.cu) against the oracle's restatement of
    parallel::coarsen_matrix (src/AMG_cycle_utilities.cpp:126-146) — row pointers and sorted column indices bit-exact,
    values to 1e-13 — and against this repository's host product, whose bits it must reproduce (same traversal order,
    unfused arithmetic): aggregation P (HEM), classical P (Beck) on 3D Poisson and on the bundled FE system, and a whole
    hierarchy built with options().gpu_rap = 1."""
    from sparsh_amg_b200 import host

    F, _ = fixture_system
    cases = []
    for A in (oracle.gen_poisson3d(20, 18, 16), F):
        nc, agg = oracle.hem(A, 0)
        cases.append((A, CSR(A.nrow, nc, np.arange(A.nrow + 1, dtype=np.int32), agg, np.ones(A.nrow))))
        cases.append((A, oracle.beck(A)))
    for A, P in cases:
        got = sp.galerkin_rap(A, P)
        assert got is not None
        want = oracle.rap(A, P)
        np.testing.assert_array_equal(got[0], want.rowptr)
        np.testing.assert_array_equal(got[1], want.colindex)
        np.testing.assert_allclose(got[2], want.val, rtol=1e-13, atol=1e-13 * np.abs(want.val).max())
    # a whole hierarchy, host product against device product: identical bits on every level
    # (the products chain on the device: level l's product is level l+1's fine matrix, sparsh_galerkin_rap_next; the large
    # grid moves its arrays through the pinned staging buffers on several host threads)
    host.set_options(threads=4, max_levels=32, print_setup=0, coarse_upper=300, coarse_lower=100)
    try:
        for coarsening, grid in ((0, (24, 20, 18)), (1, (24, 20, 18)), (2, (24, 20, 18)), (0, (112, 96, 80))):
            host.set_options(coarsening=coarsening, gpu_rap=0)
            M = host.HostMatrix.poisson3d(*grid)
            h0 = host.HostAmg(M)
            host.set_options(gpu_rap=1)
            h1 = host.HostAmg(M)
            assert h0.nlevels == h1.nlevels and h0.nlevels >= 3
            for L0, L1 in zip(h0.levels(), h1.levels()):
                for key in ("rowptr", "colindex", "val"):
                    np.testing.assert_array_equal(getattr(L0["A"], key), getattr(L1["A"], key))
                np.testing.assert_array_equal(L0["diag"], L1["diag"])
            h0.free()
            h1.free()
            M.free()
    finally:
        host.set_options(coarsening=0, gpu_rap=0, coarse_upper=4000, coarse_lower=2000, max_levels=6, print_setup=1)


def test_edge_cases(sp, oracle):
    # 1x1
    A = CSR(1, 1, [0, 1], [0], [2.0])
    assert sp.DeviceMatrix.from_csr(A).spmv(sp.DeviceVector(data=[3.0])).download()[0] == 6.0
    # ragged with empty rows, all families
    rng = np.random.default_rng(2)
    n = 1000
    lens = rng.integers(0, 9, n)
    lens[::7] = 0
    rp = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    ci = np.concatenate([np.sort(rng.choice(n, l, replace=False)) for l in lens] + [np.zeros(0, int)]).astype(np.int32)
    M = CSR(n, n, rp, ci, rng.standard_normal(len(ci)))
    x = rng.standard_normal(n)
    want = oracle.spmv(M, x)
    for kname, kind, tl in KINDS:
        got = sp.DeviceMatrix.from_csr(M).force_kernel(kind, tl).spmv(sp.DeviceVector(data=x)).download()
        if kname == "vector":
            rel_close(got, want, 1e-12)
        else:
            np.testing.assert_array_equal(got, want)
    # row counts that are not multiples of the CTA tile
    for nx in (1, 5, 129, 257):
        A = oracle.gen_poisson2d(nx, 3)
        x = rng.standard_normal(A.nrow)
        np.testing.assert_array_equal(sp.DeviceMatrix.from_csr(A).spmv(sp.DeviceVector(data=x)).download(),
                                      oracle.spmv(A, x))
    # invalid input is an error, not a crash
    with pytest.raises(sp.SparshError):
        sp.DeviceMatrix(2, 2, [0, 1, 2], [0, 5], [1.0, 1.0])


def test_blas1(sp):
    rng = np.random.default_rng(3)
    for n in (1, 31, 1000, 1 << 20, (1 << 20) + 3):
        x, y, z = rng.standard_normal(n), rng.standard_normal(n), rng.standard_normal(n)
        dx, dy, dz = sp.DeviceVector(data=x), sp.DeviceVector(data=y), sp.DeviceVector(data=z)
        np.testing.assert_allclose(sp.dot(dx, dy), np.dot(x, y), rtol=1e-12, atol=1e-12 * np.sqrt(n))
        np.testing.assert_allclose(sp.nrm2(dx), np.linalg.norm(x), rtol=1e-13)
        assert sp.dot(dx, dy) == sp.dot(dx, dy)  # fixed reduction tree: bit-reproducible
        sp.axpy(0.37, dx, dy)
        y = y + 0.37 * x
        np.testing.assert_array_equal(dy.download(), y)
        sp.axpby(1.5, dx, -0.25, dy)
        y = 1.5 * x + (-0.25) * y
        np.testing.assert_array_equal(dy.download(), y)
        sp.axpbypcz(0.1, dx, 0.2, dy, 0.3, dz)
        z = (0.1 * x + 0.2 * y) + 0.3 * z
        np.testing.assert_array_equal(dz.download(), z)
        np.testing.assert_array_equal(sp.DeviceVector(n).fill(2.5).download(), np.full(n, 2.5))


def test_multicolour_sor(sp, oracle, fixture_system, golden):
    """K6: colour-permuted system from the reference's colouring (integers bit-exact, checked in the CPU suite)."""
    A, b = fixture_system
    nc, perm, cc, Q = oracle.color_reorder(A)
    qd = Q.diagonal()
    dQ = sp.DeviceMatrix.from_csr(Q, diag=qd)
    bp = b[perm]
    want = oracle.sor_multicolor(Q, qd, cc, bp, np.zeros(A.nrow), OMEGA, 3)
    got = dQ.mc_sor(cc, sp.DeviceVector(data=bp), sp.DeviceVector(data=np.zeros(A.nrow)), OMEGA, 3).download()
    np.testing.assert_array_equal(got, want)
    np.testing.assert_allclose(got[:8], golden["fixture"]["sor_probe"]["x_head"], rtol=1e-12)
    # judged by iteration count (north_star): sweeps needed to cut ||Ax-b|| tenfold must match the oracle's
    r_start = oracle.residual(Q, bp, np.zeros(A.nrow))

    def sweeps_to(step):
        x = np.zeros(A.nrow)
        for k in range(1, 2000):
            x = step(x)
            if oracle.residual(Q, bp, x) <= 0.1 * r_start:
                return k
        return -1

    dx, db = sp.DeviceVector(A.nrow), sp.DeviceVector(data=bp)

    def gpu_step(x):
        dx.upload(x)
        return dQ.mc_sor(cc, db, dx, OMEGA, 1).download()

    k_gpu = sweeps_to(gpu_step)
    k_cpu = sweeps_to(lambda x: oracle.sor_multicolor(Q, qd, cc, bp, x, OMEGA, 1))
    assert k_gpu == k_cpu and k_gpu > 0


# ------------------------------------------------------------------------------------------------ hierarchy
@pytest.mark.parametrize("coarsening", ["hem", "beck"])
def test_coarse_solve(sp, oracle, fixture_hierarchies, coarsening):
    amg = fixture_hierarchies[coarsening]
    H = amg.hierarchy()
    dH = sp.DeviceHierarchy(H.levels)
    n = H.levels[-1]["A"].nrow
    b = np.random.default_rng(9).standard_normal(n)
    got = dH.coarse_solve(sp.DeviceVector(data=b)).download()
    want = amg.coarse_solve(b)
    rel_close(got, want, 1e-10)
    # and it really solves the system
    r = b - H.levels[-1]["A"].to_scipy() @ got
    assert np.linalg.norm(r) <= 1e-11 * np.linalg.norm(b) * 1e3


CASES = ["fixture", "poisson3d_24_ones", "poisson3d_24_axstar", "poisson2d_96_ones", "poisson2d_96_axstar"]


@pytest.mark.parametrize("case", CASES + ["poisson3d_40_ones"])
@pytest.mark.parametrize("coarsening", ["hem", "beck"])
def test_vcycle_amg_pcg_against_reference_goldens(sp, oracle, fixture_system, golden, case, coarsening):
    A, b = system_by_name(case, oracle, fixture_system)
    g = golden[case][coarsening]
    amg = OracleAmg(A, coarsening=0 if coarsening == "hem" else 1)
    dH = sp.DeviceHierarchy(amg.hierarchy().levels)
    db = sp.DeviceVector(data=b)
    # one V-cycle from a seeded random start (AMG_solve_jacobi(b,x,1))
    xr = np.random.default_rng(g["vcycle_probe"]["seed"]).random(A.nrow)
    x1 = dH.vcycle(db, sp.DeviceVector(data=xr), 1).download()
    np.testing.assert_allclose(x1[:8], g["vcycle_probe"]["x_head"], rtol=1e-10)
    np.testing.assert_allclose(np.linalg.norm(x1), g["vcycle_probe"]["x_norm"], rtol=1e-10)
    rel_close(x1, amg.vcycle(b, xr, 1), 1e-10)
    # AMG as solver, absolute 1e-8 as the reference (AMG_Solver_CPU_baseline / AMG_Solver_CPU_GPU_MI)
    dx = sp.DeviceVector(A.nrow).fill(0.0)
    it, hist, ok = dH.amg_solve(db, dx, 1e-8)
    assert ok
    assert_hist(hist[1:], g["amg_solve_hist"], r0=hist[0])
    np.testing.assert_allclose(hist[0], golden[case]["b_norm"], rtol=1e-12)
    # AMG-PCG (Solver_PCG_1 semantics behind Solver_PCG_4)
    dx.fill(0.0)
    it, hist, ok = dH.pcg(db, dx, 1e-8)
    assert ok
    assert_hist(hist, g["pcg_hist"])
    x = dx.download()
    assert np.linalg.norm(b - A.to_scipy() @ x) <= 2e-8


@pytest.mark.parametrize("case", CASES)
def test_shipped_entry_point_histories(sp, oracle, fixture_system, golden, case):
    """HEM as shipped: AMG_Solver_CPU_baseline, Solver_PCG_1, Solver_PBiCG_1 histories from the reference's prints."""
    A, b = system_by_name(case, oracle, fixture_system)
    g = golden[case]
    dH = sp.DeviceHierarchy(OracleAmg(A).hierarchy().levels)
    db, dx = sp.DeviceVector(data=b), sp.DeviceVector(A.nrow)
    it, hist, ok = dH.amg_solve(db, dx.fill(0.0), 1e-8)
    assert_hist(hist[1:], g["AMG_Solver_CPU_baseline"]["hist"], r0=hist[0])
    it, hist, ok = dH.pcg(db, dx.fill(0.0), 1e-8)
    assert_hist(hist[1:], g["Solver_PCG_1"]["hist"], r0=hist[0])
    np.testing.assert_allclose(np.linalg.norm(dx.download()), g["Solver_PCG_1"]["x_norm"], rtol=1e-9)
    it, hist, ok = dH.pbicgstab(db, dx.fill(0.0), 1e-8)
    assert ok
    assert_hist(hist[1:], g["Solver_PBiCG_1"]["hist"], rtol=1e-8, r0=hist[0])  # BiCGStab amplifies rounding; counts must still match


def test_fixture_headline_counts_on_gpu(sp, oracle, fixture_system):
    """SURVEY Appendix C: 30 V-cycles, 13 PCG iterations, 7 PBiCGStab iterations on the bundled matrix."""
    A, b = fixture_system
    dH = sp.DeviceHierarchy(OracleAmg(A).hierarchy().levels)
    db, dx = sp.DeviceVector(data=b), sp.DeviceVector(A.nrow)
    assert dH.amg_solve(db, dx.fill(0.0), 1e-8)[0] == 30
    assert dH.pcg(db, dx.fill(0.0), 1e-8)[0] == 13
    assert dH.pbicgstab(db, dx.fill(0.0), 1e-8)[0] == 7


def test_unpreconditioned_krylov(sp, fixture_system, golden):
    A, b = fixture_system
    dA = sp.DeviceMatrix.from_csr(A)
    db, dx = sp.DeviceVector(data=b), sp.DeviceVector(A.nrow)
    for fn, key in [(dA.cg, "Solver_CG_1"), (dA.bicgstab, "Solver_BiCG_1")]:
        it, hist, ok = fn(db, dx.fill(0.0), 1e-8, 2000)
        g = golden["fixture"][key]
        # hundreds of unpreconditioned iterations amplify rounding chaotically (BiCGStab most of all): the count is
        # only loosely comparable, the first residuals and the final answer are not
        assert ok and abs(it - g["iters"]) <= g["iters"] // 4
        np.testing.assert_allclose(hist[1:6], g["head"], rtol=1e-9)
        assert np.linalg.norm(b - A.to_scipy() @ dx.download()) <= 1e-7


def test_graph_and_direct_launch_agree_bitwise(sp, oracle, fixture_system):
    A, b = fixture_system
    levels = OracleAmg(A).hierarchy().levels
    db = sp.DeviceVector(data=b)
    out = []
    for use_graph in (False, True):
        dH = sp.DeviceHierarchy(levels, use_graph=use_graph)
        dx = sp.DeviceVector(A.nrow).fill(0.0)
        it, hist, ok = dH.pcg(db, dx, 1e-8)
        out.append((it, hist.copy(), dx.download()))
        dx.fill(0.0)
        it2, hist2, _ = dH.pcg(db, dx, 1e-8)  # second solve on the same handle replays cached graphs
        assert it2 == it and np.array_equal(hist2, hist)
    assert out[0][0] == out[1][0]
    np.testing.assert_array_equal(out[0][1], out[1][1])
    np.testing.assert_array_equal(out[0][2], out[1][2])


def test_graph_and_direct_solves_agree_bitwise_on_hem_and_beck(sp, oracle):
    """V-cycle, AMG-PCG and BiCGStab leave the same bits behind with and without CUDA graphs (HEM and Beck hierarchies),
    and agree with the oracle"""
    A = oracle.gen_poisson3d(40, 36, 32)
    b = np.ones(A.nrow)
    xr = np.random.default_rng(9).standard_normal(A.nrow)
    for coarsening in (0, 1):
        amg = OracleAmg(A, coarsening=coarsening, limit_upper=400, limit_lower=200)
        levels = amg.hierarchy().levels
        assert len(levels) >= 4
        out = {}
        for graph in (True, False):
            dH = sp.DeviceHierarchy(levels, use_graph=graph)
            db = sp.DeviceVector(data=b)
            v = dH.vcycle(db, sp.DeviceVector(data=xr), 2).download()
            dx = sp.DeviceVector(A.nrow).fill(0.0)
            it, hist, ok = dH.pcg(db, dx, 1e-8)
            dy = sp.DeviceVector(A.nrow).fill(0.0)
            itb, histb, okb = dH.pbicgstab(db, dy, 1e-8)
            assert ok and okb
            out[graph] = (v, it, hist, dx.download(), itb, histb, dy.download())
        ref = out[True]
        for key, got in out.items():
            np.testing.assert_array_equal(got[0], ref[0])
            assert got[1] == ref[1] and got[4] == ref[4]
            np.testing.assert_array_equal(got[2], ref[2])
            np.testing.assert_array_equal(got[3], ref[3])
            np.testing.assert_array_equal(got[5], ref[5])
            np.testing.assert_array_equal(got[6], ref[6])
        _, want = amg.pcg(b, np.zeros(A.nrow), 1e-8)
        assert ref[1] == len(want) - 1
        assert_hist(ref[2], want)


def test_sweep_count_and_zero_guess_semantics(sp, oracle, fixture_system):
    """6 sweeps = the reference GPU path's count (SURVEY F7); x_is_zero must equal an explicit zero vector."""
    A, b = fixture_system
    amg = OracleAmg(A)
    levels = amg.hierarchy().levels
    amg.set_smoother(OMEGA, 5)  # oracle runs smooth_iter+1 = 6 sweeps
    dH = sp.DeviceHierarchy(levels, pre_sweeps=6, post_sweeps=6)
    db = sp.DeviceVector(data=b)
    x_a = dH.vcycle(db, sp.DeviceVector(A.nrow).fill(0.0), 1, x_is_zero=False).download()
    x_b = dH.vcycle(db, sp.DeviceVector(A.nrow).fill(123.0), 1, x_is_zero=True).download()
    np.testing.assert_array_equal(x_a, x_b)
    rel_close(x_a, amg.vcycle(b, np.zeros(A.nrow), 1), 1e-10)
    it, hist, ok = dH.amg_solve(db, sp.DeviceVector(A.nrow).fill(0.0), 1e-8)
    assert it == 31  # SURVEY Appendix C, 6-sweep column


def test_host_buffer_entry_point(sp, oracle, fixture_system, golden):
    A, b = fixture_system
    dH = sp.DeviceHierarchy(OracleAmg(A).hierarchy().levels)
    x = np.zeros(A.nrow)
    it, hist, ok = dH.solve_host("pcg", b, x, 1e-8)
    assert ok and it == 13
    assert np.linalg.norm(b - A.to_scipy() @ x) <= 2e-8
    assert sp.launch_count() > 0


# ------------------------------------------------------------------------ larger sizes: size-independent properties
def test_properties_at_scale(sp, oracle):
    """3D 7-point 96^3 (885k rows): linearity, A*1 = row sums, Jacobi fixed point, PCG true residual."""
    nx = 96
    A = oracle.gen_poisson3d(nx, nx, nx)
    n = A.nrow
    dA = sp.DeviceMatrix.from_csr(A)
    rng = np.random.default_rng(4)
    x, y = rng.standard_normal(n), rng.standard_normal(n)
    dx, dy = sp.DeviceVector(data=x), sp.DeviceVector(data=y)
    ones = dA.spmv(sp.DeviceVector(n).fill(1.0)).download()
    rowsum = np.add.reduceat(A.val, A.rowptr[:-1])
    np.testing.assert_array_equal(ones, rowsum)
    np.testing.assert_array_equal(dA.spmv(dx).download(), oracle.spmv(A, x))
    lhs = dA.spmv(sp.DeviceVector(data=2.0 * x + y)).download()
    rel_close(lhs, 2.0 * dA.spmv(dx).download() + dA.spmv(dy).download(), 1e-13)
    b = oracle.spmv(A, x)
    fixed = dA.jacobi(sp.DeviceVector(data=b), sp.DeviceVector(data=x), OMEGA, 3).download()
    rel_close(fixed, x, 1e-13)
    assert dA.residual_norm(sp.DeviceVector(data=b), dx) <= 1e-10 * np.linalg.norm(b)

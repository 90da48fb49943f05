"""V-cycle grid transfers on aggregation operators.

HEM's prolongator P has one 1.0 per row and its restriction R = P^T rows of one or two 1.0.  The upload recognises both
(sparsh_matrix_transfer_info); the V-cycle then runs the residual and the restriction as one fused pass
(sparsh_residual_restrict), the prolongation with the aggregation kernel (no rowptr, no val), and its first sweep from
x = 0 with the diagonal read through the csr-pattern8 twin (sparsh_jacobi_zero).  Each is compared with the kernels it
replaces, bit for bit: every level of a 48^3 HEM hierarchy, rows that take the table walk and the escape path, and x and
b holding Inf, NaN and -0.  A Beck hierarchy (no aggregation operators) keeps the general path and still solves."""
import os

import numpy as np
import pytest
from oracle_bindings import CSR, OracleAmg

OMEGA = 0.66667


def hem_levels(n):
    from sparsh_amg_b200 import generators, host

    host.set_options(threads=min(8, os.cpu_count() or 1), max_levels=32, print_setup=0, print_solve=0, coarsening=0)
    amg = host.HostAmg(host.HostMatrix.from_csr(generators.poisson_7pt(n, n, n)))
    return amg, amg.levels()


@pytest.fixture(scope="module")
def sp():
    import sparsh_amg_b200 as s

    s.init(0)
    return s


@pytest.fixture(scope="module")
def hierarchy48():
    return hem_levels(48)


def same_bits(got, want, msg):
    """NaN where the other has NaN, the same bits everywhere else (-0 and +0 differ).  A NaN's sign and payload are not
    compared: which NaN operand an add propagates is the compiler's choice."""
    nan = np.isnan(want)
    np.testing.assert_array_equal(np.isnan(got), nan, err_msg=msg)
    np.testing.assert_array_equal(np.ascontiguousarray(got[~nan]).view(np.uint64), np.ascontiguousarray(want[~nan]).view(np.uint64),
                                  err_msg=msg)


def fused_applies(sp, dA, dR):
    return dA.kernel()[0] == sp.capi.KIND_PATTERN and dA.kernel_name("residual").startswith("csr_pat2_kernel") and dR.transfer_info()[1]


def check_resid_restrict(sp, M, diag, P, x, b, msg):
    """sparsh_residual_restrict against sparsh_residual + sparsh_restrict with R on the plain scalar kernel; returns
    (fused path taken, result)"""
    dA = sp.DeviceMatrix.from_csr(M, diag=diag)
    dR = sp.DeviceMatrix.from_csr(P, transpose=True)
    dR_ref = sp.DeviceMatrix.from_csr(P, transpose=True).force_kernel(sp.capi.KIND_SCALAR, 256)
    dx, db = sp.DeviceVector(data=x), sp.DeviceVector(data=b)
    got = dA.residual_restrict(dR, db, dx).download()
    want = dR_ref.restrict(dA.residual(db, dx)).download()
    same_bits(got, want, msg)
    return fused_applies(sp, dA, dR), got


def check_prolong(sp, P, xc, xf, msg):
    dP = sp.DeviceMatrix.from_csr(P)
    dP_ref = sp.DeviceMatrix.from_csr(P).force_kernel(sp.capi.KIND_SCALAR, 256)
    assert dP.kernel_name("prolong").startswith("csr_agg_kernel"), msg
    assert dP_ref.kernel_name("prolong").startswith("csr_scalar_kernel"), msg
    got = dP.prolong_add(sp.DeviceVector(data=xc), sp.DeviceVector(data=xf)).download()
    want = dP_ref.prolong_add(sp.DeviceVector(data=xc), sp.DeviceVector(data=xf)).download()
    same_bits(got, want, msg + " prolong")
    same_bits(dP.spmv(sp.DeviceVector(data=xc)).download(), dP_ref.spmv(sp.DeviceVector(data=xc)).download(), msg + " spmv")
    return got


def perturbed_level(L, seed):
    """boundary rows with a perturbed value become patterns of their own (table walk); rows whose smoothing diagonal
    differs from the tabulated one become escapes (CSR arrays)"""
    M0, diag = L["A"], np.ascontiguousarray(L["diag"]).copy()
    M = CSR(M0.nrow, M0.ncol, M0.rowptr.copy(), M0.colindex.copy(), M0.val.copy())
    lens = np.diff(M.rowptr)
    rng = np.random.default_rng(seed)
    short = np.flatnonzero(lens < lens.max())  # boundary rows
    for r in rng.choice(short, min(40, len(short)), replace=False):
        M.val[M.rowptr[r]] *= 1.0 + 1e-3
    esc = rng.choice(np.flatnonzero(lens == lens.max()), 5, replace=False)
    diag[esc] *= 1.0 + 1e-9
    return M, diag


# ------------------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_hem_transfer_operators_are_detected(sp, hierarchy48):
    _amg, levels = hierarchy48
    for k, L in enumerate(levels[:-1]):
        P = L["P"]
        assert sp.DeviceMatrix.from_csr(P).transfer_info() == (True, True, 1.0), k
        one, uni, v = sp.DeviceMatrix.from_csr(P, transpose=True).transfer_info()
        assert uni and v == 1.0, k
        assert not sp.DeviceMatrix.from_csr(L["A"], diag=L["diag"]).transfer_info()[0], k
    # the uploaded hierarchy's own operators
    dH = sp.DeviceHierarchy(levels)
    for k in range(len(levels) - 1):
        _A, dP, dR = dH.level(k)
        assert dP.transfer_info() == (True, True, 1.0) and dR.transfer_info()[1], k
        assert dP.kernel_name("prolong") == "csr_agg_kernel<EPI_PROLONG,true>", k
    dH.free()


@pytest.mark.gpu
def test_fused_residual_restriction_is_bit_identical_on_every_hem_level(sp, hierarchy48):
    _amg, levels = hierarchy48
    rng = np.random.default_rng(41)
    fused = 0
    for k, L in enumerate(levels[:-1]):
        M, diag = L["A"], np.ascontiguousarray(L["diag"])
        x, b = rng.standard_normal(M.nrow), rng.standard_normal(M.nrow)
        fused += check_resid_restrict(sp, M, diag, L["P"], x, b, f"level {k}")[0]
    assert fused >= 4


@pytest.mark.gpu
def test_fused_residual_restriction_on_table_and_escape_rows(sp, hierarchy48):
    _amg, levels = hierarchy48
    for lev in (0, 1, 3):
        M, diag = perturbed_level(levels[lev], 43 + lev)
        dA = sp.DeviceMatrix.from_csr(M, diag=diag)
        n_pat, _, n_esc, _ = dA.pattern_stats()
        n_masked, _ = dA.pattern_mask_stats()
        assert n_esc >= 5 and n_pat - 1 - n_masked > 0, lev  # both rare paths are reached
        rng = np.random.default_rng(47 + lev)
        x, b = rng.standard_normal(M.nrow), rng.standard_normal(M.nrow)
        assert check_resid_restrict(sp, M, diag, levels[lev]["P"], x, b, f"level {lev}")[0], lev


@pytest.mark.gpu
def test_fused_residual_restriction_with_inf_nan_and_negative_zero(sp, hierarchy48):
    _amg, levels = hierarchy48
    for lev in (0, 2):
        L = levels[lev]
        M, diag, P = L["A"], np.ascontiguousarray(L["diag"]), L["P"]
        rng = np.random.default_rng(53 + lev)
        x, b = rng.standard_normal(M.nrow), rng.standard_normal(M.nrow)
        for i, c in enumerate(rng.choice(M.nrow, 30, replace=False)):
            x[c] = (np.inf, np.nan, -0.0, -np.inf)[i % 4]
        for i, c in enumerate(rng.choice(M.nrow, 30, replace=False)):
            b[c] = (np.nan, -0.0, np.inf)[i % 3]
        # a pair whose residuals are both -0 (b = -0, every x the rows touch 0): the sum is 0 + (-0) + (-0) = +0, as in
        # the scalar kernel; starting the sum from the first product would give -0
        Rt = CSR(P.ncol, P.nrow, *transpose(P))
        pairs = np.flatnonzero(np.diff(Rt.rowptr) == 2)
        pair = int(pairs[len(pairs) // 2])
        for j in Rt.colindex[Rt.rowptr[pair]:Rt.rowptr[pair] + 2]:
            x[M.colindex[M.rowptr[j]:M.rowptr[j + 1]]] = 0.0
            b[j] = -0.0
        fused, got = check_resid_restrict(sp, M, diag, P, x, b, f"level {lev}")
        assert fused, lev
        assert got[pair] == 0.0 and not np.signbit(got[pair]), lev
        assert np.isnan(got).any() and np.isinf(got).any(), lev


def transpose(P):
    """R = P^T as (rowptr, colindex, val), rows listing the fine rows in ascending order (as the upload builds it)"""
    order = np.argsort(P.colindex, kind="stable")
    rp = np.concatenate([[0], np.cumsum(np.bincount(P.colindex, minlength=P.ncol))]).astype(np.int32)
    rows = np.repeat(np.arange(P.nrow, dtype=np.int32), np.diff(P.rowptr))
    return rp, rows[order].astype(np.int32), np.asarray(P.val)[order]


@pytest.mark.gpu
def test_aggregation_prolongation_is_bit_identical(sp, hierarchy48):
    _amg, levels = hierarchy48
    for k, L in enumerate(levels[:-1]):
        P = L["P"]
        rng = np.random.default_rng(59 + k)
        xc, xf = rng.standard_normal(P.ncol), rng.standard_normal(P.nrow)
        check_prolong(sp, P, xc, xf, f"level {k}")
    # special values: x_c = -0 with x_f = -0 gives +0 (0 + 1*(-0) = +0, then +0 + -0 = +0), Inf and NaN propagate
    P = levels[0]["P"]
    rng = np.random.default_rng(61)
    xc, xf = rng.standard_normal(P.ncol), rng.standard_normal(P.nrow)
    xc[:12] = [np.inf, np.nan, -0.0, -np.inf] * 3
    zero_rows = np.flatnonzero(P.colindex == 2)
    xf[zero_rows] = -0.0
    xf[-8:] = [np.nan, np.inf, -0.0, -np.inf] * 2
    got = check_prolong(sp, P, xc, xf, "special values")
    assert np.all(got[zero_rows] == 0.0) and not np.signbit(got[zero_rows]).any()
    # a non-uniform one-entry-per-row operator reads its values
    Pv = CSR(P.nrow, P.ncol, P.rowptr, P.colindex, rng.standard_normal(P.nnz))
    assert sp.DeviceMatrix.from_csr(Pv).transfer_info()[:2] == (True, False)
    assert sp.DeviceMatrix.from_csr(Pv).kernel_name("prolong") == "csr_agg_kernel<EPI_PROLONG,false>"
    check_prolong(sp, Pv, xc, xf, "non-uniform values")


@pytest.mark.gpu
def test_zero_sweep_reads_the_pattern_diagonal(sp, hierarchy48):
    """x = (omega*b)/d: IEEE multiplication and division are correctly rounded on both sides, so numpy gives the bits"""
    _amg, levels = hierarchy48
    rng = np.random.default_rng(67)
    cases = [(L["A"], np.ascontiguousarray(L["diag"]), f"level {k}") for k, L in enumerate(levels)]
    M, diag = perturbed_level(levels[1], 71)
    cases.append((M, diag, "escapes"))
    lean = 0
    for M, diag, msg in cases:
        dA = sp.DeviceMatrix.from_csr(M, diag=diag)
        lean += dA.kernel_name("jacobi").startswith("csr_pat2_kernel")
        b = rng.standard_normal(M.nrow)
        b[:6] = [np.inf, -0.0, np.nan, 0.0, -np.inf, 1e-310]
        got = dA.jacobi_zero(sp.DeviceVector(data=b), OMEGA).download()
        same_bits(got, (OMEGA * b) / diag, msg)
    assert lean >= 5
    assert sp.DeviceMatrix.from_csr(M, diag=diag).pattern_stats()[2] >= 5


@pytest.mark.gpu
def test_beck_hierarchy_keeps_the_general_path_and_solves(sp, oracle):
    A = oracle.gen_poisson3d(24, 24, 24)
    amg = OracleAmg(A, coarsening=1)
    levels = amg.hierarchy().levels
    for k, L in enumerate(levels[:-1]):
        one, uni, _ = sp.DeviceMatrix.from_csr(L["P"]).transfer_info()
        assert not one and not uni, k
        assert not sp.DeviceMatrix.from_csr(L["P"], transpose=True).transfer_info()[1], k
    dH = sp.DeviceHierarchy(levels)
    b = np.ones(A.nrow)
    dx = sp.DeviceVector(A.nrow).fill(0.0)
    it, hist, ok = dH.pcg(sp.DeviceVector(data=b), dx, 1e-8)
    _, want = amg.pcg(b, np.zeros(A.nrow), 1e-8)
    assert ok and abs(it - (len(want) - 1)) <= 1, (it, len(want) - 1)
    m = min(len(hist), len(want))
    np.testing.assert_allclose(hist[:m], want[:m], rtol=1e-10, atol=1e-13 * want[0])
    dH.free()

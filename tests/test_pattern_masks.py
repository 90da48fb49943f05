"""Masked pattern-0 rows of the lean csr-pattern8 kernel (csr_pat2_kernel).

A pattern whose (offset, value bits) list is an in-order subsequence of pattern 0's, with pattern 0's diagonal, is
evaluated as pattern 0 with the missing terms skipped instead of being walked from the table.  CPU: the mask
derivation (sparsh_pattern_masks) on hand-made tables and on every level of a 48^3 HEM hierarchy.  GPU: the kernel
bit-identical to the stream kernel and to the oracle on that hierarchy, on rows that must leave the masked path, on x
holding Inf, NaN and -0 where masked rows skip a term, for every epilogue and both tile shapes."""
import ctypes as C
import os

import numpy as np
import pytest
from oracle_bindings import CSR
from test_host_setup import _pattern_encode

VALID = 0x80
OMEGA = 0.66667
N7 = [-2304, -48, -1, 0, 1, 48, 2304]
V7 = [-1.0, -1.0, -1.0, 6.0, -1.0, -1.0, -1.0]


def masks(patterns):
    """sparsh_pattern_masks over a table given as a list of [(offset, value), ...], pattern 0 first"""
    import sparsh_amg_b200 as sp

    start = np.concatenate([[0], np.cumsum([len(p) for p in patterns])]).astype(np.int32)
    off = np.array([o for p in patterns for o, _ in p] or [0], dtype=np.int32)
    val = np.array([v for p in patterns for _, v in p] or [0.0], dtype=np.float64)
    m = np.full(256, 0x55, dtype=np.uint8)
    sp.capi.check(sp.capi.load().sparsh_pattern_masks(len(patterns), sp.capi.ip(start), sp.capi.dp(val), sp.capi.ip(off),
                                                      m.ctypes.data_as(C.c_void_p)))
    return m


def bits(*ks):
    return VALID | sum(1 << k for k in ks)


def test_masks_of_hand_made_tables():
    p0 = list(zip(N7, V7))
    nudged = np.nextafter(-1.0, 0.0)
    cases = [
        [(-48, -1.0), (-1, -1.0), (0, 6.0), (1, -1.0), (2304, -1.0)],  # a subsequence (a boundary row)
        [(-2304, -1.0), (-48, -1.0), (-1, nudged), (0, 6.0), (1, -1.0), (48, -1.0), (2304, -1.0)],  # one value, last bit
        [(-48, -1.0), (-1, -1.0), (1, -1.0), (48, -1.0)],  # no diagonal entry: its diagonal is 0, not 6
        [(-2304, -1.0), (-48, -1.0), (-1, -1.0), (0, 6.0), (1, -1.0), (2, -1.0), (48, -1.0)],  # an extra entry
        [(-48, -1.0), (-2304, -1.0), (0, 6.0)],  # a reordered entry
        [(0, 6.0)],  # the diagonal alone
    ]
    m = masks([p0] + cases)
    assert m[0] == bits(0, 1, 2, 3, 4, 5, 6)
    assert m[1] == bits(1, 2, 3, 4, 6)
    assert list(m[2:6]) == [0, 0, 0, 0]
    assert m[6] == bits(3)
    assert not np.any(m[7:])  # ids the table does not have, the escape id 255 included
    # pattern 0 with two offset-0 entries: a row keeping only the second has a different tabulated diagonal
    m = masks([[(-1, -1.0), (0, 5.0), (0, 1.0), (1, -1.0)], [(-1, -1.0), (0, 1.0)], [(0, 5.0), (1, -1.0)]])
    assert m[1] == 0 and m[2] == bits(1, 3)
    # the 5-point stencil: every subsequence with the diagonal is masked
    p5 = [(-96, -1.0), (-1, -1.0), (0, 4.0), (1, -1.0), (96, -1.0)]
    m = masks([p5, p5[1:], p5[:4], p5[1:4], p5[2:3]])
    assert list(m[:5]) == [bits(0, 1, 2, 3, 4), bits(1, 2, 3, 4), bits(0, 1, 2, 3), bits(1, 2, 3), bits(2)]
    # more than 7 entries in pattern 0: no masks at all (the kernel holds one bit per entry of pattern 0)
    p8 = [(o, -1.0) for o in range(-4, 4)]
    assert not np.any(masks([p8, p8[1:]]))
    assert not np.any(masks([]))
    # a full table, as the encoder can return it: 255 patterns (ids 0..254), the escape id 255 stays unmasked
    full = [p5] + [p5[1:]] * 253 + [p5[:2]]
    m = masks(full)
    assert m[253] == bits(1, 2, 3, 4) and m[254] == 0 and m[255] == 0  # the last one lacks the diagonal
    import sparsh_amg_b200 as sp

    with pytest.raises(sp.SparshError):
        masks(full + [p5])  # 256 patterns: more ids than a pattern byte holds


def hem_levels(n):
    from sparsh_amg_b200 import generators, host

    host.set_options(threads=min(8, os.cpu_count() or 1), max_levels=32, print_setup=0, print_solve=0, coarsening=0)
    amg = host.HostAmg(host.HostMatrix.from_csr(generators.poisson_7pt(n, n, n)))
    return amg, amg.levels()


def level_masks(M, diag):
    pat, ent_val, ent_off, start, n_pat, n_esc = _pattern_encode(M, np.ascontiguousarray(diag))
    return pat, masks([list(zip(ent_off[start[p]:start[p + 1]], ent_val[start[p]:start[p + 1]])) for p in range(n_pat)]), n_pat, n_esc


def test_every_boundary_pattern_of_a_hem_hierarchy_is_masked():
    """on every level of the 48^3 HEM hierarchy each pattern other than the interior one is the interior row with terms
    left out (Dirichlet boundary rows and their Galerkin coarsenings): no row needs the table walk"""
    _amg, levels = hem_levels(48)
    assert len(levels) >= 6
    for k, L in enumerate(levels):
        pat, m, n_pat, n_esc = level_masks(L["A"], L["diag"])
        assert n_pat > 1 and n_esc == 0, k
        assert np.all(m[:n_pat] & VALID), (k, m[:n_pat])
        assert m[0] == bits(*range(7)), k


# ------------------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def sp():
    import sparsh_amg_b200 as s

    s.init(0)
    return s


def assert_same_bits(got, want, msg):
    """NaN where the other has NaN, the same bits everywhere else (-0 and +0 differ).  A NaN's payload and sign are not
    compared: the compiler orders the operands of an add freely, and of two NaN operands the result keeps one's payload."""
    nan = np.isnan(want)
    np.testing.assert_array_equal(np.isnan(got), nan, err_msg=msg)
    np.testing.assert_array_equal(np.ascontiguousarray(got[~nan]).view(np.uint64), np.ascontiguousarray(want[~nan]).view(np.uint64),
                                  err_msg=msg)


def run_ops(sp, dA, M, x, b, xc):
    """every epilogue on M: SpMV, residual, Jacobi (2 and 7 sweeps), prolongation-correction (M as the transfer),
    SpMV+dot, residual norm, and one row-by-row SOR sweep (one colour per row: a deterministic Gauss-Seidel sweep)"""
    dx, db = sp.DeviceVector(data=x), sp.DeviceVector(data=b)
    y, pdot = dA.spmv_dot(dx)
    out = [dA.spmv(dx).download(), dA.residual(db, dx).download(), dA.jacobi(db, sp.DeviceVector(data=x), OMEGA, 2).download(),
           dA.jacobi(db, sp.DeviceVector(data=x), OMEGA, 7).download(),
           dA.prolong_add(sp.DeviceVector(data=xc), sp.DeviceVector(data=x)).download(), y.download()]
    if M.nrow <= 4096:
        out.append(dA.mc_sor(np.arange(M.nrow + 1), db, sp.DeviceVector(data=x), OMEGA, 1).download())
    return out, pdot, dA.residual_norm(db, dx)


def oracle_ops(oracle, M, diag, x, b, xc):
    want = [oracle.spmv(M, x), oracle.store_residual(M, b, x), oracle.jacobi(M, diag, b, x, OMEGA, 1),
            oracle.jacobi(M, diag, b, x, OMEGA, 6), oracle.transfer_solution(M, xc, x), oracle.spmv(M, x)]
    if M.nrow <= 4096:
        want.append(oracle.sor_multicolor(M, diag, np.arange(M.nrow + 1), b, x, OMEGA, 1))
    return want


def check_lean(sp, oracle, M, diag, x, b, threads):
    """the lean kernel against the stream kernel (bit for bit) and the oracle; False when the lean kernel does not apply"""
    dA = sp.DeviceMatrix.from_csr(M, diag=diag)
    dA.force_kernel(sp.capi.KIND_PATTERN, threads)
    if not dA.kernel_name("jacobi").startswith("csr_pat2_kernel"):
        return False
    xc = np.random.default_rng(3).standard_normal(M.nrow)
    lean, lean_dot, lean_nrm = run_ops(sp, dA, M, x, b, xc)
    dA.force_kernel(sp.capi.KIND_STREAM, threads)
    ref, ref_dot, ref_nrm = run_ops(sp, dA, M, x, b, xc)
    for i, (got, w, o) in enumerate(zip(lean, ref, oracle_ops(oracle, M, diag, x, b, xc))):
        assert_same_bits(got, w, f"op {i}")
        np.testing.assert_array_equal(got, o, err_msg=f"op {i}")
    # fused reductions: identical contributions, fixed but different summation trees in the two kernels
    np.testing.assert_allclose(lean_dot, ref_dot, rtol=1e-12)
    np.testing.assert_allclose(lean_nrm, ref_nrm, rtol=1e-12)
    return True


@pytest.fixture(scope="module")
def hierarchy48():
    return hem_levels(48)


@pytest.mark.gpu
@pytest.mark.parametrize("threads", [256, 128])
def test_lean_kernel_is_bit_identical_on_every_hem_level(sp, oracle, hierarchy48, threads, monkeypatch):
    monkeypatch.setenv("SPARSH_PATTERN", "2")  # build the twin, keep the default kernel; the test forces kinds
    _amg, levels = hierarchy48
    rng = np.random.default_rng(29)
    used = 0
    for L in levels:
        M, diag = L["A"], np.ascontiguousarray(L["diag"])
        dA = sp.DeviceMatrix.from_csr(M, diag=diag)
        n_masked, cover = dA.pattern_mask_stats()
        if dA.pattern_stats()[0] > 1:
            assert n_masked == dA.pattern_stats()[0] - 1 and cover == 1.0
        x, b = rng.standard_normal(M.nrow), rng.standard_normal(M.nrow)
        used += check_lean(sp, oracle, M, diag, x, b, threads)
    assert used >= 5


@pytest.mark.gpu
@pytest.mark.parametrize("threads", [256, 128])
def test_rows_that_are_not_masked_take_the_table_or_the_escape(sp, oracle, hierarchy48, threads, monkeypatch):
    """perturbed values make boundary rows patterns of their own (table path); a smoothing diagonal that differs from
    the tabulated one makes rows escapes (CSR path); the masked rows around them stay exact"""
    monkeypatch.setenv("SPARSH_PATTERN", "2")
    _amg, levels = hierarchy48
    L = levels[1]
    M0, diag = L["A"], np.ascontiguousarray(L["diag"]).copy()
    M = CSR(M0.nrow, M0.ncol, M0.rowptr.copy(), M0.colindex.copy(), M0.val.copy())
    pat, m, _n_pat, _ = level_masks(M0, diag)
    boundary = np.flatnonzero(pat != 0)
    rng = np.random.default_rng(31)
    for r in rng.choice(boundary, 40, replace=False):
        M.val[M.rowptr[r]] *= 1.0 + 1e-3
    esc = rng.choice(np.flatnonzero(pat == 0), 5, replace=False)
    diag[esc] *= 1.0 + 1e-9
    dA = sp.DeviceMatrix.from_csr(M, diag=diag)
    n_pat, _, n_esc, _ = dA.pattern_stats()
    n_masked, _ = dA.pattern_mask_stats()
    assert n_esc >= 5 and n_pat - 1 - n_masked > 0 and n_masked > 0
    x, b = rng.standard_normal(M.nrow), rng.standard_normal(M.nrow)
    assert check_lean(sp, oracle, M, diag, x, b, threads)


@pytest.mark.gpu
@pytest.mark.parametrize("threads", [256, 128])
def test_masked_rows_ignore_inf_nan_and_negative_zero_they_skip(sp, oracle, hierarchy48, threads, monkeypatch):
    """x holds Inf, NaN and -0 at columns that masked rows do NOT have (their missing neighbours): a kernel that zeroed
    the product instead of skipping the add would turn those rows into NaN or change a sign"""
    monkeypatch.setenv("SPARSH_PATTERN", "2")
    _amg, levels = hierarchy48
    for lev in (0, len(levels) - 3):
        L = levels[lev]
        M, diag = L["A"], np.ascontiguousarray(L["diag"])
        pat, m, n_pat, _ = level_masks(M, diag)
        _, ent_val, ent_off, start, _, _ = _pattern_encode(M, diag)
        off0 = ent_off[start[0]:start[1]]
        rng = np.random.default_rng(37 + lev)
        x, b = rng.standard_normal(M.nrow), rng.standard_normal(M.nrow)
        skipped = []
        for r in np.flatnonzero(pat != 0):
            for k, o in enumerate(off0):
                if not m[pat[r]] & (1 << k) and 0 <= r + o < M.ncol:
                    skipped.append((r, r + o))
        assert skipped, lev
        picks = [skipped[i] for i in rng.choice(len(skipped), min(12, len(skipped)), replace=False)]
        for i, (_r, c) in enumerate(picks):
            x[c] = (np.inf, np.nan, -0.0)[i % 3]
        assert check_lean(sp, oracle, M, diag, x, b, threads)
        spmv = sp.DeviceMatrix.from_csr(M, diag=diag).spmv(sp.DeviceVector(data=x)).download()
        assert np.isfinite(spmv[[r for r, c in picks if not np.isfinite(x[c])]]).any()

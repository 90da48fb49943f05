"""Refreshing a resident hierarchy's coefficients (sparsh_hierarchy_refresh) and a matrix's values
(sparsh_matrix_update_values).

A refresh keeps P_l and R_l and recomputes every A_{l+1} = P_l^T A_l P_l on the device, then rebuilds each level's
twins and the coarse inverse.  Its result is pinned bit for bit to what the repository already builds: the host setup's
levels (a refresh with the values a hierarchy already holds), and a fresh DeviceHierarchy built from the new A_0, the
same P_l and the device Galerkin products (new values).  A matrix's value update is pinned to sparsh_matrix_create on
the same arrays: kernel family, twins, and the SpMV, residual and Jacobi bits of every family."""
import os

import numpy as np
import pytest
from oracle_bindings import CSR

pytestmark = pytest.mark.gpu

OMEGA = 0.66667
EPIS = ["spmv", "residual", "jacobi", "prolong", "sor", "spmv_dot", "resnorm"]


@pytest.fixture(scope="module")
def sp():
    import sparsh_amg_b200 as s

    s.init(0)
    return s


def same_bits(got, want, msg):
    """NaN where the other has NaN, the same bits everywhere else (-0 and +0 differ)"""
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, (msg, got.shape, want.shape)
    nan = np.isnan(want)
    np.testing.assert_array_equal(np.isnan(got), nan, err_msg=msg)
    np.testing.assert_array_equal(np.ascontiguousarray(got[~nan]).view(np.uint64), np.ascontiguousarray(want[~nan]).view(np.uint64),
                                  err_msg=msg)


def host_levels(kind, n=32):
    """(levels as CSR copies, the HostAmg) for 'hem' | 'beck' | 'sa' | 'sor' (HEM, multicolour SOR) on 3D Poisson n^3,
    or 'diffusion27' (HEM on the 27-point variable-coefficient operator)"""
    from sparsh_amg_b200 import host

    coarsening = {"hem": 0, "beck": 1, "sa": 2, "sor": 0, "diffusion27": 0}[kind]
    host.set_options(threads=min(8, os.cpu_count() or 1), max_levels=32, print_setup=0, print_solve=0, coarsening=coarsening,
                     relax=0.66667, coarse_upper=500 if kind == "sa" else 4000, coarse_lower=100 if kind == "sa" else 2000)
    M = host.HostMatrix.diffusion27(n, n, n) if kind == "diffusion27" else host.HostMatrix.poisson3d(n, n, n)
    amg = host.HostAmg(M, sor=kind == "sor")
    levels = []
    for L in amg.levels():
        A, P = L["A"], L["P"]
        levels.append(dict(A=CSR(A.nrow, A.ncol, A.rowptr.copy(), A.colindex.copy(), A.val.copy()), diag=np.array(L["diag"]),
                           P=None if P is None else CSR(P.nrow, P.ncol, P.rowptr.copy(), P.colindex.copy(), P.val.copy())))
    assert len(levels) >= 3
    return levels, amg, M


def extracted_diag(A):
    """sp_matrix_fill_diagonal: the first stored entry with col == row, else 0"""
    d = np.zeros(A.nrow)
    for i in range(A.nrow):
        lo, hi = A.rowptr[i], A.rowptr[i + 1]
        hit = np.flatnonzero(A.colindex[lo:hi] == i)
        if hit.size:
            d[i] = A.val[lo + hit[0]]
    return d


def galerkin_levels(sp, A0, diag0, levels):
    """A_0 with the given diagonal, the same P_l, A_{l+1} = device Galerkin product, diagonals extracted"""
    out, A = [], A0
    for k, L in enumerate(levels):
        out.append(dict(A=A, diag=diag0 if k == 0 else extracted_diag(A), P=L["P"]))
        if L["P"] is not None:
            got = sp.galerkin_rap(A, L["P"])
            assert got is not None
            A = CSR(L["P"].ncol, L["P"].ncol, *got)
    return out


def with_values(A, val):
    return CSR(A.nrow, A.ncol, A.rowptr, A.colindex, np.ascontiguousarray(val, dtype=np.float64))


def shifted(A, sigma):
    """A + sigma I on the stored diagonal entries (the time-step case)"""
    v = A.val.copy()
    rows = np.repeat(np.arange(A.nrow), np.diff(A.rowptr))
    v[A.colindex == rows] += sigma
    return with_values(A, v)


def describe(M):
    """every value-derived choice of a device matrix"""
    if M is None:
        return None
    return (M.kernel(), [M.kernel_name(e) for e in EPIS], M.pattern_stats(), M.pattern_mask_stats(), M.transfer_info())


def hierarchy_state(dH):
    return [tuple(describe(m) for m in dH.level(k)) for k in range(dH.nlevels)]


def assert_levels_equal(sp, dH, levels, msg):
    for k, L in enumerate(levels):
        A = dH.level(k)[0]
        rp, ci, v, d = A.fetch()
        np.testing.assert_array_equal(rp, L["A"].rowptr, err_msg=f"{msg} level {k} rowptr")
        np.testing.assert_array_equal(ci, L["A"].colindex, err_msg=f"{msg} level {k} colindex")
        same_bits(v, L["A"].val, f"{msg} level {k} val")
        same_bits(d, L["diag"], f"{msg} level {k} diag")


def pcg(sp, dH, b, tol=1e-9):
    x = sp.DeviceVector(dH.n).fill(0.0)
    it, hist, ok = dH.pcg(sp.DeviceVector(data=b), x, tol, max_iter=200)
    return it, hist, x.download()


def assert_same_hierarchy(sp, got, want, nlev, msg):
    """levels' arrays, choices, per-level kernels, coarse solve, a V-cycle from 0 and a PCG solve, bit for bit"""
    assert hierarchy_state(got) == hierarchy_state(want), msg
    rng = np.random.default_rng(5)
    for k in range(nlev):
        ga, wa = got.level(k)[0], want.level(k)[0]
        g, w = ga.fetch(), wa.fetch()
        for name, a, b in zip(("rowptr", "colindex", "val", "diag"), g, w):
            same_bits(a.astype(np.float64) if a.dtype != np.float64 else a, b.astype(np.float64) if b.dtype != np.float64 else b,
                      f"{msg} level {k} {name}")
        x, b = rng.standard_normal(ga.nrow), rng.standard_normal(ga.nrow)
        same_bits(ga.spmv(sp.DeviceVector(data=x)).download(), wa.spmv(sp.DeviceVector(data=x)).download(), f"{msg} {k} spmv")
        same_bits(ga.residual(sp.DeviceVector(data=b), sp.DeviceVector(data=x)).download(),
                  wa.residual(sp.DeviceVector(data=b), sp.DeviceVector(data=x)).download(), f"{msg} {k} residual")
        same_bits(ga.jacobi(sp.DeviceVector(data=b), sp.DeviceVector(data=x), OMEGA, 3).download(),
                  wa.jacobi(sp.DeviceVector(data=b), sp.DeviceVector(data=x), OMEGA, 3).download(), f"{msg} {k} jacobi")
    bc = sp.DeviceVector(data=rng.standard_normal(got.level(nlev - 1)[0].nrow))
    same_bits(got.coarse_solve(bc).download(), want.coarse_solve(bc).download(), f"{msg} coarse solve")
    b0 = rng.standard_normal(got.n)
    xs = [h.vcycle(sp.DeviceVector(data=b0), sp.DeviceVector(got.n).fill(0.0), 1, x_is_zero=True).download() for h in (got, want)]
    same_bits(xs[0], xs[1], f"{msg} vcycle")
    (ig, hg, xg), (iw, hw, xw) = pcg(sp, got, b0), pcg(sp, want, b0)
    assert ig == iw, msg
    same_bits(hg, hw, f"{msg} pcg history")
    same_bits(xg, xw, f"{msg} pcg x")


@pytest.mark.parametrize("kind", ["hem", "beck", "sa", "sor", "diffusion27"])
def test_refresh_with_the_same_values_reproduces_the_host_setup(sp, kind):
    levels, amg, M = host_levels(kind)
    dH = amg.upload() if kind == "sor" else sp.DeviceHierarchy(levels)
    before = hierarchy_state(dH)
    dH.refresh(levels[0]["A"].val, diag=levels[0]["diag"])
    assert_levels_equal(sp, dH, levels, kind)
    assert hierarchy_state(dH) == before
    amg.free()


@pytest.mark.parametrize("kind", ["hem", "beck", "sa"])
def test_refresh_with_new_values_equals_a_fresh_build(sp, kind):
    from oracle_bindings import Oracle

    levels, amg, M = host_levels(kind)
    dH = sp.DeviceHierarchy(levels, use_graph=False)
    for sigma in (0.5, 3.0, 1e-3):
        A0 = shifted(levels[0]["A"], sigma)
        diag0 = extracted_diag(A0) * (1.0 + 1e-3)  # a smoothing diagonal that is not the extracted one
        dH.refresh(A0.val, diag=sp.DeviceVector(data=diag0))
        want_levels = galerkin_levels(sp, A0, diag0, levels)
        fresh = sp.DeviceHierarchy(want_levels, use_graph=False)
        assert_levels_equal(sp, dH, want_levels, f"{kind} sigma={sigma}")
        assert_same_hierarchy(sp, dH, fresh, len(levels), f"{kind} sigma={sigma}")
        for k in range(1, len(levels)):  # and the oracle's product of the refreshed levels
            rp, ci, v, _ = dH.level(k)[0].fetch()
            Af = dH.level(k - 1)[0].fetch()
            want = Oracle.get().rap(CSR(Af[0].size - 1, Af[0].size - 1, Af[0], Af[1], Af[2]), levels[k - 1]["P"])
            np.testing.assert_array_equal(rp, want.rowptr)
            np.testing.assert_array_equal(ci, want.colindex)
            np.testing.assert_allclose(v, want.val, rtol=1e-13, atol=1e-13 * np.abs(want.val).max())
        fresh.free()
    dH.free()
    amg.free()


@pytest.mark.parametrize("env", [{}, {"SPARSH_PATTERN": "0"}, {"SPARSH_DICT": "2"}])
def test_refresh_changes_kernel_families_as_create_does(sp, monkeypatch, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    levels, amg, M = host_levels("hem")
    dH = sp.DeviceHierarchy(levels, use_graph=False)
    before = hierarchy_state(dH)
    A0 = levels[0]["A"]
    d = np.random.default_rng(3).uniform(0.5, 2.0, A0.nrow)  # D A D: rows stop repeating
    rows = np.repeat(np.arange(A0.nrow), np.diff(A0.rowptr))
    dH.refresh(d[rows] * A0.val * d[A0.colindex])
    for k in range(len(levels)):
        got = dH.level(k)[0]
        rp, ci, v, dg = got.fetch()
        want = sp.DeviceMatrix(got.nrow, got.ncol, rp, ci, v)
        assert describe(got) == describe(want), (env, k)
        same_bits(dg, want.fetch()[3], f"level {k} diag")
    if not env:
        assert dH.level(0)[0].pattern_stats()[0] == 0  # no repeating rows on level 0 any more
    dH.refresh(A0.val, diag=levels[0]["diag"])  # back to constant coefficients: the pattern twin and the lean kernel return
    assert hierarchy_state(dH) == before
    assert_levels_equal(sp, dH, levels, f"back {env}")
    if not env:
        assert dH.level(0)[0].kernel_name("jacobi").startswith("csr_pat2_kernel")
    amg.free()


def test_refresh_drops_captured_graphs(sp):
    levels, amg, M = host_levels("hem")
    dH = sp.DeviceHierarchy(levels, use_graph=True)
    b = np.random.default_rng(9).standard_normal(dH.n)
    for _ in range(2):  # first use runs directly, the second captures and replays
        pcg(sp, dH, b)
    A0 = shifted(levels[0]["A"], 2.0)
    dH.refresh(A0.val)
    fresh = sp.DeviceHierarchy(galerkin_levels(sp, A0, extracted_diag(A0), levels), use_graph=True)
    for _ in range(2):
        (ig, hg, xg), (iw, hw, xw) = pcg(sp, dH, b), pcg(sp, fresh, b)
        assert ig == iw
        same_bits(hg, hw, "pcg history")
        same_bits(xg, xw, "pcg x")
    amg.free()


def test_two_refreshes_equal_one(sp):
    levels, amg, M = host_levels("beck")
    twice = sp.DeviceHierarchy(levels, use_graph=False)
    once = sp.DeviceHierarchy(levels, use_graph=False)
    A1, A2 = shifted(levels[0]["A"], 5.0), shifted(levels[0]["A"], 0.25)
    twice.refresh(A1.val)
    twice.refresh(A2.val)
    once.refresh(A2.val)
    assert_same_hierarchy(sp, twice, once, len(levels), "twice")
    amg.free()


def matrices():
    """stencil, ragged random and rectangular matrices, each with two sets of values"""
    from sparsh_amg_b200 import generators
    import scipy.sparse as sps

    rng = np.random.default_rng(17)
    S = generators.poisson_7pt(14, 13, 12)
    out = [("stencil", CSR(S.nrow, S.ncol, S.rowptr, S.colindex, S.val))]
    R = (sps.random(3000, 3000, density=0.004, random_state=4, format="csr") + sps.eye(3000) * 8.0).tocsr()
    R.sort_indices()
    out.append(("ragged", CSR(3000, 3000, R.indptr, R.indices, R.data)))
    Q = sps.random(2000, 700, density=0.01, random_state=6, format="csr")
    Q.sort_indices()
    out.append(("rectangular", CSR(2000, 700, Q.indptr, Q.indices, Q.data)))
    for name, A in out:  # the stencil's second values come from 40 numbers: no repeating rows, but a csr-dict16 twin
        yield name, A, rng.choice(np.linspace(-1.0, 1.0, 40), A.nnz) if name == "stencil" else rng.uniform(-1.0, 1.0, A.nnz)


def families(M, sp):
    K = sp.capi
    out = [(K.KIND_SCALAR, 256), (K.KIND_STREAM, 128), (K.KIND_STREAM, 256), (K.KIND_VECTOR, 4), (K.KIND_VECTOR, 32)]
    if M.pattern_stats()[0]:
        out += [(K.KIND_PATTERN, 128), (K.KIND_PATTERN, 256)]
    return out


@pytest.mark.parametrize("env", [{}, {"SPARSH_DICT": "2"}])
def test_matrix_update_values_equals_create(sp, monkeypatch, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    rng = np.random.default_rng(23)
    for name, A, v2 in matrices():
        B = with_values(A, v2)
        for new in (B, A):  # to other values and back
            got = sp.DeviceMatrix.from_csr(A if new is B else B)
            got.force_kernel(sp.capi.KIND_VECTOR, 2)  # forgotten by the update
            got.update_values(new.val)
            want = sp.DeviceMatrix.from_csr(new)
            assert describe(got) == describe(want), (name, env)
            g, w = got.fetch(), want.fetch()
            for a, b in zip(g, w):
                if b is None:
                    assert a is None
                else:
                    np.testing.assert_array_equal(a, b)
            x, b = rng.standard_normal(A.ncol), rng.standard_normal(A.nrow)
            kinds = families(want, sp) + ([(sp.capi.KIND_DICT, 128)] if want.kernel()[0] == sp.capi.KIND_DICT else [])
            for kind, tl in kinds:
                got.force_kernel(kind, tl)
                want.force_kernel(kind, tl)
                msg = f"{name} {env} kind {kind}/{tl}"
                same_bits(got.spmv(sp.DeviceVector(data=x)).download(), want.spmv(sp.DeviceVector(data=x)).download(), msg)
                if A.nrow == A.ncol:
                    same_bits(got.residual(sp.DeviceVector(data=b), sp.DeviceVector(data=x)).download(),
                              want.residual(sp.DeviceVector(data=b), sp.DeviceVector(data=x)).download(), msg)
                    same_bits(got.jacobi(sp.DeviceVector(data=b), sp.DeviceVector(data=x), OMEGA, 2).download(),
                              want.jacobi(sp.DeviceVector(data=b), sp.DeviceVector(data=x), OMEGA, 2).download(), msg)


def test_refresh_of_a_non_galerkin_hierarchy_is_refused_before_writing(sp):
    levels, amg, M = host_levels("hem")
    L1 = levels[1]["A"]
    # drop the last off-diagonal entry of row 0: level 1 is no longer P^T A P's structure
    lo, hi = L1.rowptr[0], L1.rowptr[1]
    drop = lo + max(j for j in range(hi - lo) if L1.colindex[lo + j] != 0)
    keep = np.ones(L1.nnz, dtype=bool)
    keep[drop] = False
    rp = L1.rowptr.copy()
    rp[1:] -= 1
    bad = [dict(L) for L in levels]
    bad[1]["A"] = CSR(L1.nrow, L1.ncol, rp, L1.colindex[keep], L1.val[keep])
    bad[1]["diag"] = extracted_diag(bad[1]["A"])
    dH = sp.DeviceHierarchy(bad, use_graph=True)
    b = np.random.default_rng(2).standard_normal(dH.n)
    before = pcg(sp, dH, b)
    state = hierarchy_state(dH)
    with pytest.raises(sp.SparshError, match="error 2"):
        dH.refresh(shifted(levels[0]["A"], 1.0).val)
    after = pcg(sp, dH, b)
    assert before[0] == after[0]
    same_bits(after[1], before[1], "history")
    same_bits(after[2], before[2], "x")
    assert hierarchy_state(dH) == state
    amg.free()


def test_singular_refresh_marks_the_hierarchy_stale_until_a_valid_one(sp):
    levels, amg, M = host_levels("hem")
    dH = sp.DeviceHierarchy(levels, use_graph=True)
    b = np.random.default_rng(4).standard_normal(dH.n)
    pcg(sp, dH, b)
    with pytest.raises(sp.SparshError, match="error 2"):
        dH.refresh(np.zeros(levels[0]["A"].nnz))
    x = sp.DeviceVector(dH.n).fill(0.0)
    for call in (lambda: dH.pcg(sp.DeviceVector(data=b), x, 1e-9), lambda: dH.vcycle(sp.DeviceVector(data=b), x),
                 lambda: dH.amg_solve(sp.DeviceVector(data=b), x, 1e-9), lambda: dH.coarse_solve(sp.DeviceVector(10))):
        with pytest.raises(sp.SparshError, match="error 2"):
            call()
    A0 = shifted(levels[0]["A"], 0.75)
    dH.refresh(A0.val)
    fresh = sp.DeviceHierarchy(galerkin_levels(sp, A0, extracted_diag(A0), levels), use_graph=True)
    assert_same_hierarchy(sp, dH, fresh, len(levels), "after the stale state")
    amg.free()

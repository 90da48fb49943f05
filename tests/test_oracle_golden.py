"""CPU tests: the C restatement (oracle/sparsh_oracle.c) against the golden vectors produced by the reference itself
(tests/golden/make_golden.py), and — when the prebuilt oracle/_ref library is present — against the reference live."""
import hashlib
import os

import numpy as np
import pytest
from conftest import system_by_name
from oracle_bindings import CSR, OracleAmg, OracleOps, Ref, RefAmg, have_ref, primitive_outputs

CASES = ["fixture", "poisson3d_24_ones", "poisson3d_24_axstar", "poisson2d_96_ones", "poisson2d_96_axstar"]
RTOL_HIST = 1e-10  # north_star: V-cycle / PCG residual histories within 1e-10 relative


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def assert_hist(got, want, rtol=RTOL_HIST):
    got, want = np.asarray(got), np.asarray(want)
    assert abs(len(got) - len(want)) <= 1, (len(got), len(want))  # north_star: same iteration count (+-1)
    m = min(len(got), len(want))
    np.testing.assert_allclose(got[:m], want[:m], rtol=rtol, atol=0)


@pytest.mark.parametrize("case", CASES + ["poisson3d_40_ones"])
@pytest.mark.parametrize("coarsening", ["hem", "beck"])
def test_hierarchy_matches_reference(case, coarsening, oracle, fixture_system, golden):
    A, b = system_by_name(case, oracle, fixture_system)
    amg = OracleAmg(A, coarsening=0 if coarsening == "hem" else 1)
    H = amg.hierarchy()
    want = golden[case][coarsening]["levels"]
    assert H.nlevels == len(want)
    for L, w in zip(H.levels, want):
        assert (L["A"].nrow, L["A"].nnz) == (w["nrow"], w["nnz"])
        # integer data bit-exact
        assert sha(L["A"].rowptr) == w["rowptr_sha"]
        assert sha(L["A"].colindex) == w["colindex_sha"]
        np.testing.assert_allclose(np.sum(L["A"].val), w["val_sum"], rtol=1e-12, atol=1e-9)
        np.testing.assert_allclose(np.sum(np.abs(L["A"].val)), w["val_abs_sum"], rtol=1e-12)
        np.testing.assert_allclose(np.sum(L["diag"]), w["diag_sum"], rtol=1e-12)
        if L["P"] is not None:
            assert (L["P"].ncol, L["P"].nnz) == (w["p_ncol"], w["p_nnz"])
            assert sha(L["P"].rowptr) == w["p_rowptr_sha"]
            assert sha(L["P"].colindex) == w["p_colindex_sha"]


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("coarsening", ["hem", "beck"])
def test_amg_solve_history(case, coarsening, oracle, fixture_system, golden):
    A, b = system_by_name(case, oracle, fixture_system)
    amg = OracleAmg(A, coarsening=0 if coarsening == "hem" else 1)
    x, hist = amg.solve(b, np.zeros(A.nrow), 1e-8)
    assert_hist(hist[1:], golden[case][coarsening]["amg_solve_hist"])
    np.testing.assert_allclose(np.sum(x), golden[case][coarsening]["amg_solve_x_sum"], rtol=1e-9)


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("coarsening", ["hem", "beck"])
def test_vcycle_probe_and_pcg(case, coarsening, oracle, fixture_system, golden):
    A, b = system_by_name(case, oracle, fixture_system)
    g = golden[case][coarsening]
    amg = OracleAmg(A, coarsening=0 if coarsening == "hem" else 1)
    xr = np.random.default_rng(g["vcycle_probe"]["seed"]).random(A.nrow)
    x1 = amg.vcycle(b, xr, 1)
    np.testing.assert_allclose(x1[:8], g["vcycle_probe"]["x_head"], rtol=1e-12)
    np.testing.assert_allclose(np.linalg.norm(x1), g["vcycle_probe"]["x_norm"], rtol=1e-12)
    x, hist = amg.pcg(b, np.zeros(A.nrow), 1e-8)
    assert_hist(hist, g["pcg_hist"])


@pytest.mark.parametrize("case", CASES)
def test_shipped_entry_points(case, oracle, fixture_system, golden):
    """AMG_Solver_CPU_baseline / Solver_PCG_1 / Solver_PBiCG_1 exactly as shipped (HEM)."""
    A, b = system_by_name(case, oracle, fixture_system)
    g = golden[case]
    amg = OracleAmg(A)
    x0 = np.zeros(A.nrow)
    _, h = amg.solve(b, x0, 1e-8)
    assert_hist(h[1:], g["AMG_Solver_CPU_baseline"]["hist"])
    _, h = amg.pcg(b, x0, 1e-8)
    assert_hist(h[1:], g["Solver_PCG_1"]["hist"])
    _, h = amg.pbicgstab(b, x0, 1e-8)
    assert_hist(h[1:], g["Solver_PBiCG_1"]["hist"])


def test_fixture_headline_counts(golden):
    """SURVEY Appendix C / BASELINE.md §5: 30 cycles, 13 PCG its, 7 PBiCGStab its (HEM); 18 / 10 (Beck)."""
    f = golden["fixture"]
    assert len(f["AMG_Solver_CPU_baseline"]["hist"]) == 30
    assert len(f["Solver_PCG_1"]["hist"]) == 13
    assert len(f["Solver_PBiCG_1"]["hist"]) == 7
    assert len(f["beck"]["amg_solve_hist"]) == 18
    assert len(f["beck"]["pcg_hist"]) - 1 == 10
    assert abs(f["AMG_Solver_CPU_baseline"]["hist"][0] - 0.35307) < 1e-5


def test_unpreconditioned_krylov(oracle, fixture_system, golden):
    A, b = fixture_system
    n = A.nrow
    from oracle_bindings import dp, ip

    for fn, key in [(oracle.lib.so_cg, "Solver_CG_1"), (oracle.lib.so_bicgstab, "Solver_BiCG_1")]:
        x = np.zeros(n)
        hist = np.zeros(2001)
        k = fn(n, ip(A.rowptr), ip(A.colindex), dp(A.val), dp(b), dp(x), 1e-8, 2000, dp(hist))
        g = golden["fixture"][key]
        # long unpreconditioned recurrences amplify rounding: count within 1%, first residuals tight
        assert abs(k - g["iters"]) <= max(1, g["iters"] // 100)
        np.testing.assert_allclose(hist[1:6], g["head"], rtol=1e-9)


def test_coloring_and_sor(oracle, fixture_system, golden):
    A, b = fixture_system
    g = golden["fixture"]["coloring"]
    nc, perm, cc, Q = oracle.color_reorder(A)
    assert nc == g["total_colors"]
    assert cc.tolist() == g["color_count"]
    assert sha(perm) == g["perm_sha"]  # integer permutation bit-exact
    assert sha(Q.rowptr) == g["q_rowptr_sha"] and sha(Q.colindex) == g["q_colindex_sha"]
    xs = oracle.sor_multicolor(Q, Q.diagonal(), cc, b[perm], np.zeros(A.nrow), 0.66667, 3)
    np.testing.assert_allclose(xs[:8], golden["fixture"]["sor_probe"]["x_head"], rtol=1e-12)
    np.testing.assert_allclose(np.linalg.norm(xs), golden["fixture"]["sor_probe"]["x_norm"], rtol=1e-12)


def test_direct_solver_accuracy(oracle):
    A = oracle.gen_poisson3d(14, 14, 14)
    xs = np.random.default_rng(3).random(A.nrow)
    b = A.to_scipy() @ xs
    x = oracle.lu_solve(A, b)
    np.testing.assert_allclose(x, xs, rtol=1e-11)


def test_edge_cases(oracle):
    # 1x1, diagonal-only, and a ragged matrix with an empty row
    A = CSR(1, 1, [0, 1], [0], [2.0])
    assert oracle.spmv(A, np.array([3.0]))[0] == 6.0
    A = CSR(3, 3, [0, 2, 2, 3], [0, 2, 2], [1.0, 2.0, 4.0])
    np.testing.assert_array_equal(oracle.spmv(A, np.array([1.0, 5.0, 2.0])), [5.0, 0.0, 8.0])
    P = CSR(3, 2, [0, 1, 2, 3], [0, 0, 1], [1.0, 1.0, 1.0])
    np.testing.assert_array_equal(oracle.transfer_residual(P, np.array([1.0, 2.0, 4.0])), [3.0, 4.0])
    np.testing.assert_array_equal(oracle.transfer_solution(P, np.array([10.0, 20.0]), np.array([1.0, 1.0, 1.0])),
                                  [11.0, 11.0, 21.0])


PRIMITIVE_TOL = {"spmv": (1e-12, 1e-14), "jacobi": (1e-12, 0), "store_residual": (1e-12, 1e-14),
                 "residual": (1e-12, 0), "transfer_residual": (1e-12, 0), "transfer_solution": (1e-12, 0),
                 "coarse_solve": (1e-10, 0)}  # (rtol, atol)


def assert_primitives(got, want, rows=None):
    assert set(got) == set(want)
    for key, w in want.items():
        rtol, atol = PRIMITIVE_TOL[key.split("/")[-1]]
        g = got[key] if rows is None else got[key][rows[key]]
        np.testing.assert_allclose(g, w, rtol=rtol, atol=atol, err_msg=key)


@pytest.mark.parametrize("coarsening", [0, 1])
def test_primitives_against_live_reference(coarsening, oracle, fixture_system):
    """Per-op parity (1e-12) of the restatement on every level: against the per-op outputs stored by
    tests/golden/make_primitives.py (a fixed sample of rows of each output), and, where oracle/_ref is built, against
    the reference's own primitives live."""
    A, b = fixture_system
    H = OracleAmg(A, coarsening).hierarchy()  # integers pinned to the reference's by test_hierarchy_matches_reference
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "primitives_fixture.npz"))
    prefix = f"{coarsening}:"
    want = {k[len(prefix):]: z[k] for k in z.files if k.startswith(prefix) and not k.endswith("@rows")}
    rows = {k: z[prefix + k + "@rows"] for k in want}
    assert_primitives(primitive_outputs(H, OracleOps(oracle, H)), want, rows)
    if have_ref():
        Ref.get().set_threads(4)
        ref = RefAmg(A, coarsening)
        H = ref.hierarchy()
        assert_primitives(primitive_outputs(H, OracleOps(oracle, H)), primitive_outputs(H, ref))


def test_sor_vcycle_solver_matches_reference(oracle, fixture_system, golden):
    """AMG_Solver_2 (multicolour-SOR V-cycles): the restatement reproduces the reference's 28 cycles and its history,
    and — unlike the reference, which never copies x back (SURVEY Appendix B) — really returns the solution."""
    A, b = fixture_system
    g = golden["fixture"]["AMG_Solver_2"]
    amg = OracleAmg(A, sor=True)
    x, hist = amg.solve_sor(b, np.zeros(A.nrow), 1e-8)
    assert len(hist) - 1 == g["cycles"] == 28
    np.testing.assert_allclose(hist[1:], g["hist"], rtol=1e-10)
    assert np.linalg.norm(b - A.to_scipy() @ x) <= 1e-8


def test_gmres_restatement_against_scipy(oracle, fixture_system):
    """GMRES(m) is not in the reference (F3); the oracle's statement of it is pinned to scipy's on a nonsymmetric
    matrix (inner-iteration residual estimates), to the minimal-residual property, and to restart behaviour."""
    import scipy.sparse as sps
    import scipy.sparse.linalg as spla

    rng = np.random.default_rng(11)
    n = 300
    S = sps.diags([-1.3, 2.6, -0.7], [-1, 0, 1], shape=(n, n)) + sps.random(n, n, density=0.01, random_state=3) * 0.2
    S = S.tocsr()
    S.sort_indices()
    A = CSR(n, n, S.indptr, S.indices, S.data)
    b = rng.standard_normal(n)
    tol = 1e-9 * np.linalg.norm(b)
    # full GMRES (restart >= iterations): estimates equal scipy's per-iteration preconditioned-residual norms
    seen = []
    xs, info = spla.gmres(S, b, x0=np.zeros(n), rtol=1e-9, atol=0.0, restart=200, maxiter=1,
                          callback=lambda r: seen.append(r), callback_type="pr_norm")
    assert info == 0
    x, hist = oracle.gmres(A, b, np.zeros(n), tol, restart=200, max_iter=200)
    k = len(hist) - 1
    assert k == len(seen)
    np.testing.assert_allclose(hist[1:k] / hist[0], seen[: k - 1], rtol=1e-8)  # scipy reports relative norms
    assert np.linalg.norm(b - S @ x) <= tol * (1 + 1e-6) and hist[-1] == pytest.approx(np.linalg.norm(b - S @ x), rel=1e-6)
    # minimal residual over the Krylov space after 7 iterations
    x7, h7 = oracle.gmres(A, b, np.zeros(n), 0.0, restart=50, max_iter=7)
    K = np.zeros((n, 7))
    K[:, 0] = b
    for j in range(1, 7):
        K[:, j] = S @ K[:, j - 1]
    Q, _ = np.linalg.qr(K)
    c = np.linalg.lstsq(S @ Q, b, rcond=None)[0]
    assert h7[-1] == pytest.approx(np.linalg.norm(b - S @ (Q @ c)), rel=1e-9)
    # restarts: still converges, needs at least as many iterations, monotone within a cycle
    xr, hr = oracle.gmres(A, b, np.zeros(n), tol, restart=10, max_iter=2000)
    assert len(hr) >= len(hist) and np.linalg.norm(b - S @ xr) <= tol * (1 + 1e-6)
    assert all(hr[i + 1] <= hr[i] * (1 + 1e-12) for i in range(9))
    # V-cycle as right preconditioner on the bundled SPD system: far fewer iterations than without
    F, fb = fixture_system
    amg = OracleAmg(F)
    xp, hp = amg.pgmres(fb, np.zeros(F.nrow), 1e-8, restart=30)
    assert np.linalg.norm(fb - F.to_scipy() @ xp) <= 1e-8 * (1 + 1e-6)
    _, hpcg = amg.pcg(fb, np.zeros(F.nrow), 1e-8)
    assert len(hp) - 1 <= len(hpcg) - 1 + 2  # GMRES minimises the residual: no worse than PCG (+restart slack)


def test_oracle_pcg_128_matches_the_reference_solver(oracle):
    """the C restatement against the reference's stock Solver_PCG_1 at 128^3 (2.1M rows, 11 levels): iteration count and
    residual history frozen by tools/pin_reference_pcg.py (the 256^3 twin of this golden gates the GPU path at full size)"""
    import json
    import os

    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "pcg_poisson3d_128_ref.json")))
    A = oracle.gen_poisson3d(128, 128, 128)
    assert (A.nrow, A.nnz) == (g["rows"], g["nnz"])
    b = np.ones(A.nrow)
    _, hist = OracleAmg(A).pcg(b, np.zeros(A.nrow), g["tol_abs"])
    assert len(hist) - 1 == g["iterations"]
    np.testing.assert_allclose(hist[0], g["initial_residual"], rtol=1e-15)
    np.testing.assert_allclose(hist[1:], g["history_after_iteration"], rtol=1e-10, atol=1e-13 * hist[0])

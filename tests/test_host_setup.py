"""CPU tests of the product's host side: the C-ABI library loads and exports every symbol include/sparsh_b200.h
declares (no compute without a GPU), and the native setup phase (HEM / Beck / Galerkin / colouring) reproduces the
reference's hierarchy — integer data bit-exact, coarse values to rounding."""
import hashlib
import os
import re

import numpy as np
import pytest
from conftest import ROOT, system_by_name
from oracle_bindings import OracleAmg


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def test_cabi_exports_every_declared_symbol():
    import sparsh_amg_b200 as sp

    header = open(os.path.join(ROOT, "include", "sparsh_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(sparsh_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 45
    lib = sp.capi.load()
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/sparsh_b200.h but not exported"
    assert declared == set(sp.capi.SIGNATURES), declared ^ set(sp.capi.SIGNATURES)


def test_no_cpu_fallback_without_gpu():
    """On a box without a GPU the product must fail loudly, never compute on the CPU."""
    import sparsh_amg_b200 as sp

    try:
        import torch

        if torch.cuda.is_available():
            pytest.skip("GPU present")
    except ImportError:
        pass
    with pytest.raises(sp.SparshError):
        sp.init(0)
    with pytest.raises(sp.SparshError):
        sp.DeviceVector(data=np.ones(4))


def test_product_does_not_touch_the_oracle():
    """Only tests/, smoke() and bench.py may reach oracle/ — the package sources must not mention it."""
    pkg = os.path.join(ROOT, "sparsh_amg_b200")
    for dirpath, _, files in os.walk(pkg):
        if os.sep + "build" in dirpath or dirpath.endswith("lib"):
            continue
        for f in files:
            if f.endswith((".py", ".cpp", ".cu", ".cuh", ".hpp", ".h", "Makefile")):
                text = open(os.path.join(dirpath, f), errors="replace").read()
                assert "sparsh_oracle" not in text and "oracle/" not in text and "libsparsh_ref" not in text, f


@pytest.fixture(scope="module")
def host():
    from sparsh_amg_b200 import host as h

    h.set_options(threads=min(8, os.cpu_count() or 1), max_levels=32, print_setup=0, print_solve=0)
    return h


CASES = ["fixture", "poisson3d_24_ones", "poisson2d_96_ones", "poisson3d_40_ones"]


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("coarsening", ["hem", "beck"])
def test_native_setup_matches_reference_hierarchy(host, oracle, fixture_system, golden, case, coarsening):
    A, b = system_by_name(case, oracle, fixture_system)
    host.set_options(coarsening=0 if coarsening == "hem" else 1)
    M = host.HostMatrix.from_csr(A)
    amg = host.HostAmg(M)
    levels = amg.levels()
    want = golden[case][coarsening]["levels"]
    ref_levels = OracleAmg(A, coarsening=0 if coarsening == "hem" else 1).hierarchy().levels
    assert len(levels) == len(want)
    for L, w, R in zip(levels, want, ref_levels):
        assert (L["A"].nrow, L["A"].nnz) == (w["nrow"], w["nnz"])
        assert sha(L["A"].rowptr) == w["rowptr_sha"]          # integer data bit-exact vs the reference run
        assert sha(L["A"].colindex) == w["colindex_sha"]
        np.testing.assert_allclose(L["A"].val, R["A"].val, rtol=1e-13, atol=1e-13)
        np.testing.assert_allclose(L["diag"], R["diag"], rtol=1e-13)
        np.testing.assert_allclose(np.sum(L["A"].val), w["val_sum"], rtol=1e-12, atol=1e-9)
        if L["P"] is not None:
            assert (L["P"].ncol, L["P"].nnz) == (w["p_ncol"], w["p_nnz"])
            assert sha(L["P"].rowptr) == w["p_rowptr_sha"]
            assert sha(L["P"].colindex) == w["p_colindex_sha"]
            np.testing.assert_array_equal(L["P"].val, R["P"].val)
    amg.free()
    M.free()
    host.set_options(coarsening=0)


def test_native_colouring_matches_reference(host, fixture_system, golden, oracle):
    A, b = fixture_system
    M = host.HostMatrix.from_csr(A)
    nc, perm, cc = M.color_reorder()
    g = golden["fixture"]["coloring"]
    assert nc == g["total_colors"] and cc.tolist() == g["color_count"]
    assert sha(perm) == g["perm_sha"]
    assert sha(M.rowptr) == g["q_rowptr_sha"] and sha(M.colindex) == g["q_colindex_sha"]
    np.testing.assert_allclose(np.sum(M.val), g["q_val_sum"], rtol=1e-13)
    M.free()


def test_generators_match_oracle_generators(host, oracle):
    for (nx, ny, nz) in [(7, 5, 3), (16, 16, 16), (1, 1, 1)]:
        M = host.HostMatrix.poisson3d(nx, ny, nz)
        O = oracle.gen_poisson3d(nx, ny, nz)
        assert np.array_equal(M.rowptr, O.rowptr) and np.array_equal(M.colindex, O.colindex)
        assert np.array_equal(M.val, O.val)
        M.free()
    M = host.HostMatrix.poisson2d(33, 17)
    O = oracle.gen_poisson2d(33, 17)
    assert np.array_equal(M.rowptr, O.rowptr) and np.array_equal(M.colindex, O.colindex) and np.array_equal(M.val, O.val)
    # SURVEY §8d nnz formulas: 2D 5n - 2(nx+ny), 3D 7n - 2(nx ny + ny nz + nx nz), 27-pt (3n-2)^3 for a cube
    assert M.nnz == 5 * 33 * 17 - 2 * (33 + 17)
    M.free()
    D = host.HostMatrix.diffusion27(6, 6, 6)
    assert D.nnz == (3 * 6 - 2) ** 3
    S = D  # SPD-like checks: symmetric, positive diagonal, zero row sums only away from the Dirichlet boundary
    import scipy.sparse as sps

    T = sps.csr_matrix((S.val, S.colindex, S.rowptr), shape=(S.nrow, S.ncol))
    assert abs(T - T.T).max() < 1e-12 * abs(T).max()
    assert np.all(T.diagonal() > 0)
    w = np.linalg.eigvalsh(T.toarray())
    assert w.min() > 0
    D.free()


def test_reader_roundtrip(host, tmp_path, fixture_system):
    A, b = fixture_system
    n = 200  # leading principal block of the bundled matrix, written in the reference's two-file format
    rp = A.rowptr[: n + 1]
    keep = [(i, A.colindex[j], A.val[j]) for i in range(n) for j in range(rp[i], rp[i + 1]) if A.colindex[j] < n]
    mf, rf = tmp_path / "m.txt", tmp_path / "rhs.txt"
    with open(mf, "w") as f:
        f.write(f"{n} {n} {len(keep)}\n")
        for i, c, v in keep:
            f.write(f"{i}\t{int(c)}\t{float(v)!r}\t\n")
    with open(rf, "w") as f:
        f.write(f"{n}\n" + "\n".join(repr(float(x)) for x in b[:n]) + "\n")
    M, bb = host.HostMatrix.read(str(mf), str(rf))
    assert (M.nrow, M.nnz) == (n, len(keep))
    np.testing.assert_array_equal(bb, b[:n])
    np.testing.assert_array_equal(M.val, [v for _, _, v in keep])
    M.free()


def test_matrix_market_reader(host, tmp_path, fixture_system):
    """standard MatrixMarket files (1-based, unsorted, general and symmetric) — SURVEY §8f.3"""
    import scipy.io
    import scipy.sparse as sps

    A, _ = fixture_system
    S = A.to_scipy()[:300, :300].tocsr()
    S.eliminate_zeros()
    S = ((S + S.T) * 0.5).tocsr()  # exactly symmetric so that the symmetric writer keeps one triangle
    S.sort_indices()
    rng = np.random.default_rng(0)
    for sym in ("general", "symmetric"):
        path = tmp_path / f"m_{sym}.mtx"
        coo = S.tocoo()
        perm = rng.permutation(coo.nnz)  # entries in random order
        scipy.io.mmwrite(str(path), sps.coo_matrix((coo.data[perm], (coo.row[perm], coo.col[perm])), shape=S.shape),
                         symmetry=sym, precision=17)
        M = host.HostMatrix.read_matrix_market(str(path))
        assert (M.nrow, M.ncol, M.nnz) == (300, 300, S.nnz)
        np.testing.assert_array_equal(M.rowptr, S.indptr)
        np.testing.assert_array_equal(M.colindex, S.indices)
        np.testing.assert_allclose(M.val, S.data, rtol=1e-15)
        M.free()
    with open(tmp_path / "bad.mtx", "w") as f:
        f.write("not a matrix\n")
    with pytest.raises(Exception):
        host.HostMatrix.read_matrix_market(str(tmp_path / "bad.mtx"))


def test_shared_hierarchy_roundtrip_and_plans(host, oracle, tmp_path):
    """rank 0 saves, every rank maps read-only (host/share.cpp): identical levels and identical partition plans"""
    from sparsh_amg_b200.distributed import DistPlan

    host.set_options(coarse_upper=500, coarse_lower=250)
    A = host.HostMatrix.poisson3d(18, 16, 20)
    amg = host.HostAmg(A)
    d = str(tmp_path / "hier")
    amg.save(d)
    # the loaded object sizes its per-level arrays from the file, whatever max_levels says at that moment (a solver
    # constructed under a smaller max_levels used to overrun them), and leaves the global option alone
    assert amg.nlevels > 2
    host.set_options(max_levels=2)
    shared = host.HostAmg.load(d)
    two = host.HostAmg(A)
    assert two.nlevels == 2  # max_levels = 2 still governs a fresh setup
    two.free()
    host.set_options(max_levels=32)
    assert shared.nlevels == amg.nlevels
    for L0, L1 in zip(amg.levels(), shared.levels()):
        for key in ("rowptr", "colindex", "val"):
            np.testing.assert_array_equal(getattr(L0["A"], key), getattr(L1["A"], key))
            if L0["P"] is not None:
                np.testing.assert_array_equal(getattr(L0["P"], key), getattr(L1["P"], key))
        np.testing.assert_array_equal(L0["diag"], L1["diag"])
    for rank in range(3):
        p0, p1 = DistPlan(amg, 3, rank, tail_threshold=700), DistPlan(shared, 3, rank, tail_threshold=700)
        assert (p0.nd, p0.nlevels) == (p1.nd, p1.nlevels)
        for l in range(p0.nd):
            np.testing.assert_array_equal(p0.rows(l), p1.rows(l))
            for which in "APR":
                a, b = p0.op(l, which), p1.op(l, which)
                for key in ("rowptr", "colindex", "val", "send_idx", "send_rank", "recv_rank", "recv_ptr", "halo_global"):
                    np.testing.assert_array_equal(a[key], b[key])
                assert a["interior"] == b["interior"]
        p0.free()
        p1.free()
    shared.free()
    amg.free()
    A.free()
    host.set_options(coarse_upper=4000, coarse_lower=2000)


def _dict_encode(A):
    import ctypes as C
    import sparsh_amg_b200 as sp

    lib = sp.capi.load()
    code = np.zeros(max(A.nnz, 1), dtype=np.uint16)
    dval, doff = np.zeros(256), np.zeros(256, dtype=np.int32)
    nv, no = C.c_int(-1), C.c_int(-1)
    rc = lib.sparsh_dict_encode(A.nrow, A.ncol, A.nnz, sp.capi.ip(A.rowptr), sp.capi.ip(A.colindex), sp.capi.dp(A.val),
                                code.ctypes.data_as(C.c_void_p), sp.capi.dp(dval), sp.capi.ip(doff), C.byref(nv),
                                C.byref(no))
    assert rc == 0
    return code, dval[: nv.value], doff[: no.value]


def test_csr_dict16_encoding_is_lossless(host, fixture_system):
    """The csr-dict16 twin the stream kernel runs on must decode to exactly the CSR it came from (values by bit
    pattern), and must decline matrices whose dictionaries do not fit (they stay plain CSR)."""
    import sparsh_amg_b200 as sp
    from sparsh_amg_b200.generators import HostCSR, poisson_7pt

    # constant-coefficient stencil and its Galerkin coarse operators
    A = poisson_7pt(40, 36, 32)
    amg = host.HostAmg(host.HostMatrix.from_csr(A))
    assert amg.nlevels >= 3
    representable = 0
    for k, lev in enumerate(amg.levels()):
        M = lev["A"]
        code, dval, doff = _dict_encode(M)
        if k == 0:
            assert len(dval) == 2 and len(doff) == 7
        if len(dval) == 0:
            continue
        representable += 1
        rows = np.repeat(np.arange(M.nrow, dtype=np.int64), np.diff(M.rowptr))
        assert np.array_equal(dval[code >> 8].view(np.uint64), np.ascontiguousarray(M.val).view(np.uint64))
        assert np.array_equal(rows + doff[code & 255], M.colindex)
    assert representable >= 2
    # large enough for the multi-threaded scan: dictionaries still come out in order of first appearance
    B = poisson_7pt(70, 64, 60)
    code, dval, doff = _dict_encode(B)
    rows = np.repeat(np.arange(B.nrow, dtype=np.int64), np.diff(B.rowptr))
    for got, seq in ((dval, B.val), (doff, B.colindex - rows)):
        _, first = np.unique(seq, return_index=True)
        np.testing.assert_array_equal(got, seq[np.sort(first)])
    assert np.array_equal(dval[code >> 8], B.val) and np.array_equal(rows + doff[code & 255], B.colindex)
    # -0.0 and 0.0 are different dictionary entries (bit pattern, not ==)
    Z = HostCSR(2, 2, [0, 1, 2], [0, 1], [0.0, -0.0])
    code, dval, _ = _dict_encode(Z)
    assert len(dval) == 2 and np.signbit(dval[code[1] >> 8]) and not np.signbit(dval[code[0] >> 8])
    # more than 256 distinct values (the unstructured fixture) or offsets: not representable
    F, _ = fixture_system
    assert len(_dict_encode(F)[1]) == 0
    n = 300
    W = HostCSR(1, n, [0, n], np.arange(n), np.ones(n))
    assert len(_dict_encode(W)[1]) == 0


def _pattern_encode(A, diag=None):
    import ctypes as C
    import sparsh_amg_b200 as sp

    lib = sp.capi.load()
    pat = np.full(max(A.nrow, 1), 7, dtype=np.uint8)
    ent_val, ent_off = np.zeros(2048), np.zeros(2048, dtype=np.int32)
    start = np.zeros(256, dtype=np.int32)
    n_pat, n_esc = C.c_int(-1), C.c_int(-1)
    rc = lib.sparsh_pattern_encode(A.nrow, A.ncol, A.nnz, sp.capi.ip(A.rowptr), sp.capi.ip(A.colindex),
                                   sp.capi.dp(A.val), None if diag is None else sp.capi.dp(diag),
                                   pat.ctypes.data_as(C.c_void_p), sp.capi.dp(ent_val), sp.capi.ip(ent_off),
                                   sp.capi.ip(start), C.byref(n_pat), C.byref(n_esc))
    assert rc == 0
    return pat, ent_val, ent_off, start[: n_pat.value + 1], n_pat.value, n_esc.value


def _check_pattern_decode(M, pat, ent_val, ent_off, start, n_pat, n_esc):
    """every tabulated row must decode to exactly its CSR row (order, columns, value bits)"""
    rp = M.rowptr.astype(np.int64)
    assert np.count_nonzero(pat == 255) == n_esc
    assert pat[pat != 255].max(initial=0) < n_pat
    counts = np.bincount(pat[pat != 255], minlength=n_pat)
    assert np.all(np.diff(counts) <= 0)  # numbered by decreasing row count
    vbits = np.ascontiguousarray(M.val).view(np.uint64)
    for p in range(n_pat):
        rows = np.flatnonzero(pat == p)
        assert len(rows) > 0
        ln = start[p + 1] - start[p]
        assert np.all(np.diff(M.rowptr)[rows] == ln)
        idx = rp[rows][:, None] + np.arange(ln)[None, :]
        assert np.array_equal(M.colindex[idx], rows[:, None] + ent_off[start[p]: start[p + 1]][None, :])
        want = np.broadcast_to(ent_val[start[p]: start[p + 1]].view(np.uint64)[None, :], idx.shape)
        assert np.array_equal(vbits[idx], want)


def test_csr_pattern8_encoding_is_lossless(host, fixture_system):
    """csr-pattern8 (one byte per row): tabulated rows decode to exactly their CSR rows; rows that do not repeat, or
    whose smoothing diagonal differs from the tabulated one, are escapes served from the CSR arrays."""
    from sparsh_amg_b200.generators import HostCSR, poisson_7pt

    A = poisson_7pt(40, 36, 32)
    amg = host.HostAmg(host.HostMatrix.from_csr(A))
    for k, lev in enumerate(amg.levels()):
        M = lev["A"]
        enc = _pattern_encode(M, np.ascontiguousarray(lev["diag"]))
        _check_pattern_decode(M, *enc)
        assert enc[4] == 27 and enc[5] == 0  # 3 x 3 x 3 boundary classes at every level, nothing escapes
    # a caller-supplied diagonal that differs on some rows: exactly those rows escape
    d = np.full(A.nrow, 6.0)
    d[[5, 77, 1234]] = 6.5
    pat, *_rest, n_esc = _pattern_encode(A, d)
    assert n_esc == 3 and set(np.flatnonzero(pat == 255)) == {5, 77, 1234}
    # a row longer than 64 entries and a unique row are escapes; the repeated rows are tabulated
    n = 200
    rp = np.arange(n + 1, dtype=np.int32) * 2
    ci = np.stack([np.arange(n), (np.arange(n) + 1) % n], axis=1).astype(np.int32)
    ci.sort(axis=1)
    v = np.tile([2.0, -1.0], n)
    W = HostCSR(n, n, rp, ci.ravel(), v)
    enc = _pattern_encode(W)
    _check_pattern_decode(W, *enc)
    assert enc[4] == 2 and enc[5] == 0  # the wrap-around row (sorted columns: offsets 0 - (n-1), 0) is its own pattern
    # unstructured matrix: whatever is tabulated still decodes, but almost nothing repeats (the library keeps CSR)
    F, _ = fixture_system
    enc = _pattern_encode(F)
    _check_pattern_decode(F, *enc)
    assert enc[5] > 0.25 * F.nrow


def test_binary_csr_roundtrip(host, tmp_path, fixture_system):
    """SURVEY §8f.3: binary CSR written and read back bit for bit; damaged files are refused"""
    A, _ = fixture_system
    M = host.HostMatrix.from_csr(A)
    path = str(tmp_path / "a.csr")
    M.write_binary(path)
    B = host.HostMatrix.read_binary(path)
    assert (B.nrow, B.ncol) == (A.nrow, A.ncol)
    np.testing.assert_array_equal(B.rowptr, M.rowptr)
    np.testing.assert_array_equal(B.colindex, M.colindex)
    np.testing.assert_array_equal(B.val.view(np.uint64), M.val.view(np.uint64))
    raw = open(path, "rb").read()
    assert raw[:8] == b"SPRSHCSR" and len(raw) == 8 + 4 * 3 + 8 + 4 * (A.nrow + 1) + 12 * A.nnz
    for name, data in [("trunc", raw[:-16]), ("magic", b"XXXXXXXX" + raw[8:]),
                       ("col", raw[:28 + 4 * (A.nrow + 1)] + (10 ** 9).to_bytes(4, "little") + raw[32 + 4 * (A.nrow + 1):])]:
        bad = str(tmp_path / name)
        open(bad, "wb").write(data)
        with pytest.raises(Exception):
            host.HostMatrix.read_binary(bad)
    with pytest.raises(Exception):
        host.HostMatrix.read_binary(str(tmp_path / "missing"))
    B.free()
    M.free()


def _sa_restatement(A, level, theta=0.08, relax=4.0 / 3.0):
    """plain-Python restatement of smoothed aggregation as documented in host/setup.cpp (SA_Prolongator)"""
    n, rp, ci, v = A.nrow, A.rowptr, A.colindex, A.val
    dabs = np.zeros(n)
    for i in range(n):
        for j in range(rp[i], rp[i + 1]):
            if ci[j] == i:
                dabs[i] = abs(v[j])
                break
    th = theta * 0.5 ** level
    strong = np.zeros(len(ci), dtype=bool)
    for i in range(n):
        for j in range(rp[i], rp[i + 1]):
            strong[j] = ci[j] != i and v[j] != 0.0 and abs(v[j]) >= th * np.sqrt(dabs[i] * dabs[ci[j]])
    agg = -np.ones(n, dtype=np.int64)
    nagg = 0
    for i in range(n):
        if agg[i] != -1:
            continue
        nb = [ci[j] for j in range(rp[i], rp[i + 1]) if strong[j]]
        if nb and all(agg[c] == -1 for c in nb):
            agg[i] = nagg
            agg[nb] = nagg
            nagg += 1
    snap = agg.copy()
    for i in range(n):
        if snap[i] != -1:
            continue
        best, to = 0.0, -1
        for j in range(rp[i], rp[i + 1]):
            if strong[j] and snap[ci[j]] != -1 and abs(v[j]) > best:
                best, to = abs(v[j]), snap[ci[j]]
        if to != -1:
            agg[i] = to
    for i in range(n):
        if agg[i] != -1:
            continue
        agg[i] = nagg
        for j in range(rp[i], rp[i + 1]):
            if strong[j] and agg[ci[j]] == -1:
                agg[ci[j]] = nagg
        nagg += 1
    dF, rho = np.zeros(n), 0.0
    for i in range(n):
        off = 0.0
        for j in range(rp[i], rp[i + 1]):
            if ci[j] == i or not strong[j]:
                dF[i] += v[j]
            else:
                off += abs(v[j])
        if dF[i] != 0.0:
            rho = max(rho, (abs(dF[i]) + off) / abs(dF[i]))
    omega = relax / rho
    P = np.zeros((n, nagg))
    for i in range(n):
        P[i, agg[i]] += 1.0
        if dF[i] != 0.0:
            P[i, agg[i]] -= omega
            for j in range(rp[i], rp[i + 1]):
                if strong[j]:
                    P[i, agg[ci[j]]] -= omega / dF[i] * v[j]
    return agg, P


@pytest.mark.parametrize("case", ["poisson2d", "poisson3d", "aniso27", "fixture_head"])
def test_smoothed_aggregation_setup(host, oracle, fixture_system, case):
    """SURVEY §8f.2 (absent from the reference, F2): the native smoothed-aggregation setup equals its plain-Python
    restatement (aggregates exactly, P to rounding), reproduces constants where A annihilates them, and its hierarchy
    converges in fewer AMG-PCG iterations than the shipped unsmoothed pairwise aggregation."""
    from sparsh_amg_b200.generators import HostCSR

    if case == "poisson2d":
        M = host.HostMatrix.poisson2d(14, 11)
    elif case == "poisson3d":
        M = host.HostMatrix.poisson3d(7, 6, 5)
    elif case == "aniso27":
        M = host.HostMatrix.diffusion27(6, 5, 4)
    else:  # leading principal block of the unstructured FE matrix
        F, _ = fixture_system
        S = F.to_scipy().tocsr()[:400, :400].tocsr()
        S.sort_indices()
        M = host.HostMatrix.from_csr(HostCSR(400, 400, S.indptr, S.indices, S.data))
    host.set_options(coarsening=2, coarse_upper=20, coarse_lower=1, max_levels=2, print_setup=0)
    try:
        amg = host.HostAmg(M)
        assert amg.nlevels == 2
        L0 = amg.levels()[0]
        P = L0["P"]
        agg, Pref = _sa_restatement(L0["A"], 0)
        assert P.ncol == Pref.shape[1] < M.nrow / 2
        dense = np.zeros_like(Pref)
        rows = np.repeat(np.arange(P.nrow), np.diff(P.rowptr))
        dense[rows, P.colindex] = P.val
        np.testing.assert_allclose(dense, Pref, rtol=0, atol=1e-14)
        assert np.all(np.diff(P.colindex)[np.diff(rows) == 0] > 0)  # columns sorted within a row
        # rows of A with zero row sum and no weak couplings keep the partition of unity
        A = L0["A"]
        rs = np.add.reduceat(A.val, A.rowptr[:-1])
        inner = np.abs(rs) < 1e-12
        if inner.any() and case != "aniso27":
            np.testing.assert_allclose(dense.sum(axis=1)[inner], 1.0, atol=1e-13)
        amg.free()
    finally:
        host.set_options(coarsening=0, coarse_upper=4000, coarse_lower=2000, max_levels=6, print_setup=1)
    M.free()


def test_smoothed_aggregation_converges_faster(host, oracle):
    from oracle_bindings import CSR, Hierarchy, OracleAmg

    A = host.HostMatrix.poisson3d(32, 32, 32)
    its = {}
    for name, c in (("hem", 0), ("sa", 2)):
        host.set_options(coarsening=c, coarse_upper=500, coarse_lower=250, max_levels=32, print_setup=0)
        amg = host.HostAmg(A)
        levels = []
        for L in amg.levels():
            M, P = L["A"], L["P"]
            levels.append(dict(A=CSR(M.nrow, M.ncol, M.rowptr.copy(), M.colindex.copy(), M.val.copy()),
                               diag=np.array(L["diag"]),
                               P=None if P is None else CSR(P.nrow, P.ncol, P.rowptr.copy(), P.colindex.copy(), P.val.copy())))
        b = np.ones(A.nrow)
        _, hist = OracleAmg(hierarchy=Hierarchy(levels)).pcg(b, np.zeros(A.nrow), 1e-8 * np.linalg.norm(b))
        its[name] = (len(hist) - 1, amg.nlevels, sum(amg.level_dims(k)[1] for k in range(amg.nlevels)) / A.nnz)
        amg.free()
    host.set_options(coarsening=0, coarse_upper=4000, coarse_lower=2000, max_levels=6, print_setup=1)
    A.free()
    assert its["sa"][0] < its["hem"][0] and its["sa"][1] < its["hem"][1] and its["sa"][2] < its["hem"][2], its


def test_fused_aggregation_product_equals_the_two_general_products(host, fixture_system, monkeypatch):
    """parallel::coarsen_matrix (reference src/AMG_cycle_utilities.cpp:126-146): for a prolongator with one entry per row
    (HEM) the host setup computes P^T (A P) in one sweep over the aggregates (setup.cpp: aggregation_rap).  It must give
    the BITS of the two general row-wise products (SPARSH_RAP_GENERAL=1) on every level: same first-touch column order
    before the sort, same accumulation order, same unfused arithmetic — on the bundled FE system, on a 3D grid (forward
    and backward sweeps, singletons numbered last) and on a 2D grid."""
    F, _ = fixture_system
    mats = [host.HostMatrix.from_csr(F), host.HostMatrix.poisson3d(40, 36, 30), host.HostMatrix.poisson2d(150, 131)]
    host.set_options(coarsening=0, coarse_upper=200, coarse_lower=50, max_levels=32, print_setup=0, threads=4)
    try:
        for M in mats:
            monkeypatch.delenv("SPARSH_RAP_GENERAL", raising=False)
            fused = host.HostAmg(M)
            monkeypatch.setenv("SPARSH_RAP_GENERAL", "1")
            general = host.HostAmg(M)
            assert fused.nlevels == general.nlevels and fused.nlevels >= 4
            for Lf, Lg in zip(fused.levels(), general.levels()):
                for key in ("rowptr", "colindex", "val"):
                    a, b = np.asarray(getattr(Lf["A"], key)), np.asarray(getattr(Lg["A"], key))
                    assert a.shape == b.shape and a.tobytes() == b.tobytes(), key
                assert np.asarray(Lf["diag"]).tobytes() == np.asarray(Lg["diag"]).tobytes()
            fused.free()
            general.free()
    finally:
        monkeypatch.delenv("SPARSH_RAP_GENERAL", raising=False)
        host.set_options(coarsening=0, coarse_upper=4000, coarse_lower=2000, max_levels=6, print_setup=1)
        for M in mats:
            M.free()


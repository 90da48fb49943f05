"""ctypes bindings for the CPU checkers (TEST INFRASTRUCTURE — never imported by the product package).

* ``Oracle``  -> oracle/libsparsh_oracle.so  (plain-C restatement, oracle/sparsh_oracle.c)
* ``Ref``     -> oracle/_ref/libsparsh_ref.so (the reference's own host sources compiled unmodified against the
                 MKL shim, driven through oracle/ref_harness.cpp).  Prebuilt in the build container; it travels
                 to the GPU box with the snapshot.  /root/reference itself is never read at test time.
"""
import ctypes as C
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_SO = os.path.join(ROOT, "oracle", "libsparsh_oracle.so")
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libsparsh_ref.so")

c_int_p = C.POINTER(C.c_int)
c_dbl_p = C.POINTER(C.c_double)


def ip(a):
    assert a.dtype == np.int32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(c_int_p)


def dp(a):
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(c_dbl_p)


class CSR:
    """0-based int32/fp64 CSR, the reference's sp_matrix layout (include/AMG_matrix.hpp:6-32)."""

    def __init__(self, nrow, ncol, rowptr, colindex, val):
        self.nrow, self.ncol = int(nrow), int(ncol)
        self.rowptr = np.ascontiguousarray(rowptr, dtype=np.int32)
        self.colindex = np.ascontiguousarray(colindex, dtype=np.int32)
        self.val = np.ascontiguousarray(val, dtype=np.float64)
        self.nnz = int(self.rowptr[-1])

    def to_scipy(self):
        import scipy.sparse as sp

        return sp.csr_matrix((self.val, self.colindex, self.rowptr), shape=(self.nrow, self.ncol))

    def diagonal(self):
        d = np.zeros(self.nrow)
        Oracle.get().lib.so_fill_diagonal(self.nrow, ip(self.rowptr), ip(self.colindex), dp(self.val), dp(d))
        return d


def _take(lib, ptr, n, dtype):
    """copy n elements from a malloc'ed C array and free it"""
    ct = C.c_int if dtype == np.int32 else C.c_double
    arr = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ct)), shape=(max(int(n), 1),))[: int(n)].copy()
    lib.so_free(C.cast(ptr, C.c_void_p))
    return arr.astype(dtype, copy=False)


class Oracle:
    _inst = None

    @classmethod
    def get(cls):
        if cls._inst is None:
            cls._inst = cls()
        return cls._inst

    def __init__(self):
        if not os.path.exists(ORACLE_SO):
            raise RuntimeError(f"{ORACLE_SO} missing: run __graft_entry__.build() (or make -C oracle oracle)")
        lib = self.lib = C.CDLL(ORACLE_SO)
        lib.so_dot.restype = C.c_double
        lib.so_nrm2.restype = C.c_double
        lib.so_residual.restype = C.c_double
        lib.so_lu_factor.restype = C.c_void_p
        lib.so_lu_solve.argtypes = [C.c_void_p, c_dbl_p, c_dbl_p]
        lib.so_lu_free.argtypes = [C.c_void_p]
        lib.so_lu_bandwidth.argtypes = [C.c_void_p]
        lib.so_free.argtypes = [C.c_void_p]
        lib.so_amg_setup.restype = C.c_void_p
        lib.so_amg_from_levels.restype = C.c_void_p
        lib.so_gmres.argtypes = [C.c_void_p, C.c_int, c_int_p, c_int_p, c_dbl_p, c_dbl_p, c_dbl_p, C.c_double, C.c_int,
                                 C.c_int, c_dbl_p]
        lib.so_amg_setup_sor.restype = C.c_void_p
        lib.so_amg_solve_sor.argtypes = [C.c_void_p, c_dbl_p, c_dbl_p, C.c_double, C.c_int, c_dbl_p]
        for f in ("so_amg_free", "so_amg_nlevels"):
            getattr(lib, f).argtypes = [C.c_void_p]
        lib.so_amg_level_dims.argtypes = [C.c_void_p, C.c_int] + [c_int_p] * 4
        lib.so_amg_level_get.argtypes = [C.c_void_p, C.c_int] + [C.POINTER(C.c_void_p)] * 7
        lib.so_amg_set_smoother.argtypes = [C.c_void_p, C.c_double, C.c_int]
        lib.so_amg_vcycle.argtypes = [C.c_void_p, c_dbl_p, c_dbl_p, C.c_int]
        lib.so_amg_solve.argtypes = [C.c_void_p, c_dbl_p, c_dbl_p, C.c_double, C.c_int, c_dbl_p]
        lib.so_amg_coarse_solve.argtypes = [C.c_void_p, c_dbl_p, c_dbl_p]
        lib.so_pcg.argtypes = [C.c_void_p, c_dbl_p, c_dbl_p, C.c_double, C.c_int, c_dbl_p]
        lib.so_pbicgstab.argtypes = [C.c_void_p, c_dbl_p, c_dbl_p, C.c_double, C.c_int, c_dbl_p]
        lib.so_cg.argtypes = [C.c_int, c_int_p, c_int_p, c_dbl_p, c_dbl_p, c_dbl_p, C.c_double, C.c_int, c_dbl_p]
        lib.so_bicgstab.argtypes = lib.so_cg.argtypes
        lib.so_jacobi.argtypes = [C.c_int, c_int_p, c_int_p, c_dbl_p, c_dbl_p, c_dbl_p, c_dbl_p, c_dbl_p,
                                  C.c_double, C.c_int]
        lib.so_sor_multicolor.argtypes = [C.c_int, c_int_p, c_int_p, c_dbl_p, c_dbl_p, c_int_p, C.c_int, c_dbl_p,
                                          c_dbl_p, c_dbl_p, C.c_double, C.c_int]

    # ---- primitives -------------------------------------------------------------------------------------
    def set_threads(self, nt):
        self.lib.so_set_threads(int(nt))

    def spmv(self, A, x):
        y = np.empty(A.nrow)
        self.lib.so_spmv(A.nrow, ip(A.rowptr), ip(A.colindex), dp(A.val), dp(x), dp(y))
        return y

    def gmres(self, A, b, x, tol, restart=30, max_iter=500):
        """unpreconditioned GMRES(restart): (x, hist)"""
        x = x.copy()
        hist = np.zeros(max_iter + 1)
        k = self.lib.so_gmres(None, A.nrow, ip(A.rowptr), ip(A.colindex), dp(A.val), dp(b), dp(x), tol, restart, max_iter,
                              dp(hist))
        return x, hist[: k + 1]

    def jacobi(self, A, diag, b, x, omega, iteration):
        x = x.copy()
        h = np.empty(A.nrow)
        self.lib.so_jacobi(A.nrow, ip(A.rowptr), ip(A.colindex), dp(A.val), dp(diag), dp(b), dp(x), dp(h),
                           omega, iteration)
        return x

    def residual(self, A, b, x):
        h = np.empty(A.nrow)
        return self.lib.so_residual(A.nrow, ip(A.rowptr), ip(A.colindex), dp(A.val), dp(b), dp(x), dp(h))

    def store_residual(self, A, b, x):
        r = np.empty(A.nrow)
        self.lib.so_store_residual(A.nrow, ip(A.rowptr), ip(A.colindex), dp(A.val), dp(b), dp(x), dp(r))
        return r

    def transfer_residual(self, P, r):
        bc = np.empty(P.ncol)
        self.lib.so_transfer_residual(P.nrow, P.ncol, ip(P.rowptr), ip(P.colindex), dp(P.val), dp(r), dp(bc))
        return bc

    def transfer_solution(self, P, xc, xf):
        xf = xf.copy()
        self.lib.so_transfer_solution(P.nrow, ip(P.rowptr), ip(P.colindex), dp(P.val), dp(xc), dp(xf))
        return xf

    def sor_multicolor(self, A, diag, color_count, b, x, omega, iteration):
        x = x.copy()
        h = np.zeros(A.nrow)
        cc = np.ascontiguousarray(color_count, dtype=np.int32)
        self.lib.so_sor_multicolor(A.nrow, ip(A.rowptr), ip(A.colindex), dp(A.val), dp(diag), ip(cc), len(cc) - 1,
                                   dp(b), dp(x), dp(h), omega, iteration)
        return x

    def dot(self, x, y):
        return self.lib.so_dot(len(x), dp(x), dp(y))

    def nrm2(self, x):
        return self.lib.so_nrm2(len(x), dp(x))

    # ---- setup ------------------------------------------------------------------------------------------
    def hem(self, A, level):
        agg = np.empty(A.nrow, dtype=np.int32)
        nc = self.lib.so_hem(A.nrow, ip(A.rowptr), ip(A.colindex), dp(A.val), level, ip(agg))
        return nc, agg

    def beck(self, A):
        nc = C.c_int()
        prp, pci, pv = C.c_void_p(), C.c_void_p(), C.c_void_p()
        self.lib.so_beck(A.nrow, ip(A.rowptr), ip(A.colindex), C.byref(nc), C.byref(prp), C.byref(pci), C.byref(pv))
        rp = _take(self.lib, prp, A.nrow + 1, np.int32)
        return CSR(A.nrow, nc.value, rp, _take(self.lib, pci, rp[-1], np.int32), _take(self.lib, pv, rp[-1], np.float64))

    def rap(self, A, P):
        crp, cci, cv = C.c_void_p(), C.c_void_p(), C.c_void_p()
        self.lib.so_rap(A.nrow, ip(A.rowptr), ip(A.colindex), dp(A.val), P.ncol, ip(P.rowptr), ip(P.colindex),
                        dp(P.val), C.byref(crp), C.byref(cci), C.byref(cv))
        rp = _take(self.lib, crp, P.ncol + 1, np.int32)
        return CSR(P.ncol, P.ncol, rp, _take(self.lib, cci, rp[-1], np.int32), _take(self.lib, cv, rp[-1], np.float64))

    def color_reorder(self, A):
        perm = np.empty(A.nrow, dtype=np.int32)
        maxdeg = int(np.max(np.diff(A.rowptr)))
        cc = np.zeros(maxdeg + 2, dtype=np.int32)
        qrp, qci, qv = C.c_void_p(), C.c_void_p(), C.c_void_p()
        nc = self.lib.so_color_reorder(A.nrow, ip(A.rowptr), ip(A.colindex), dp(A.val), ip(perm), ip(cc),
                                       C.byref(qrp), C.byref(qci), C.byref(qv))
        rp = _take(self.lib, qrp, A.nrow + 1, np.int32)
        Q = CSR(A.nrow, A.nrow, rp, _take(self.lib, qci, rp[-1], np.int32), _take(self.lib, qv, rp[-1], np.float64))
        return nc, perm, cc[: nc + 1].copy(), Q

    def lu_solve(self, A, b):
        f = self.lib.so_lu_factor(A.nrow, ip(A.rowptr), ip(A.colindex), dp(A.val))
        x = np.empty(A.nrow)
        self.lib.so_lu_solve(f, dp(b), dp(x))
        self.lib.so_lu_free(f)
        return x

    def gen_poisson3d(self, nx, ny, nz):
        rp, ci, v = C.c_void_p(), C.c_void_p(), C.c_void_p()
        self.lib.so_gen_poisson3d_7pt(nx, ny, nz, C.byref(rp), C.byref(ci), C.byref(v))
        n = nx * ny * nz
        rowptr = _take(self.lib, rp, n + 1, np.int32)
        return CSR(n, n, rowptr, _take(self.lib, ci, rowptr[-1], np.int32), _take(self.lib, v, rowptr[-1], np.float64))

    def gen_poisson2d(self, nx, ny):
        rp, ci, v = C.c_void_p(), C.c_void_p(), C.c_void_p()
        self.lib.so_gen_poisson2d_5pt(nx, ny, C.byref(rp), C.byref(ci), C.byref(v))
        n = nx * ny
        rowptr = _take(self.lib, rp, n + 1, np.int32)
        return CSR(n, n, rowptr, _take(self.lib, ci, rowptr[-1], np.int32), _take(self.lib, v, rowptr[-1], np.float64))


class Hierarchy:
    """levels[k] = dict(A=CSR, diag=ndarray, P=CSR|None) — common shape for oracle, reference and product."""

    def __init__(self, levels):
        self.levels = levels

    @property
    def nlevels(self):
        return len(self.levels)


class OracleAmg:
    def __init__(self, A=None, coarsening=0, max_levels=32, limit_upper=4000, limit_lower=2000, hierarchy=None,
                 sor=False):
        self.o = Oracle.get()
        lib = self.o.lib
        if sor:
            self.h = lib.so_amg_setup_sor(A.nrow, ip(A.rowptr), ip(A.colindex), dp(A.val), max_levels, limit_upper,
                                          limit_lower)
        elif hierarchy is None:
            self.h = lib.so_amg_setup(A.nrow, ip(A.rowptr), ip(A.colindex), dp(A.val), coarsening, max_levels,
                                      limit_upper, limit_lower)
        else:
            L = hierarchy.levels
            n = len(L)
            self._keep = L
            nrow = (C.c_int * n)(*[l["A"].nrow for l in L])
            pncol = (C.c_int * n)(*[(l["P"].ncol if l["P"] is not None else 0) for l in L])

            def parr(getter, ctype):
                return (C.POINTER(ctype) * n)(*[getter(l) for l in L])

            null_i, null_d = C.POINTER(C.c_int)(), C.POINTER(C.c_double)()
            self.h = lib.so_amg_from_levels(
                n, nrow,
                parr(lambda l: ip(l["A"].rowptr), C.c_int), parr(lambda l: ip(l["A"].colindex), C.c_int),
                parr(lambda l: dp(l["A"].val), C.c_double), pncol,
                parr(lambda l: ip(l["P"].rowptr) if l["P"] is not None else null_i, C.c_int),
                parr(lambda l: ip(l["P"].colindex) if l["P"] is not None else null_i, C.c_int),
                parr(lambda l: dp(l["P"].val) if l["P"] is not None else null_d, C.c_double))
        self.n = self.level_dims(0)[0]

    def __del__(self):
        try:
            self.o.lib.so_amg_free(self.h)
        except Exception:
            pass

    @property
    def nlevels(self):
        return self.o.lib.so_amg_nlevels(self.h)

    def level_dims(self, k):
        a, b, c, d = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        self.o.lib.so_amg_level_dims(self.h, k, C.byref(a), C.byref(b), C.byref(c), C.byref(d))
        return a.value, b.value, c.value, d.value

    def hierarchy(self):
        levels = []
        for k in range(self.nlevels):
            nrow, nnz, pncol, pnnz = self.level_dims(k)
            ptrs = [C.c_void_p() for _ in range(7)]
            self.o.lib.so_amg_level_get(self.h, k, *[C.byref(p) for p in ptrs])

            def arr(p, n, ct, dt):
                return np.ctypeslib.as_array(C.cast(p, C.POINTER(ct)), shape=(max(n, 1),))[:n].astype(dt, copy=True)

            A = CSR(nrow, nrow, arr(ptrs[0], nrow + 1, C.c_int, np.int32), arr(ptrs[1], nnz, C.c_int, np.int32),
                    arr(ptrs[2], nnz, C.c_double, np.float64))
            diag = arr(ptrs[3], nrow, C.c_double, np.float64)
            P = None
            if k < self.nlevels - 1:
                P = CSR(nrow, pncol, arr(ptrs[4], nrow + 1, C.c_int, np.int32),
                        arr(ptrs[5], pnnz, C.c_int, np.int32), arr(ptrs[6], pnnz, C.c_double, np.float64))
            levels.append(dict(A=A, diag=diag, P=P))
        return Hierarchy(levels)

    def set_smoother(self, omega, smooth_iter):
        self.o.lib.so_amg_set_smoother(self.h, omega, smooth_iter)

    def vcycle(self, b, x, cycles=1):
        x = x.copy()
        self.o.lib.so_amg_vcycle(self.h, dp(b), dp(x), cycles)
        return x

    def solve(self, b, x, tol, max_cycles=500):
        x = x.copy()
        hist = np.zeros(max_cycles + 1)
        k = self.o.lib.so_amg_solve(self.h, dp(b), dp(x), tol, max_cycles, dp(hist))
        return x, hist[: k + 1]

    def coarse_solve(self, b):
        x = np.empty_like(b)
        self.o.lib.so_amg_coarse_solve(self.h, dp(b), dp(x))
        return x

    def solve_sor(self, b, x, tol, max_cycles=500):
        x = x.copy()
        hist = np.zeros(max_cycles + 1)
        k = self.o.lib.so_amg_solve_sor(self.h, dp(b), dp(x), tol, max_cycles, dp(hist))
        return x, hist[: k + 1]

    def pgmres(self, b, x, tol, restart=30, max_iter=500):
        x = x.copy()
        hist = np.zeros(max_iter + 1)
        k = self.o.lib.so_gmres(self.h, 0, None, None, None, dp(b), dp(x), tol, restart, max_iter, dp(hist))
        return x, hist[: k + 1]

    def pcg(self, b, x, tol, max_iter=500):
        x = x.copy()
        hist = np.zeros(max_iter + 1)
        k = self.o.lib.so_pcg(self.h, dp(b), dp(x), tol, max_iter, dp(hist))
        return x, hist[: k + 1]

    def pbicgstab(self, b, x, tol, max_iter=500):
        x = x.copy()
        hist = np.zeros(max_iter + 1)
        k = self.o.lib.so_pbicgstab(self.h, dp(b), dp(x), tol, max_iter, dp(hist))
        return x, hist[: k + 1]


class OracleOps:
    """the restatement's per-level primitives on hierarchy H, called the way RefAmg's are (by level index)"""

    def __init__(self, oracle, H):
        self.o, self.L = oracle, H.levels

    def spmv(self, k, x):
        return self.o.spmv(self.L[k]["A"], x)

    def jacobi(self, k, b, x, iteration):
        return self.o.jacobi(self.L[k]["A"], self.L[k]["diag"], b, x, 0.66667, iteration)

    def store_residual(self, k, b, x):
        return self.o.store_residual(self.L[k]["A"], b, x)

    def residual(self, k, b, x):
        return self.o.residual(self.L[k]["A"], b, x)

    def transfer_residual(self, k, r):
        return self.o.transfer_residual(self.L[k]["P"], r)

    def transfer_solution(self, k, xc, xf):
        return self.o.transfer_solution(self.L[k]["P"], xc, xf)

    def coarse_solve(self, b):
        return self.o.lu_solve(self.L[-1]["A"], b)


def primitive_outputs(H, ops):
    """{"<level>/<op>": output} of every per-level primitive of `ops` (OracleOps or RefAmg) on hierarchy H, from seeded
    random inputs, plus "coarse_solve"; the residual norm as a 1-element array"""
    rng = np.random.default_rng(11)
    out = {}
    for k, L in enumerate(H.levels):
        x, b = rng.random(L["A"].nrow), rng.random(L["A"].nrow)
        out[f"{k}/spmv"] = ops.spmv(k, x)
        out[f"{k}/jacobi"] = ops.jacobi(k, b, x, 6)
        out[f"{k}/store_residual"] = ops.store_residual(k, b, x)
        out[f"{k}/residual"] = np.array([ops.residual(k, b, x)])
        if L["P"] is not None:
            xc = rng.random(L["P"].ncol)
            out[f"{k}/transfer_residual"] = ops.transfer_residual(k, x)
            out[f"{k}/transfer_solution"] = ops.transfer_solution(k, xc, x)
    out["coarse_solve"] = ops.coarse_solve(rng.random(H.levels[-1]["A"].nrow))
    return out


def have_ref():
    return os.path.exists(REF_SO)


class Ref:
    """The reference's own host code (compiled unmodified), see oracle/ref_harness.cpp."""

    _inst = None

    @classmethod
    def get(cls):
        if cls._inst is None:
            cls._inst = cls()
        return cls._inst

    def __init__(self):
        lib = self.lib = C.CDLL(REF_SO)
        lib.ref_set_tol.argtypes = [C.c_double]
        lib.ref_set_tol_call_limit.argtypes = [C.c_long]
        lib.ref_amg_setup.restype = C.c_void_p
        lib.ref_amg_from_levels.restype = C.c_void_p
        lib.ref_amg_setup_seconds.restype = C.c_double
        lib.ref_amg_setup_seconds.argtypes = [C.c_void_p]
        lib.ref_amg_nlevels.argtypes = [C.c_void_p]
        lib.ref_amg_level_dims.argtypes = [C.c_void_p, C.c_int] + [c_int_p] * 4
        lib.ref_amg_level_copy.argtypes = [C.c_void_p, C.c_int, c_int_p, c_int_p, c_dbl_p, c_dbl_p, c_int_p, c_int_p,
                                           c_dbl_p]
        lib.ref_amg_vcycle.argtypes = [C.c_void_p, c_dbl_p, c_dbl_p, C.c_int]
        lib.ref_amg_solve.argtypes = [C.c_void_p, c_dbl_p, c_dbl_p, c_dbl_p, C.c_int]
        lib.ref_residual.restype = C.c_double
        lib.ref_residual.argtypes = [C.c_void_p, C.c_int, c_dbl_p, c_dbl_p]
        lib.ref_jacobi.argtypes = [C.c_void_p, C.c_int, c_dbl_p, c_dbl_p, C.c_int]
        lib.ref_store_residual.argtypes = [C.c_void_p, C.c_int, c_dbl_p, c_dbl_p, c_dbl_p]
        lib.ref_transfer_residual.argtypes = [C.c_void_p, C.c_int, c_dbl_p, c_dbl_p]
        lib.ref_transfer_solution.argtypes = [C.c_void_p, C.c_int, c_dbl_p, c_dbl_p]
        lib.ref_coarse_solve.argtypes = [C.c_void_p, c_dbl_p, c_dbl_p]
        lib.ref_spmv.argtypes = [C.c_void_p, C.c_int, c_dbl_p, c_dbl_p]
        lib.ref_pcg_sample.restype = C.c_double
        lib.ref_pcg_sample.argtypes = [C.c_void_p, c_dbl_p, c_dbl_p, C.c_int, c_dbl_p]
        lib.ref_pcg_solve.restype = C.c_double
        lib.ref_pcg_solve.argtypes = [C.c_void_p, c_dbl_p, c_dbl_p, C.c_double, C.c_int, c_dbl_p, c_int_p]
        lib.ref_solve.argtypes = [C.c_char_p, C.c_int, C.c_int, c_int_p, c_int_p, c_dbl_p, c_dbl_p, c_dbl_p, c_dbl_p,
                                  C.c_int]

    def set_threads(self, nt):
        self.lib.ref_set_threads(int(nt))

    def set_tol(self, tol):
        self.lib.ref_set_tol(float(tol))

    def solve(self, name, A, b, x0, maxhist=4096):
        x = x0.copy()
        hist = np.zeros(maxhist)
        k = self.lib.ref_solve(name.encode(), A.nrow, A.nnz, ip(A.rowptr), ip(A.colindex), dp(A.val), dp(b), dp(x),
                               dp(hist), maxhist)
        assert k >= 0, name
        return x, hist[:k]

    def color_reorder(self, A):
        n = A.nrow
        perm = np.empty(n, dtype=np.int32)
        cc = np.zeros(int(np.max(np.diff(A.rowptr))) + 2, dtype=np.int32)
        qrp = np.empty(n + 1, dtype=np.int32)
        qci = np.empty(A.nnz, dtype=np.int32)
        qv = np.empty(A.nnz)
        qd = np.empty(n)
        nc = self.lib.ref_color_reorder(n, A.nnz, ip(A.rowptr), ip(A.colindex), dp(A.val), ip(perm), ip(cc), ip(qrp),
                                        ip(qci), dp(qv), dp(qd))
        return nc, perm, cc[: nc + 1].copy(), CSR(n, n, qrp, qci, qv), qd

    def sor(self, Q, color_count, b, x, iteration):
        x = x.copy()
        cc = np.ascontiguousarray(color_count, dtype=np.int32)
        self.lib.ref_sor(Q.nrow, Q.nnz, ip(Q.rowptr), ip(Q.colindex), dp(Q.val), ip(cc), len(cc) - 1, dp(b), dp(x),
                         iteration)
        return x


class RefAmg:
    def __init__(self, A=None, coarsening=0, levels=None):
        self.r = Ref.get()
        if levels is None:
            self.h = self.r.lib.ref_amg_setup(A.nrow, A.nnz, ip(A.rowptr), ip(A.colindex), dp(A.val), coarsening)
            self.n = A.nrow
        else:  # adopt an existing hierarchy: list of dict(A=..., P=...) with numpy arrays
            n = len(levels)
            nrow = (C.c_int * n)(*[l["A"].nrow for l in levels])
            pncol = (C.c_int * n)(*[(l["P"].ncol if l["P"] is not None else 0) for l in levels])
            null_i, null_d = C.POINTER(C.c_int)(), C.POINTER(C.c_double)()

            def parr(getter, ctype):
                return (C.POINTER(ctype) * n)(*[getter(l) for l in levels])

            self.h = self.r.lib.ref_amg_from_levels(
                n, nrow, parr(lambda l: ip(l["A"].rowptr), C.c_int), parr(lambda l: ip(l["A"].colindex), C.c_int),
                parr(lambda l: dp(l["A"].val), C.c_double), pncol,
                parr(lambda l: ip(l["P"].rowptr) if l["P"] is not None else null_i, C.c_int),
                parr(lambda l: ip(l["P"].colindex) if l["P"] is not None else null_i, C.c_int),
                parr(lambda l: dp(l["P"].val) if l["P"] is not None else null_d, C.c_double))
            self.n = levels[0]["A"].nrow

    @property
    def nlevels(self):
        return self.r.lib.ref_amg_nlevels(self.h)

    @property
    def setup_seconds(self):
        return self.r.lib.ref_amg_setup_seconds(self.h)

    def level_dims(self, k):
        a, b, c, d = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        self.r.lib.ref_amg_level_dims(self.h, k, C.byref(a), C.byref(b), C.byref(c), C.byref(d))
        return a.value, b.value, c.value, d.value

    def hierarchy(self):
        levels = []
        for k in range(self.nlevels):
            nrow, nnz, pncol, pnnz = self.level_dims(k)
            rp, ci, v, dg = (np.empty(nrow + 1, np.int32), np.empty(nnz, np.int32), np.empty(nnz), np.empty(nrow))
            prp, pci, pv = np.empty(nrow + 1, np.int32), np.empty(max(pnnz, 1), np.int32), np.empty(max(pnnz, 1))
            self.r.lib.ref_amg_level_copy(self.h, k, ip(rp), ip(ci), dp(v), dp(dg), ip(prp), ip(pci), dp(pv))
            P = CSR(nrow, pncol, prp, pci[:pnnz], pv[:pnnz]) if k < self.nlevels - 1 else None
            levels.append(dict(A=CSR(nrow, nrow, rp, ci, v), diag=dg, P=P))
        return Hierarchy(levels)

    def vcycle(self, b, x, cycles=1):
        x = x.copy()
        self.r.lib.ref_amg_vcycle(self.h, dp(b), dp(x), cycles)
        return x

    def solve(self, b, x, maxhist=4096):
        x = x.copy()
        hist = np.zeros(maxhist)
        k = self.r.lib.ref_amg_solve(self.h, dp(b), dp(x), dp(hist), maxhist)
        return x, hist[:k]

    def residual(self, k, b, x):
        return self.r.lib.ref_residual(self.h, k, dp(b), dp(x))

    def jacobi(self, k, b, x, iteration):
        x = x.copy()
        self.r.lib.ref_jacobi(self.h, k, dp(b), dp(x), iteration)
        return x

    def store_residual(self, k, b, x):
        r = np.empty_like(b)
        self.r.lib.ref_store_residual(self.h, k, dp(b), dp(x), dp(r))
        return r

    def transfer_residual(self, k, r):
        bc = np.empty(self.level_dims(k)[2])
        self.r.lib.ref_transfer_residual(self.h, k, dp(r), dp(bc))
        return bc

    def transfer_solution(self, k, xc, xf):
        xf = xf.copy()
        self.r.lib.ref_transfer_solution(self.h, k, dp(xc), dp(xf))
        return xf

    def coarse_solve(self, b):
        x = np.empty_like(b)
        self.r.lib.ref_coarse_solve(self.h, dp(b), dp(x))
        return x

    def spmv(self, k, x):
        y = np.empty(self.level_dims(k)[0])
        self.r.lib.ref_spmv(self.h, k, dp(x), dp(y))
        return y

    def pcg_sample(self, b, x, m):
        x = x.copy()
        hist = np.zeros(m + 1)
        t = self.r.lib.ref_pcg_sample(self.h, dp(b), dp(x), m, dp(hist))
        return t, x, hist

    def pcg_solve(self, b, x, tol, max_iter=500):
        """Solver_PCG_1's loop run to ||r|| <= tol on this hierarchy -> (seconds, x, history incl. the initial residual)"""
        x = x.copy()
        hist = np.zeros(max_iter + 1)
        it = C.c_int()
        t = self.r.lib.ref_pcg_solve(self.h, dp(b), dp(x), float(tol), int(max_iter), dp(hist), C.byref(it))
        return t, x, hist[: it.value + 1]

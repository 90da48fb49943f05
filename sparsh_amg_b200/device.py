"""Thin object wrappers over the C-ABI: device vectors, device CSR matrices and the device hierarchy.

Names follow the reference: a `DeviceMatrix` is its sp_matrix_gpu, a `DeviceHierarchy` the device side of its
AMG_GPU1_solver (hierarchy resident on the GPU, "MI").  All arithmetic happens in lib/libsparsh_b200.so.
"""
import ctypes as C

import numpy as np

from . import capi
from .capi import check, dp, ip


def init(device=0):
    check(capi.load().sparsh_init(int(device)))


def sync():
    check(capi.load().sparsh_sync())


def set_stream(ptr):
    check(capi.load().sparsh_set_stream(C.c_void_p(ptr) if ptr else None))


def launch_count(reset=False):
    lib = capi.load()
    v = lib.sparsh_launch_count()
    if reset:
        lib.sparsh_launch_count_reset()
    return v


class DeviceVector:
    """n doubles in HBM"""

    def __init__(self, n=None, data=None):
        lib = capi.load()
        if data is not None:
            data = np.ascontiguousarray(data, dtype=np.float64)
            n = data.size
        self.n = int(n)
        p = C.c_void_p()
        check(lib.sparsh_malloc(max(self.n, 1) * 8, C.byref(p)))
        self.ptr = p.value
        if data is not None:
            self.upload(data)

    def upload(self, data):
        data = np.ascontiguousarray(data, dtype=np.float64)
        assert data.size == self.n
        if self.n:
            check(capi.load().sparsh_memcpy_h2d(self.ptr, data.ctypes.data, self.n * 8))
        return self

    def download(self):
        out = np.empty(self.n)
        if self.n:
            check(capi.load().sparsh_memcpy_d2h(out.ctypes.data, self.ptr, self.n * 8))
        return out

    def fill(self, value):
        check(capi.load().sparsh_fill(self.ptr, self.n, float(value)))
        return self

    def free(self):
        if getattr(self, "ptr", None):
            capi.load().sparsh_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class DeviceMatrix:
    def __init__(self, nrow=None, ncol=None, rowptr=None, colindex=None, val=None, diag=None, transpose=False,
                 handle=None, owned=True):
        self.lib = capi.load()
        self.owned = owned
        if handle is not None:
            self.h = handle
        else:
            rowptr = np.ascontiguousarray(rowptr, dtype=np.int32)
            colindex = np.ascontiguousarray(colindex, dtype=np.int32)
            val = np.ascontiguousarray(val, dtype=np.float64)
            nnz = int(rowptr[-1])
            h = C.c_void_p()
            if transpose:
                check(self.lib.sparsh_matrix_create_transpose(nrow, ncol, nnz, ip(rowptr), ip(colindex), dp(val),
                                                              C.byref(h)))
            else:
                dptr = dp(np.ascontiguousarray(diag, dtype=np.float64)) if diag is not None else None
                check(self.lib.sparsh_matrix_create(nrow, ncol, nnz, ip(rowptr), ip(colindex), dp(val), dptr,
                                                    C.byref(h)))
            self.h = h.value
        a, b, c = C.c_int(), C.c_int(), C.c_int()
        check(self.lib.sparsh_matrix_dims(self.h, C.byref(a), C.byref(b), C.byref(c)))
        self.nrow, self.ncol, self.nnz = a.value, b.value, c.value

    @classmethod
    def from_csr(cls, A, diag=None, transpose=False):
        return cls(A.nrow, A.ncol, A.rowptr, A.colindex, A.val, diag=diag, transpose=transpose)

    def kernel(self):
        a, b, c = C.c_int(), C.c_int(), C.c_int()
        check(self.lib.sparsh_matrix_kernel(self.h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def pattern_stats(self):
        """(patterns, table entries, escape rows, share of pattern 0) of the csr-pattern8 twin; patterns == 0: no twin"""
        a, b, c, d = C.c_int(), C.c_int(), C.c_int(), C.c_double()
        check(self.lib.sparsh_matrix_pattern_stats(self.h, C.byref(a), C.byref(b), C.byref(c), C.byref(d)))
        return a.value, b.value, c.value, d.value

    def pattern_mask_stats(self):
        """(patterns other than pattern 0 that the lean kernel runs as masked pattern 0, share of the rows that carry
        pattern 0 or one of them)"""
        a, b = C.c_int(), C.c_double()
        check(self.lib.sparsh_matrix_pattern_mask_stats(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def transfer_info(self):
        """(one entry per row, one value throughout, that value) as the upload found them: aggregation operators"""
        a, b, v = C.c_int(), C.c_int(), C.c_double()
        check(self.lib.sparsh_matrix_transfer_info(self.h, C.byref(a), C.byref(b), C.byref(v)))
        return bool(a.value), bool(b.value), v.value

    def kernel_name(self, epilogue):
        """name of the kernel instantiation launched for `epilogue` ('spmv' | 'residual' | 'jacobi' | 'prolong' | 'sor' |
        'spmv_dot' | 'resnorm')"""
        epi = ["spmv", "residual", "jacobi", "prolong", "sor", "spmv_dot", "resnorm"].index(epilogue)
        buf = C.create_string_buffer(200)
        check(self.lib.sparsh_matrix_kernel_name(self.h, epi, buf, 200))
        return buf.value.decode()

    def force_kernel(self, kind, threads_or_lanes):
        check(self.lib.sparsh_matrix_force_kernel(self.h, kind, threads_or_lanes))
        return self

    def update_values(self, val, diag=None):
        """new values (nnz, stored order) for the same sparsity; diag None: extracted.  numpy arrays or DeviceVectors.
        Twins, kernel family and transfer flags are chosen again as at upload (a forced kernel is forgotten)."""
        v, d = _on_device(val, self.nnz), _on_device(diag, self.nrow)
        check(self.lib.sparsh_matrix_update_values(self.h, v.ptr, d.ptr if d is not None else None))
        return self

    def fetch(self):
        """(rowptr, colindex, val, diag) copied back from the device; diag is None for a matrix without one"""
        rp = np.zeros(self.nrow + 1, dtype=np.int32)
        ci = np.zeros(max(self.nnz, 1), dtype=np.int32)
        v = np.zeros(max(self.nnz, 1))
        d = np.zeros(max(self.nrow, 1))
        try:
            check(self.lib.sparsh_matrix_fetch(self.h, ip(rp), ip(ci), dp(v), dp(d)))
        except capi.SparshError:  # no diagonal (rectangular operator)
            d = None
            check(self.lib.sparsh_matrix_fetch(self.h, ip(rp), ip(ci), dp(v), None))
        return rp, ci[: self.nnz], v[: self.nnz], (d[: self.nrow] if d is not None else None)

    # ---- per-op (device vectors in, device vectors out) ----
    def spmv(self, x, y=None):
        y = y or DeviceVector(self.nrow)
        check(self.lib.sparsh_spmv(self.h, x.ptr, y.ptr))
        return y

    def spmv_dot(self, x, y=None):
        y = y or DeviceVector(self.nrow)
        s = DeviceVector(1)
        check(self.lib.sparsh_spmv_dot(self.h, x.ptr, y.ptr, s.ptr))
        return y, float(s.download()[0])

    def residual(self, b, x, r=None):
        r = r or DeviceVector(self.nrow)
        check(self.lib.sparsh_residual(self.h, b.ptr, x.ptr, r.ptr))
        return r

    def residual_norm(self, b, x):
        out = C.c_double()
        check(self.lib.sparsh_residual_norm(self.h, b.ptr, x.ptr, C.byref(out)))
        return out.value

    def jacobi(self, b, x, omega, sweeps, tmp=None):
        tmp = tmp or DeviceVector(self.nrow)
        check(self.lib.sparsh_jacobi(self.h, b.ptr, x.ptr, tmp.ptr, float(omega), int(sweeps)))
        return x

    def mc_sor(self, color_count, b, x, omega, sweeps):
        cc = np.ascontiguousarray(color_count, dtype=np.int32)
        check(self.lib.sparsh_mc_sor(self.h, ip(cc), len(cc) - 1, b.ptr, x.ptr, float(omega), int(sweeps)))
        return x

    def restrict(self, r, bc=None):
        bc = bc or DeviceVector(self.nrow)
        check(self.lib.sparsh_restrict(self.h, r.ptr, bc.ptr))
        return bc

    def residual_restrict(self, R, b, x, bc=None):
        """bc = R (b - A x) (self is A): one fused pass where it applies, else residual + restriction"""
        bc = bc or DeviceVector(R.nrow)
        check(self.lib.sparsh_residual_restrict(self.h, R.h, b.ptr, x.ptr, bc.ptr))
        return bc

    def jacobi_zero(self, b, omega, x=None):
        """x = (omega*b)/d: the first Jacobi sweep from x = 0, d the smoothing diagonal"""
        x = x or DeviceVector(self.nrow)
        check(self.lib.sparsh_jacobi_zero(self.h, b.ptr, float(omega), x.ptr))
        return x

    def prolong_add(self, xc, xf):
        check(self.lib.sparsh_prolong_add(self.h, xc.ptr, xf.ptr))
        return xf

    def cg(self, b, x, tol, max_iter=10000):
        return _krylov(self.lib.sparsh_cg, self.h, b, x, tol, max_iter)

    def bicgstab(self, b, x, tol, max_iter=10000):
        return _krylov(self.lib.sparsh_bicgstab, self.h, b, x, tol, max_iter)

    def gmres(self, b, x, tol, restart=30, max_iter=10000):
        """unpreconditioned GMRES(restart) (addition: SURVEY §8f.2)"""
        return _gmres(self.lib.sparsh_gmres, self.h, b, x, tol, restart, max_iter)

    def free(self):
        if self.owned and getattr(self, "h", None):
            self.lib.sparsh_matrix_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _on_device(a, n):
    """a DeviceVector as given, a numpy array uploaded (None stays None)"""
    if a is None or isinstance(a, DeviceVector):
        assert a is None or a.n == n, (a.n, n)
        return a
    a = np.ascontiguousarray(a, dtype=np.float64)
    assert a.size == n, (a.size, n)
    return DeviceVector(data=a)


def _current_stream():
    s = C.c_void_p()
    check(capi.load().sparsh_get_stream(C.byref(s)))
    return s.value


def _device_ptr(v, n):
    """the device address of a DeviceVector or of a contiguous CUDA float64 tensor of n entries"""
    if isinstance(v, DeviceVector):
        assert v.n == n, (v.n, n)
        return v.ptr
    assert v.is_cuda and v.dtype.itemsize == 8 and v.dtype.is_floating_point and v.is_contiguous() and v.numel() == n
    return v.data_ptr()


class PendingSolve:
    """A solve enqueued by DeviceHierarchy.pcg_enqueue / pbicgstab_enqueue / amg_solve_enqueue: its history and status
    in device memory.  Nothing waits for the solve until result().  Pass it as `pending=` to a later enqueue to reuse
    its buffers: no allocation, which a call under stream capture requires."""

    def __init__(self, max_iter):
        self.max_iter = int(max_iter)
        self.hist = DeviceVector(self.max_iter + 1)
        self.status = DeviceVector(2)  # 16 bytes: the 3 int32 of d_status
        self.counted = True
        self.stream = None  # the library stream the last solve was enqueued on

    def result(self):
        """Synchronises the stream the last solve was enqueued on, whichever stream is current now, and returns
        (iterations, hist, converged) as pcg() etc. do.  The first call after an enqueue adds the loop's kernels to the
        launch counter.  (A solve captured into a graph of the caller's: replay it and synchronise first.)"""
        lib = capi.load()
        current = _current_stream()
        check(lib.sparsh_set_stream(self.stream))
        try:
            st = np.zeros(3, dtype=np.int32)
            check(lib.sparsh_memcpy_d2h(st.ctypes.data, self.status.ptr, st.nbytes))  # synchronises that stream first
            it, rc, kernels = int(st[0]), int(st[1]), int(st[2])
            hist = np.zeros(it + 1)
            check(lib.sparsh_memcpy_d2h(hist.ctypes.data, self.hist.ptr, hist.nbytes))
        finally:
            check(lib.sparsh_set_stream(current))
        if not self.counted:
            lib.sparsh_launch_count_add(kernels)
            self.counted = True
        return it, hist, rc == capi.SPARSH_OK


def galerkin_rap(A, P):
    """A_c = P^T (A P) computed on the device (sparsh_galerkin_rap) -> (rowptr, colindex, val) numpy arrays, or None when
    the device kernel does not apply (a product row longer than its per-thread list)"""
    lib = capi.load()
    h, nnz = C.c_void_p(), C.c_int()
    rp, ci, v = (np.ascontiguousarray(A.rowptr, dtype=np.int32), np.ascontiguousarray(A.colindex, dtype=np.int32),
                 np.ascontiguousarray(A.val, dtype=np.float64))
    prp, pci, pv = (np.ascontiguousarray(P.rowptr, dtype=np.int32), np.ascontiguousarray(P.colindex, dtype=np.int32),
                    np.ascontiguousarray(P.val, dtype=np.float64))
    check(lib.sparsh_galerkin_rap(A.nrow, ip(rp), ip(ci), dp(v), P.ncol, ip(prp), ip(pci), dp(pv), C.byref(h), C.byref(nnz)))
    if not h.value:
        return None
    out_rp = np.zeros(P.ncol + 1, dtype=np.int32)
    out_ci = np.zeros(max(nnz.value, 1), dtype=np.int32)
    out_v = np.zeros(max(nnz.value, 1))
    check(lib.sparsh_rap_fetch(h, ip(out_rp), ip(out_ci), dp(out_v)))
    check(lib.sparsh_rap_destroy(h))
    return out_rp, out_ci[: nnz.value], out_v[: nnz.value]


def _krylov(fn, handle, b, x, tol, max_iter):
    hist = np.zeros(max_iter + 1)
    it = C.c_int()
    rc = check(fn(handle, b.ptr, x.ptr, float(tol), int(max_iter), dp(hist), C.byref(it)), allow_not_converged=True)
    return it.value, hist[: it.value + 1], rc == capi.SPARSH_OK


def _gmres(fn, handle, b, x, tol, restart, max_iter):
    hist = np.zeros(max_iter + 1)
    it = C.c_int()
    rc = check(fn(handle, b.ptr, x.ptr, float(tol), int(restart), int(max_iter), dp(hist), C.byref(it)),
               allow_not_converged=True)
    return it.value, hist[: it.value + 1], rc == capi.SPARSH_OK


def dot(x, y):
    out = C.c_double()
    check(capi.load().sparsh_dot(x.n, x.ptr, y.ptr, C.byref(out)))
    return out.value


def nrm2(x):
    out = C.c_double()
    check(capi.load().sparsh_nrm2(x.n, x.ptr, C.byref(out)))
    return out.value


def axpy(a, x, y):
    check(capi.load().sparsh_axpy(x.n, float(a), x.ptr, y.ptr))


def axpby(a, x, b, y):
    check(capi.load().sparsh_axpby(x.n, float(a), x.ptr, float(b), y.ptr))


def axpbypcz(a, x, b, y, c, z):
    check(capi.load().sparsh_axpbypcz(x.n, float(a), x.ptr, float(b), y.ptr, float(c), z.ptr))


class DeviceHierarchy:
    """levels: list of dicts(A=CSR-like, diag=ndarray|None, P=CSR-like|None) with .nrow/.ncol/.rowptr/.colindex/.val"""

    def __init__(self, levels, omega=0.66667, pre_sweeps=7, post_sweeps=7, use_graph=True, smoother="jacobi"):
        self.lib = capi.load()
        n = len(levels)
        descs = (capi.LevelDesc * n)()
        keep = []
        for k, L in enumerate(levels):
            A = L["A"]
            rp = np.ascontiguousarray(A.rowptr, dtype=np.int32)
            ci = np.ascontiguousarray(A.colindex, dtype=np.int32)
            v = np.ascontiguousarray(A.val, dtype=np.float64)
            keep += [rp, ci, v]
            d = descs[k]
            d.nrow, d.nnz = A.nrow, int(rp[-1])
            d.rowptr, d.colindex, d.val = ip(rp), ip(ci), dp(v)
            if L.get("diag") is not None:
                dg = np.ascontiguousarray(L["diag"], dtype=np.float64)
                keep.append(dg)
                d.diag = dp(dg)
            P = L.get("P")
            if P is not None:
                prp = np.ascontiguousarray(P.rowptr, dtype=np.int32)
                pci = np.ascontiguousarray(P.colindex, dtype=np.int32)
                pv = np.ascontiguousarray(P.val, dtype=np.float64)
                keep += [prp, pci, pv]
                d.p_ncol, d.p_nnz = P.ncol, int(prp[-1])
                d.p_rowptr, d.p_colindex, d.p_val = ip(prp), ip(pci), dp(pv)
            if L.get("color_count") is not None:
                cc = np.ascontiguousarray(L["color_count"], dtype=np.int32)
                keep.append(cc)
                d.total_colors, d.color_count = len(cc) - 1, ip(cc)
        prm = capi.Params()
        self.lib.sparsh_params_default(C.byref(prm))
        prm.omega, prm.pre_sweeps, prm.post_sweeps, prm.use_graph = omega, pre_sweeps, post_sweeps, int(use_graph)
        prm.smoother = 1 if smoother == "sor" else 0
        h = C.c_void_p()
        check(self.lib.sparsh_hierarchy_create(n, descs, C.byref(prm), C.byref(h)))
        self.h = h.value
        self.n = levels[0]["A"].nrow
        self.nlevels = n

    def level(self, k):
        a, p, r = C.c_void_p(), C.c_void_p(), C.c_void_p()
        check(self.lib.sparsh_hierarchy_level(self.h, k, C.byref(a), C.byref(p), C.byref(r)))
        wrap = lambda hd: DeviceMatrix(handle=hd, owned=False) if hd else None  # noqa: E731
        return wrap(a.value), wrap(p.value), wrap(r.value)

    def refresh(self, val, diag=None):
        """new level-0 values (nnz, stored order; numpy array or DeviceVector) for the same sparsity: every coarse operator
        is recomputed on the device with the kept prolongators, twins and the coarse inverse are rebuilt"""
        A0 = self.level(0)[0]
        v, d = _on_device(val, A0.nnz), _on_device(diag, A0.nrow)
        check(self.lib.sparsh_hierarchy_refresh(self.h, v.ptr, d.ptr if d is not None else None))
        return self

    def coarse_solve(self, b, x=None):
        x = x or DeviceVector(b.n)
        check(self.lib.sparsh_hierarchy_coarse_solve(self.h, b.ptr, x.ptr))
        return x

    def vcycle(self, b, x, cycles=1, x_is_zero=False):
        check(self.lib.sparsh_hierarchy_vcycle(self.h, b.ptr, x.ptr, int(cycles), int(bool(x_is_zero))))
        return x

    def amg_solve(self, b, x, tol, max_cycles=500):
        return _krylov(self.lib.sparsh_hierarchy_amg_solve, self.h, b, x, tol, max_cycles)

    def pcg(self, b, x, tol, max_iter=500):
        return _krylov(self.lib.sparsh_hierarchy_pcg, self.h, b, x, tol, max_iter)

    def pbicgstab(self, b, x, tol, max_iter=500):
        return _krylov(self.lib.sparsh_hierarchy_pbicgstab, self.h, b, x, tol, max_iter)

    def pgmres(self, b, x, tol, restart=30, max_iter=500):
        """V-cycle-preconditioned GMRES(restart) (addition: SURVEY §8f.2)"""
        return _gmres(self.lib.sparsh_hierarchy_pgmres, self.h, b, x, tol, restart, max_iter)

    # ---- device-driven solves: enqueue on the library's current stream, never wait (see PendingSolve) ----
    def pcg_enqueue(self, b, x, tol, max_iter=500, pending=None):
        return self._enqueue(self.lib.sparsh_hierarchy_pcg_enqueue, b, x, tol, max_iter, pending)

    def pbicgstab_enqueue(self, b, x, tol, max_iter=500, pending=None):
        return self._enqueue(self.lib.sparsh_hierarchy_pbicgstab_enqueue, b, x, tol, max_iter, pending)

    def amg_solve_enqueue(self, b, x, tol, max_cycles=500, pending=None):
        return self._enqueue(self.lib.sparsh_hierarchy_amg_solve_enqueue, b, x, tol, max_cycles, pending)

    def _enqueue(self, fn, b, x, tol, max_iter, pending):
        """b, x: DeviceVectors or CUDA tensors of n float64"""
        p = pending if pending is not None else PendingSolve(max_iter)
        assert p.max_iter >= max_iter, (p.max_iter, max_iter)
        check(fn(self.h, _device_ptr(b, self.n), _device_ptr(x, self.n), float(tol), int(max_iter), p.hist.ptr,
                 p.status.ptr))
        p.stream = _current_stream()
        p.counted = False
        return p

    def solve_host(self, method, b_host, x_host, tol, max_iter=500):
        """method: 'amg' | 'pcg' | 'pbicgstab'; b_host/x_host are numpy arrays (x in/out)"""
        code = {"amg": 0, "pcg": 1, "pbicgstab": 2}[method]
        hist = np.zeros(max_iter + 1)
        it = C.c_int()
        rc = check(self.lib.sparsh_hierarchy_solve_host(self.h, code, b_host.ctypes.data, x_host.ctypes.data,
                                                        float(tol), int(max_iter), dp(hist), C.byref(it)),
                   allow_not_converged=True)
        return it.value, hist[: it.value + 1], rc == capi.SPARSH_OK

    def vcycle_bytes(self, x_is_zero=False):
        return self.lib.sparsh_hierarchy_vcycle_bytes(self.h, int(bool(x_is_zero)))

    def free(self):
        if getattr(self, "h", None):
            self.lib.sparsh_hierarchy_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

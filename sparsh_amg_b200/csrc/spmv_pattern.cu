// spmv_pattern.cu — csr-pattern8, lean variant: the row-sum kernel for matrices whose rows almost all repeat ONE pattern
// (the interior stencil row: 97.7 % of the rows of 3D Poisson 256^3 and of every level of its HEM hierarchy).
//
// The table kernel (spmv.cu: csr_pattern_kernel) serves every other csr-pattern8 matrix.  What it pays for and this one
// does not:
//  * two dependent memory round trips per tile (pattern byte -> table look-up -> gathers).  Pattern 0 travels BY VALUE
//    in the kernel parameters (Pat0, internal.cuh), so its offsets are constant-bank operands known before anything is
//    loaded: every thread issues the pattern byte, b, x_i AND all gathers of pattern 0 for all its rows at once —
//    one round trip — and only looks at the pattern byte when the data is there.  Rows whose pattern is pattern 0 with
//    terms left out (boundary rows, a few per cent: Pat0::mask) reuse those gathers and skip the missing terms; rows of
//    any other pattern are redone from the table in global memory, escapes from the CSR arrays;
//  * ~250 instructions per row of predicated 8-wide steps, selects and shared-memory look-ups (ncu on the dict kernel:
//    issue slots 65 % busy, ALU the top pipe).  The fast path is straight-line code: per entry one integer add, one
//    address computation, one LDG, one DMUL and one DADD whose second operands come from the constant bank;
//  * the table copy into shared memory: done only by CTAs that meet a row with another pattern.
// Same entries, same order, same unfused arithmetic as the CSR kernels: results are bit-identical.
#include "spmv_common.cuh"

namespace sparsh {

namespace {

template <bool COHERENT, bool DIST, bool SAFE>
__device__ __forceinline__ double gather(const double *x, int c, int ncol, int halo_begin) {
    if (!SAFE) c = min(max(c, 0), ncol - 1);  // speculative address of a row that may not carry pattern 0
    return load_xd<COHERENT, DIST>(x, c, halo_begin);
}

// One row of A as the lean kernel evaluates it, from the row's speculative pattern-0 gathers g (already in registers):
// pattern 0 by value, pattern 0 with terms left out (mask), another pattern from the table, or an escape from the CSR
// arrays.  NEEDS_D: d receives the row's diagonal, from the table when table_d, else (escapes always) dvec[row].
template <int LEN0, bool COH, bool DIST, bool NEEDS_D>
__device__ __forceinline__ double lean_row_sum(const CsrView &A, const PatView &P, const Pat0 &Z, const double *x, int row, int pid,
                                               const double (&g)[LEN0], bool table_d, const double *dvec, int halo_begin,
                                               double &d) {
    double sum = 0.0;
    unsigned m;
    if (pid == 0) {
#pragma unroll
        for (int k = 0; k < LEN0; k++) sum = __dadd_rn(sum, __dmul_rn(Z.val[k], g[k]));
        if (NEEDS_D && table_d) d = Z.diag;
    } else if ((m = Z.mask[pid]) & PAT_MASK_VALID) {
        // pattern 0 with terms left out (Pat0::mask: boundary rows and their Galerkin coarsenings; a quarter of the
        // warps of the finest 256^3 level and most warps of the coarse levels hold some): pattern 0's straight-line
        // code over the gathers already in registers.  A missing term's sum is discarded (the compiler selects the
        // old sum: DADD + FSEL, no branch), never its product zeroed, so an Inf, NaN or -0 in a skipped neighbour
        // changes nothing, as in the CSR kernels.
#pragma unroll
        for (int k = 0; k < LEN0; k++) {
            const double t = __dmul_rn(Z.val[k], g[k]);
            if (m & (1u << k)) sum = __dadd_rn(sum, t);
        }
        if (NEEDS_D && table_d) d = Z.diag;
    } else if (pid != PAT_ESCAPE) {
        // another pattern: walked straight from the table in global memory — a couple of KB that live in L1/L2 —
        // by the lanes concerned only: no shared-memory copy, no CTA barrier
        const int st = __ldg(P.start + pid), en = __ldg(P.start + pid + 1);
#pragma unroll 1  // rare path: small code, the instruction cache belongs to the fast path
        for (int k = st; k < en; k++) {
            const int4 q = __ldg(reinterpret_cast<const int4 *>(P.ent) + k);
            sum = __dadd_rn(sum, __dmul_rn(__hiloint2double(q.y, q.x), load_xd<COH, DIST>(x, row + q.z, halo_begin)));
        }
        if (NEEDS_D && table_d) d = __ldg(P.pdiag + pid);
    } else {
        const int lo = A.rowptr[row], hi = A.rowptr[row + 1];
#pragma unroll 1
        for (int k = lo; k < hi; k++)
            sum = __dadd_rn(sum, __dmul_rn(__ldg(A.val + k), load_xd<COH, DIST>(x, __ldg(A.col + k), halo_begin)));
        if (NEEDS_D) d = dvec[row];
    }
    return sum;
}

template <int THREADS, int RPT, int LEN0, int EPI, bool DIST>
__global__ void __launch_bounds__(THREADS)
    csr_pat2_kernel(CsrView A, PatView P, const __grid_constant__ Pat0 Z, const double *x, double *y, EpiArgs args,
                    RowRange rr, double *partials, HaloSync hs) {
    constexpr bool NEEDS_D = (EPI == EPI_JACOBI || EPI == EPI_SOR);
    constexpr bool COH = EpiTraits<EPI>::coherent_x;
    constexpr int TILE = THREADS * RPT;

    const int tid = threadIdx.x;
    int r0, row_end;
    block_rows(rr, TILE, r0, row_end);
    const int nrows = min(TILE, row_end - r0);

    HaloTurn hs_turn;
    if (DIST) hs_turn = halo_wait(hs);  // multi-GPU: the halo slices have landed before any (speculative) gather
    const bool strip_cta = !DIST || (int)blockIdx.x < hs.nstrip;
    // do the pattern-0 gathers of EVERY row of this tile stay inside the vector?  (CTA-uniform; false only at the ends)
    const bool safe = r0 + Z.lo >= 0 && r0 + TILE - 1 + Z.hi < A.ncol;
    const bool table_d = P.use_pdiag != 0;

    int pid[RPT];
    EpiRegs e[RPT];
    double g[RPT][LEN0];
#pragma unroll
    for (int s = 0; s < RPT; s++) {
        pid[s] = -1;
        if (s * THREADS + tid < nrows) {
            const int row = r0 + s * THREADS + tid;
            pid[s] = __ldg(P.pat + row);
            e[s] = epi_load<EPI, false>(args, y, row);
            if (NEEDS_D && !table_d) e[s].d = args.d[row];
            if (safe) {
#pragma unroll
                for (int k = 0; k < LEN0; k++) g[s][k] = gather<COH, DIST, true>(x, row + Z.off[k], A.ncol, hs.halo_begin);
            } else {
#pragma unroll
                for (int k = 0; k < LEN0; k++) g[s][k] = gather<COH, DIST, false>(x, row + Z.off[k], A.ncol, hs.halo_begin);
            }
        }
    }

    double contrib = 0.0;
#pragma unroll
    for (int s = 0; s < RPT; s++) {
        if (pid[s] < 0) continue;
        const int row = r0 + s * THREADS + tid;
        const double sum = lean_row_sum<LEN0, COH, DIST, NEEDS_D>(A, P, Z, x, row, pid[s], g[s], table_d, args.d, hs.halo_begin, e[s].d);
        // reduction contributions are added in row order within the thread: a fixed tree
        contrib = __dadd_rn(contrib, epi_store<EPI, DIST>(args, e[s], sum, y, row, strip_cta));
    }
    if (pushes<EPI, DIST>(args, strip_cta)) {
#pragma unroll 1
        for (int s = 0; s < RPT; s++)
            if (pid[s] >= 0) fused_push<EPI, DIST>(args, y, r0 + s * THREADS + tid);
    }
    if (EpiTraits<EPI>::reduces) block_partial<THREADS>(contrib, partials);
    if (DIST) halo_done(hs, hs_turn);
}

template <int THREADS, int RPT, int LEN0, int EPI>
int launch_cfg(const sparsh_matrix_s *A, const double *x, double *y, const EpiArgs &args, LaunchDesc d) {
    Context &c = ctx();
    const int grid = grid_for(d, THREADS * RPT);
    if (grid > RED_MAX_BLOCKS) {
        set_error("matrix too large for the reduction workspace");
        return SPARSH_ERR_INVALID;
    }
    const PatView P = A->pattern(args.d != nullptr && args.d == A->diag);
    if (d.dist)
        csr_pat2_kernel<THREADS, RPT, LEN0, EPI, true><<<grid, THREADS, 0, c.stream>>>(A->view(), P, A->pat0, x, y, args, d.rr, c.partials, d.hs);
    else
        csr_pat2_kernel<THREADS, RPT, LEN0, EPI, false><<<grid, THREADS, 0, c.stream>>>(A->view(), P, A->pat0, x, y, args, d.rr, c.partials, d.hs);
    count_launch();
    SP_CUDA(cudaGetLastError());
    if (EpiTraits<EPI>::reduces) return launch_finalize_partials(grid, args.red_out);
    return SPARSH_OK;
}

template <int LEN0, int EPI>
int launch_len(const sparsh_matrix_s *A, const double *x, double *y, const EpiArgs &args, const LaunchDesc &d) {
    // measured on B200, 3D Poisson 256^3 (profiles/r02g_pattern_lean_v3_sweep.log, r02n_kernel_probe.log): the sweeps
    // with a division in the epilogue (Jacobi, SOR) are fastest with one row per thread (256 x 1: 0.107 ms), the others
    // with two (128 x 2: SpMV 0.081 ms).  sparsh_matrix_force_kernel(KIND_PATTERN, threads) pins the CTA size (tests):
    // 256 -> 256 x 1, 128 -> 128 x 2 for every epilogue.
    const bool one_row = A->threads_forced ? A->threads == 256 : (EPI == EPI_JACOBI || EPI == EPI_SOR);
    if (one_row) return launch_cfg<256, 1, LEN0, EPI>(A, x, y, args, d);
    return launch_cfg<128, 2, LEN0, EPI>(A, x, y, args, d);
}

template <int EPI>
int launch_epi(const sparsh_matrix_s *A, const double *x, double *y, const EpiArgs &args, const LaunchDesc &d) {
    switch (A->pat0.len) {
        case 5:
            return launch_len<5, EPI>(A, x, y, args, d);
        default:
            return launch_len<7, EPI>(A, x, y, args, d);
    }
}

// V-cycle, fused residual + restriction: bc[i] = sum over the entries k of R's row i (stored order) of vR * r_j,
// r_j = b_j - (A x)_j, j = Rcol[k] — exactly what EPI_RESID followed by csr_scalar_kernel<EPI_SPMV> on R computes, with
// the residual never stored nor read back.  One thread per coarse row; fine row j is evaluated as csr_pat2_kernel does
// (lean_row_sum).  HEM's R has rows of two entries (pairs) and of one (singletons, numbered last): the loads of both
// rows of a pair — pattern byte, b and the clamped speculative pattern-0 gathers — are issued before either is used,
// so a pair costs one round trip after the Rcol load, as a row of the lean kernel does.
// (minimum 4 CTAs per SM: without it ptxas picks 40 registers and spills 16-20 B of the pair's state; with it, 40 / 46
// registers and no spill)
template <int LEN0>
__global__ void __launch_bounds__(256, 4)
    resid_restrict_kernel(CsrView A, PatView P, const __grid_constant__ Pat0 Z, const int *__restrict__ Rrp,
                          const int *__restrict__ Rcol, double vR, int nc, const double *__restrict__ b, const double *x,
                          double *bc) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= nc) return;
    const int lo = __ldg(Rrp + i), hi = __ldg(Rrp + i + 1);
    double acc = 0.0, dd = 0.0;
    if (hi - lo == 2) {
        int j[2], pid[2];
        double bj[2], g[2][LEN0];
        j[0] = __ldg(Rcol + lo);
        j[1] = __ldg(Rcol + lo + 1);
#pragma unroll
        for (int t = 0; t < 2; t++) {
            pid[t] = __ldg(P.pat + j[t]);
            bj[t] = __ldg(b + j[t]);
#pragma unroll
            for (int k = 0; k < LEN0; k++) g[t][k] = gather<false, false, false>(x, j[t] + Z.off[k], A.ncol, 0);
        }
#pragma unroll
        for (int t = 0; t < 2; t++) {
            const double s = lean_row_sum<LEN0, false, false, false>(A, P, Z, x, j[t], pid[t], g[t], false, nullptr, 0, dd);
            acc = __dadd_rn(acc, __dmul_rn(vR, __dsub_rn(bj[t], s)));
        }
    } else {
#pragma unroll 1
        for (int k = lo; k < hi; k++) {
            const int j = __ldg(Rcol + k);
            const int pid = __ldg(P.pat + j);
            const double bj = __ldg(b + j);
            double g[LEN0];
#pragma unroll
            for (int q = 0; q < LEN0; q++) g[q] = gather<false, false, false>(x, j + Z.off[q], A.ncol, 0);
            const double s = lean_row_sum<LEN0, false, false, false>(A, P, Z, x, j, pid, g, false, nullptr, 0, dd);
            acc = __dadd_rn(acc, __dmul_rn(vR, __dsub_rn(bj, s)));
        }
    }
    bc[i] = acc;
}

// First Jacobi sweep from x = 0: x = (omega*b)/d, d = A's diagonal read through the csr-pattern8 twin — pattern 0 by
// value, other patterns from the tabulated diagonals (a pattern with a valid mask has pattern 0's diagonal bits), escape
// rows from the diagonal array.  The upload makes every row whose diagonal differs from its pattern's an escape, so d
// has the bits of A->diag on every row: 17 B per row moved instead of 24.
__global__ void __launch_bounds__(256)
    jacobi_zero_pat_kernel(int n, const unsigned char *__restrict__ pat, const double *__restrict__ pdiag, double diag0,
                           const double *__restrict__ diag, const double *__restrict__ b, double omega, double *x) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const int p = __ldg(pat + i);
    const double bi = __ldg(b + i);
    double d = diag0;
    if (p == PAT_ESCAPE)
        d = __ldg(diag + i);
    else if (p != 0)
        d = __ldg(pdiag + p);
    x[i] = __ddiv_rn(__dmul_rn(omega, bi), d);
}

template <int LEN0>
int launch_rr(const sparsh_matrix_s *A, const sparsh_matrix_s *R, const double *b, const double *x, double *bc) {
    const int nc = R->nrow;
    resid_restrict_kernel<LEN0><<<(nc + 255) / 256, 256, 0, ctx().stream>>>(A->view(), A->pattern(false), A->pat0, R->rowptr, R->col,
                                                                          R->uval, nc, b, x, bc);
    count_launch();
    SP_CUDA(cudaGetLastError());
    return SPARSH_OK;
}

}  // namespace

// stencils whose interior row has 5 or 7 entries (2D/3D Poisson-like operators and their semi-coarsened Galerkin
// levels), as long as that row is the majority
bool pattern_lean_applies(const sparsh_matrix_s *A) {
    const int len = A->pat0.len;
    return A->has_pat && (len == 5 || len == 7) && A->pat0.cover >= 0.5;
}

int launch_pattern_lean(const sparsh_matrix_s *A, int epi, const double *x, double *y, const EpiArgs &args, LaunchDesc d) {
    switch (epi) {
        case EPI_SPMV:
            return launch_epi<EPI_SPMV>(A, x, y, args, d);
        case EPI_RESID:
            return launch_epi<EPI_RESID>(A, x, y, args, d);
        case EPI_JACOBI:
            return launch_epi<EPI_JACOBI>(A, x, y, args, d);
        case EPI_PROLONG:
            return launch_epi<EPI_PROLONG>(A, x, y, args, d);
        case EPI_SOR:
            return launch_epi<EPI_SOR>(A, x, y, args, d);
        case EPI_SPMV_DOT:
            return launch_epi<EPI_SPMV_DOT>(A, x, y, args, d);
        case EPI_RESNORM:
            return launch_epi<EPI_RESNORM>(A, x, y, args, d);
    }
    set_error("unknown epilogue");
    return SPARSH_ERR_INVALID;
}

bool resid_restrict_applies(const sparsh_matrix_s *A, const sparsh_matrix_s *R) {
    return A->kind == KIND_PATTERN && pattern_lean_applies(A) && R->uniform_val && R->ncol == A->nrow;
}

int launch_resid_restrict(const sparsh_matrix_s *A, const sparsh_matrix_s *R, const double *b, const double *x, double *bc) {
    if (R->nrow == 0) return SPARSH_OK;
    if (A->pat0.len == 5) return launch_rr<5>(A, R, b, x, bc);
    return launch_rr<7>(A, R, b, x, bc);
}

bool jacobi_zero_pat_applies(const sparsh_matrix_s *A) {
    return A->kind == KIND_PATTERN && pattern_lean_applies(A) && A->diag != nullptr;
}

int launch_jacobi_zero_pat(const sparsh_matrix_s *A, const double *b, double omega, double *x) {
    const int n = A->nrow;
    if (n == 0) return SPARSH_OK;
    jacobi_zero_pat_kernel<<<(n + 255) / 256, 256, 0, ctx().stream>>>(n, A->pat, A->pat_diag, A->pat0.diag, A->diag, b, omega, x);
    count_launch();
    SP_CUDA(cudaGetLastError());
    return SPARSH_OK;
}

}  // namespace sparsh

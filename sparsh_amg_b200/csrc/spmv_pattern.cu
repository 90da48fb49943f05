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
        double sum = 0.0;
        unsigned m;
        if (pid[s] == 0) {
#pragma unroll
            for (int k = 0; k < LEN0; k++) sum = __dadd_rn(sum, __dmul_rn(Z.val[k], g[s][k]));
            if (NEEDS_D && table_d) e[s].d = Z.diag;
        } else if ((m = Z.mask[pid[s]]) & PAT_MASK_VALID) {
            // pattern 0 with terms left out (Pat0::mask: boundary rows and their Galerkin coarsenings; a quarter of the
            // warps of the finest 256^3 level and most warps of the coarse levels hold some): pattern 0's straight-line
            // code over the gathers already in registers.  A missing term's sum is discarded (the compiler selects the
            // old sum: DADD + FSEL, no branch), never its product zeroed, so an Inf, NaN or -0 in a skipped neighbour
            // changes nothing, as in the CSR kernels.
#pragma unroll
            for (int k = 0; k < LEN0; k++) {
                const double t = __dmul_rn(Z.val[k], g[s][k]);
                if (m & (1u << k)) sum = __dadd_rn(sum, t);
            }
            if (NEEDS_D && table_d) e[s].d = Z.diag;
        } else if (pid[s] != PAT_ESCAPE) {
            // another pattern: walked straight from the table in global memory — a couple of KB that live in L1/L2 —
            // by the lanes concerned only: no shared-memory copy, no CTA barrier
            const int st = __ldg(P.start + pid[s]), en = __ldg(P.start + pid[s] + 1);
#pragma unroll 1  // rare path: small code, the instruction cache belongs to the fast path
            for (int k = st; k < en; k++) {
                const int4 q = __ldg(reinterpret_cast<const int4 *>(P.ent) + k);
                sum = __dadd_rn(sum, __dmul_rn(__hiloint2double(q.y, q.x), load_xd<COH, DIST>(x, row + q.z, hs.halo_begin)));
            }
            if (NEEDS_D && table_d) e[s].d = __ldg(P.pdiag + pid[s]);
        } else {
            const int lo = A.rowptr[row], hi = A.rowptr[row + 1];
#pragma unroll 1
            for (int k = lo; k < hi; k++)
                sum = __dadd_rn(sum, __dmul_rn(__ldg(A.val + k), load_xd<COH, DIST>(x, __ldg(A.col + k), hs.halo_begin)));
            if (NEEDS_D) e[s].d = args.d[row];
        }
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

}  // namespace sparsh

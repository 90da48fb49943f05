// spmv.cu — the CSR row-sum kernel family of the AMG solve phase (K1-K6, K9 of SURVEY §8a).
//
// One templated row-sum  y_i = epilogue(sum_j a_ij x_j)  serves SpMV, fused residual, fused weighted-Jacobi
// sweep, restriction (explicit R = P^T), fused prolongation-correction, one colour of multicolour SOR, and the
// fused SpMV+dot / residual-norm reductions.  Three families, chosen per matrix at upload (matrix.cu):
//
//  * STREAM (the hot one, 4-32 nnz/row): one CTA owns THREADS consecutive rows.  One elected thread issues two
//    TMA bulk copies (cp.async.bulk, SASS UBLKCP) that land the CTA's contiguous slice of `val` and `colindex`
//    in shared memory, completion signalled on an mbarrier.  Then thread t walks row t left to right out of
//    shared memory: the x gathers of neighbouring lanes hit neighbouring addresses (stencil rows), the matrix
//    stream never touches the LSU/L1 path, and several CTAs per SM keep >100 KB of HBM traffic in flight.
//    Row sums are accumulated sequentially with separate mul/add (no FMA contraction), i.e. in exactly the order
//    of the reference's CPU path (mkl_sparse_d_mv over column-sorted rows): results are bit-identical to the
//    oracle, not merely within 1e-12.
//  * DICT / PATTERN: the stream kernel's rows in two lossless compressed layouts (csr-dict16: 2 B per entry;
//    csr-pattern8: 1 B per row), for matrices whose entries / rows repeat (stencils and their Galerkin coarsenings).
//  * SCALAR (<= 2.5 nnz/row: aggregation P and R): thread per row straight from global memory (already coalesced).
//  * VECTOR (irregular / long rows): 2..32 lanes per row, shuffle-tree reduction (1e-12 parity, not bit-exact).
#include "spmv_common.cuh"

namespace sparsh {

// stage 2: a single CTA adds the partials in index order (65536 per-block atomics on one ticket cost ~60 us on a
// 256^3 SpMV; this kernel costs ~4 us and keeps the result independent of block scheduling)
__global__ void __launch_bounds__(1024) finalize_partials_kernel(const double *__restrict__ partials, int count, double *out) {
    __shared__ double sred[32];
    double acc = 0.0;
    for (int i = threadIdx.x; i < count; i += 1024) acc += partials[i];
    acc = block_sum<1024>(acc, sred);
    if (threadIdx.x == 0) *out = acc;
}

// ---------------------------------------------------------------------------------------------------------
// STREAM kernel
// ---------------------------------------------------------------------------------------------------------
template <int THREADS, int EPI, bool DIST>
__global__ void __launch_bounds__(THREADS)
    csr_stream_kernel(CsrView A, const double *x, double *y, EpiArgs args, RowRange rr, int cap, double *partials,
                      HaloSync hs) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double *sval = reinterpret_cast<double *>(smem_raw);
    int *scol = reinterpret_cast<int *>(smem_raw + (size_t)cap * sizeof(double));
    __shared__ __align__(8) uint64_t bar;
    __shared__ int s_a0;

    const int tid = threadIdx.x;
    int r0, row_end;
    block_rows(rr, THREADS, r0, row_end);
    const int nrows = min(THREADS, row_end - r0);

    if (tid == 0) {
        const int nz0 = A.rowptr[r0], nz1 = A.rowptr[r0 + nrows];
        const int a0 = nz0 & ~3;         // val + a0 is 32-byte, col + a0 16-byte aligned
        const int a1 = (nz1 + 3) & ~3;   // arrays are padded past nnz (matrix.cu)
        const int cnt = a1 - a0;
        s_a0 = a0;
        mbar_init(&bar, 1);
        fence_barrier_init();
        if (cnt > 0) {
            mbar_arrive_expect_tx(&bar, (uint32_t)cnt * 12u);
            bulk_g2s(sval, A.val + a0, (uint32_t)cnt * 8u, &bar);
            bulk_g2s(scol, A.col + a0, (uint32_t)cnt * 4u, &bar);
        } else {
            mbar_arrive(&bar);
        }
    }
    // per-row operands are fetched while the bulk copies are in flight
    int lo = 0, hi = 0;
    EpiRegs e;
    const int row = r0 + tid;
    const bool active = tid < nrows;
    if (active) {
        lo = A.rowptr[row];
        hi = A.rowptr[row + 1];
        e = epi_load<EPI>(args, y, row);
    }
    HaloTurn hs_turn;
    if (DIST) hs_turn = halo_wait(hs);  // multi-GPU: neighbours' halo slices have landed
    const bool strip_cta = !DIST || (int)blockIdx.x < hs.nstrip;
    __syncthreads();  // barrier init and s_a0 visible to everyone
    mbar_wait(&bar, 0);

    double contrib = 0.0;
    if (active) {
        const int a0 = s_a0;
        double s = 0.0;
        for (int k = lo - a0; k < hi - a0; k += 8) {
            double v[8], xv[8];
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const bool ok = k + j < hi - a0;
                v[j] = ok ? sval[k + j] : 0.0;
                const int c = ok ? scol[k + j] : 0;
                xv[j] = ok ? load_xd<EpiTraits<EPI>::coherent_x, DIST>(x, c, hs.halo_begin) : 0.0;
            }
#pragma unroll
            for (int j = 0; j < 8; j++)
                if (k + j < hi - a0) s = __dadd_rn(s, __dmul_rn(v[j], xv[j]));
        }
        contrib = epi_store<EPI, DIST>(args, e, s, y, row, strip_cta);
    }
    if (pushes<EPI, DIST>(args, strip_cta) && active) fused_push<EPI, DIST>(args, y, row);
    if (EpiTraits<EPI>::reduces) block_partial<THREADS>(contrib, partials);
    if (DIST) halo_done(hs, hs_turn);
}

// ---------------------------------------------------------------------------------------------------------
// DICT kernel: the stream kernel on the csr-dict16 twin.  The CTA's slice of 16-bit codes arrives by one TMA bulk
// copy (2 B/nnz of HBM traffic instead of 12), the two small dictionaries sit in shared memory, and thread t walks
// row t exactly as before — same values, same order, same unfused arithmetic: results stay bit-identical.
// ---------------------------------------------------------------------------------------------------------
template <int THREADS, int RPT, int EPI, bool DIST>
__global__ void __launch_bounds__(THREADS)
    csr_dict_kernel(CsrView A, DictView D, const double *x, double *y, EpiArgs args, RowRange rr, int cap,
                    double *partials, HaloSync hs) {
    // One CTA owns THREADS*RPT consecutive rows, thread t the rows r0 + s*THREADS + t (s < RPT).  With 2 B/nnz a
    // 256-row tile is only ~4 KB of matrix: a CTA must own several tiles' worth of rows, or the fixed cost of a CTA
    // (row pointer fetch -> bulk copy -> wait) caps the bytes in flight per SM below what saturates HBM.
    extern __shared__ __align__(128) unsigned char smem_raw[];
    unsigned short *scode = reinterpret_cast<unsigned short *>(smem_raw);
    double *sdv = reinterpret_cast<double *>(smem_raw + (size_t)cap * sizeof(unsigned short));
    int *sdo = reinterpret_cast<int *>(sdv + D.n_val);
    __shared__ __align__(8) uint64_t bar;
    __shared__ int s_a0;

    const int tid = threadIdx.x;
    int r0, row_end;
    block_rows(rr, THREADS * RPT, r0, row_end);
    const int nrows = min(THREADS * RPT, row_end - r0);

    if (tid == 0) {
        const int nz0 = A.rowptr[r0], nz1 = A.rowptr[r0 + nrows];
        const int a0 = nz0 & ~7;        // code + a0 is 16-byte aligned
        const int a1 = (nz1 + 7) & ~7;  // the code array is padded past nnz (matrix.cu)
        const int cnt = a1 - a0;
        s_a0 = a0;
        mbar_init(&bar, 1);
        fence_barrier_init();
        if (cnt > 0) {
            mbar_arrive_expect_tx(&bar, (uint32_t)cnt * 2u);
            bulk_g2s(scode, D.code + a0, (uint32_t)cnt * 2u, &bar);
        } else {
            mbar_arrive(&bar);
        }
    }
    for (int i = tid; i < D.n_val; i += THREADS) sdv[i] = D.val[i];
    for (int i = tid; i < D.n_off; i += THREADS) sdo[i] = D.off[i];
    // every per-row operand of all RPT rows is requested before anything is waited for
    int lo[RPT], hi[RPT];
    EpiRegs e[RPT];
#pragma unroll
    for (int s = 0; s < RPT; s++) {
        lo[s] = 0;
        hi[s] = 0;
        if (s * THREADS + tid < nrows) {
            const int row = r0 + s * THREADS + tid;
            lo[s] = A.rowptr[row];
            hi[s] = A.rowptr[row + 1];
            e[s] = epi_load<EPI>(args, y, row);
        }
    }
    HaloTurn hs_turn;
    if (DIST) hs_turn = halo_wait(hs);
    const bool strip_cta = !DIST || (int)blockIdx.x < hs.nstrip;
    __syncthreads();  // barrier init, s_a0 and the dictionaries visible to everyone
    mbar_wait(&bar, 0);

    double contrib = 0.0;
    const int a0 = s_a0;
#pragma unroll
    for (int s = 0; s < RPT; s++) {
        if (s * THREADS + tid < nrows) {
            const int row = r0 + s * THREADS + tid;
            double sum = 0.0;
            for (int k = lo[s] - a0; k < hi[s] - a0; k += 8) {
                double v[8], xv[8];
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const bool ok = k + j < hi[s] - a0;
                    const unsigned int code = ok ? scode[k + j] : 0u;
                    v[j] = ok ? sdv[code >> 8] : 0.0;
                    const int c = ok ? row + sdo[code & 255u] : 0;
                    xv[j] = ok ? load_xd<EpiTraits<EPI>::coherent_x, DIST>(x, c, hs.halo_begin) : 0.0;
                }
#pragma unroll
                for (int j = 0; j < 8; j++)
                    if (k + j < hi[s] - a0) sum = __dadd_rn(sum, __dmul_rn(v[j], xv[j]));
            }
            // reduction contributions are added in row order within the thread: still a fixed tree
            contrib = __dadd_rn(contrib, epi_store<EPI, DIST>(args, e[s], sum, y, row, strip_cta));
        }
    }
    if (pushes<EPI, DIST>(args, strip_cta)) {
#pragma unroll 1
        for (int s = 0; s < RPT; s++)
            if (s * THREADS + tid < nrows) fused_push<EPI, DIST>(args, y, r0 + s * THREADS + tid);
    }
    if (EpiTraits<EPI>::reduces) block_partial<THREADS>(contrib, partials);
    if (DIST) halo_done(hs, hs_turn);
}

// ---------------------------------------------------------------------------------------------------------
// PATTERN kernel: csr-pattern8 (PatView, internal.cuh).  One byte per row selects the row's list of (offset, value)
// pairs in a small table that each CTA copies into shared memory (a few KB out of L2; a warp whose rows share a
// pattern — the common case — reads each entry as one broadcast).  No matrix stream is left to stage: per
// row the kernel moves the pattern byte, the vector operands and the result, which is what bounds it.  Thread t owns
// rows r0 + s*THREADS + t (s < RPT); all their pattern bytes and per-row operands are requested before the table copy
// is waited for, together with an L2 prefetch of the one x line per row that no earlier row has touched (offset
// far_off: the next grid plane), so that the gathers that follow the table look-up find everything in L1/L2.
// Escape rows (id 255) are walked from the resident CSR arrays.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

template <int THREADS, int RPT, int JB, int EPI, bool DIST>
__global__ void __launch_bounds__(THREADS)
    csr_pattern_kernel(CsrView A, PatView P, const double *x, double *y, EpiArgs args, RowRange rr, double *partials,
                       HaloSync hs) {
    constexpr bool NEEDS_D = (EPI == EPI_JACOBI || EPI == EPI_SOR);
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double *sval = reinterpret_cast<double *>(smem_raw);   // n_ent values
    double *sdiag = sval + P.n_ent;                        // n_pat
    int *soff = reinterpret_cast<int *>(sdiag + P.n_pat);  // n_ent offsets
    int *sstart = soff + P.n_ent;                          // n_pat + 1

    const int tid = threadIdx.x;
    int r0, row_end;
    block_rows(rr, THREADS * RPT, r0, row_end);
    const int nrows = min(THREADS * RPT, row_end - r0);

    int pid[RPT];
    EpiRegs e[RPT];
#pragma unroll
    for (int s = 0; s < RPT; s++) {
        pid[s] = -1;
        if (s * THREADS + tid < nrows) {
            const int row = r0 + s * THREADS + tid;
            pid[s] = P.pat[row];
            e[s] = epi_load<EPI, false>(args, y, row);
            // one lane in 16 (= one per 128-byte line) asks L2 for the far line its rows will gather from
            if (P.far_off > 0 && (row & 15) == 0 && row + P.far_off < A.ncol) prefetch_l2(x + row + P.far_off);
        }
    }
    for (int i = tid; i < P.n_ent; i += THREADS) {
        const int4 q = __ldg(reinterpret_cast<const int4 *>(P.ent) + i);
        sval[i] = __hiloint2double(q.y, q.x);
        soff[i] = q.z;
    }
    for (int i = tid; i < P.n_pat; i += THREADS) sdiag[i] = __ldg(P.pdiag + i);
    for (int i = tid; i <= P.n_pat; i += THREADS) sstart[i] = __ldg(P.start + i);
    HaloTurn hs_turn;
    if (DIST) hs_turn = halo_wait(hs);
    const bool strip_cta = !DIST || (int)blockIdx.x < hs.nstrip;
    __syncthreads();  // the table is in place

    // The RPT rows of a thread advance together, JB entries each per step: RPT*JB independent gathers are in flight
    // per thread instead of one row's (each row's sum still runs left to right over its own entries).
    int st[RPT], len[RPT];
    double sum[RPT];
    int maxlen = 0;
#pragma unroll
    for (int s = 0; s < RPT; s++) {
        st[s] = 0;
        len[s] = 0;
        sum[s] = 0.0;
        if (pid[s] >= 0 && pid[s] != PAT_ESCAPE) {
            st[s] = sstart[pid[s]];
            len[s] = sstart[pid[s] + 1] - st[s];
            if (NEEDS_D) e[s].d = P.use_pdiag ? sdiag[pid[s]] : args.d[r0 + s * THREADS + tid];
        }
        maxlen = max(maxlen, len[s]);
    }
    for (int k = 0; k < maxlen; k += JB) {
        double v[RPT][JB], xv[RPT][JB];
#pragma unroll
        for (int s = 0; s < RPT; s++)
#pragma unroll
            for (int j = 0; j < JB; j++) {
                const bool ok = k + j < len[s];
                v[s][j] = ok ? sval[st[s] + k + j] : 0.0;
                const int c = ok ? r0 + s * THREADS + tid + soff[st[s] + k + j] : 0;
                xv[s][j] = ok ? load_xd<EpiTraits<EPI>::coherent_x, DIST>(x, c, hs.halo_begin) : 0.0;
            }
#pragma unroll
        for (int s = 0; s < RPT; s++)
#pragma unroll
            for (int j = 0; j < JB; j++)
                if (k + j < len[s]) sum[s] = __dadd_rn(sum[s], __dmul_rn(v[s][j], xv[s][j]));
    }

    double contrib = 0.0;
#pragma unroll
    for (int s = 0; s < RPT; s++) {
        if (pid[s] >= 0) {
            const int row = r0 + s * THREADS + tid;
            if (pid[s] == PAT_ESCAPE) {
                const int lo = A.rowptr[row], hi = A.rowptr[row + 1];
#pragma unroll 1  // rare path: keep it out of the instruction cache's way
                for (int k = lo; k < hi; k++)
                    sum[s] = __dadd_rn(sum[s], __dmul_rn(__ldg(A.val + k),
                                                         load_xd<EpiTraits<EPI>::coherent_x, DIST>(x, __ldg(A.col + k), hs.halo_begin)));
                if (NEEDS_D) e[s].d = args.d[row];
            }
            // reduction contributions are added in row order within the thread: still a fixed tree
            contrib = __dadd_rn(contrib, epi_store<EPI, DIST>(args, e[s], sum[s], y, row, strip_cta));
        }
    }
    if (pushes<EPI, DIST>(args, strip_cta)) {
#pragma unroll 1
        for (int s = 0; s < RPT; s++)
            if (pid[s] >= 0) fused_push<EPI, DIST>(args, y, r0 + s * THREADS + tid);
    }
    if (EpiTraits<EPI>::reduces) block_partial<THREADS>(contrib, partials);
    if (DIST) halo_done(hs, hs_turn);
}

// ---------------------------------------------------------------------------------------------------------
// SCALAR kernel: thread per row, rows of 1-2 entries (aggregation P / R): global loads are already coalesced
// ---------------------------------------------------------------------------------------------------------
template <int THREADS, int EPI, bool DIST>
__global__ void __launch_bounds__(THREADS)
    csr_scalar_kernel(CsrView A, const double *x, double *y, EpiArgs args, RowRange rr, double *partials, HaloSync hs) {
    int r0, row_end;
    block_rows(rr, THREADS, r0, row_end);
    const int row = r0 + threadIdx.x;
    HaloTurn hs_turn;
    if (DIST) hs_turn = halo_wait(hs);
    const bool strip_cta = !DIST || (int)blockIdx.x < hs.nstrip;
    double contrib = 0.0;
    if (row < row_end) {
        const int lo = A.rowptr[row], hi = A.rowptr[row + 1];
        EpiRegs e = epi_load<EPI>(args, y, row);
        double s = 0.0;
        for (int k = lo; k < hi; k++)
            s = __dadd_rn(s, __dmul_rn(__ldg(A.val + k), load_xd<EpiTraits<EPI>::coherent_x, DIST>(x, __ldg(A.col + k), hs.halo_begin)));
        contrib = epi_store<EPI, DIST>(args, e, s, y, row, strip_cta);
        if (pushes<EPI, DIST>(args, strip_cta)) fused_push<EPI, DIST>(args, y, row);
    }
    if (EpiTraits<EPI>::reduces) block_partial<THREADS>(contrib, partials);
    if (DIST) halo_done(hs, hs_turn);
}

// ---------------------------------------------------------------------------------------------------------
// AGGREGATION kernel: SpMV / prolongation with an operator of exactly one entry per row (rowptr[i] == i: HEM's P).  The
// scalar kernel's arithmetic in its order — s = 0 + v*x[col[i]] (the 0 + turns a -0 product into +0), then the epilogue
// — without reading rowptr, and without val when every stored value is the same (v passed by value, UNIFORM).
// ---------------------------------------------------------------------------------------------------------
template <int EPI, bool UNIFORM>
__global__ void __launch_bounds__(256)
    csr_agg_kernel(const int *__restrict__ col, const double *__restrict__ val, double v, const double *__restrict__ x, double *y,
                   RowRange rr) {
    int r0, row_end;
    block_rows(rr, 256, r0, row_end);
    const int row = r0 + threadIdx.x;
    if (row >= row_end) return;
    const double a = UNIFORM ? v : __ldg(val + row);
    const double s = __dadd_rn(0.0, __dmul_rn(a, __ldg(x + __ldg(col + row))));
    if (EPI == EPI_PROLONG)
        y[row] = __dadd_rn(s, y[row]);
    else
        y[row] = s;
}

// ---------------------------------------------------------------------------------------------------------
// VECTOR kernel: LANES lanes per row, fixed shuffle tree
// ---------------------------------------------------------------------------------------------------------
template <int LANES, int EPI, bool DIST>
__global__ void __launch_bounds__(256)
    csr_vector_kernel(CsrView A, const double *x, double *y, EpiArgs args, RowRange rr, double *partials, HaloSync hs) {
    constexpr int ROWS_PER_CTA = 256 / LANES;
    const int lane = threadIdx.x % LANES;
    int r0, row_end;
    block_rows(rr, ROWS_PER_CTA, r0, row_end);
    const int row = r0 + threadIdx.x / LANES;
    const bool active = row < row_end;
    HaloTurn hs_turn;
    if (DIST) hs_turn = halo_wait(hs);
    const bool strip_cta = !DIST || (int)blockIdx.x < hs.nstrip;
    double s = 0.0;
    EpiRegs e;
    if (active) {
        const int lo = A.rowptr[row], hi = A.rowptr[row + 1];
        if (lane == 0) e = epi_load<EPI>(args, y, row);
        for (int k = lo + lane; k < hi; k += LANES)
            s = __dadd_rn(s, __dmul_rn(__ldg(A.val + k), load_xd<EpiTraits<EPI>::coherent_x, DIST>(x, __ldg(A.col + k), hs.halo_begin)));
    }
#pragma unroll
    for (int off = LANES / 2; off > 0; off >>= 1) s += __shfl_down_sync(0xffffffffu, s, off, LANES);
    double contrib = 0.0;
    if (active && lane == 0) {
        contrib = epi_store<EPI, DIST>(args, e, s, y, row, strip_cta);
        if (pushes<EPI, DIST>(args, strip_cta)) fused_push<EPI, DIST>(args, y, row);
    }
    if (EpiTraits<EPI>::reduces) block_partial<256>(contrib, partials);
    if (DIST) halo_done(hs, hs_turn);
}

// ---------------------------------------------------------------------------------------------------------
// dispatch
// ---------------------------------------------------------------------------------------------------------
int launch_finalize_partials(int count, double *out) {
    Context &c = ctx();
    finalize_partials_kernel<<<1, 1024, 0, c.stream>>>(c.partials, count, out);
    count_launch();
    SP_CUDA(cudaGetLastError());
    return SPARSH_OK;
}

template <int EPI>
static int finish_launch(int grid, const EpiArgs &args) {
    count_launch();
    SP_CUDA(cudaGetLastError());
    if (EpiTraits<EPI>::reduces) return launch_finalize_partials(grid, args.red_out);
    return SPARSH_OK;
}

template <int THREADS, int EPI>
static int launch_stream(const sparsh_matrix_s *A, const double *x, double *y, const EpiArgs &args, LaunchDesc d) {
    Context &c = ctx();
    static bool attr_set = false;
    if (!attr_set) {
        SP_CUDA(cudaFuncSetAttribute(csr_stream_kernel<THREADS, EPI, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     200 * 1024));
        SP_CUDA(cudaFuncSetAttribute(csr_stream_kernel<THREADS, EPI, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     200 * 1024));
        attr_set = true;
    }
    const int win = THREADS == 256 ? A->win256 : A->win128;
    const int cap = ((win + 8) + 3) & ~3;
    const size_t smem = (size_t)cap * 12;
    const int grid = grid_for(d, THREADS);
    if (grid > RED_MAX_BLOCKS) {
        set_error("matrix too large for the reduction workspace");
        return SPARSH_ERR_INVALID;
    }
    if (d.dist)
        csr_stream_kernel<THREADS, EPI, true><<<grid, THREADS, smem, c.stream>>>(A->view(), x, y, args, d.rr, cap, c.partials, d.hs);
    else
        csr_stream_kernel<THREADS, EPI, false><<<grid, THREADS, smem, c.stream>>>(A->view(), x, y, args, d.rr, cap, c.partials, d.hs);
    return finish_launch<EPI>(grid, args);
}

template <int THREADS, int RPT, int EPI>
static int launch_dict_rpt(const sparsh_matrix_s *A, const double *x, double *y, const EpiArgs &args, LaunchDesc d) {
    Context &c = ctx();
    static bool attr_set = false;
    if (!attr_set) {
        SP_CUDA(cudaFuncSetAttribute(csr_dict_kernel<THREADS, RPT, EPI, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        SP_CUDA(cudaFuncSetAttribute(csr_dict_kernel<THREADS, RPT, EPI, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        attr_set = true;
    }
    const int win = RPT * (THREADS == 256 ? A->win256 : A->win128);  // bound for any THREADS*RPT-row window
    const int cap = ((win + 16) + 7) & ~7;
    const size_t smem = (size_t)cap * 2 + (size_t)A->n_dval * 8 + (size_t)A->n_doff * 4 + 16;
    if (smem > 200 * 1024) {
        set_error("csr-dict16 tile does not fit in shared memory");
        return SPARSH_ERR_INVALID;
    }
    const int grid = grid_for(d, THREADS * RPT);
    if (grid > RED_MAX_BLOCKS) {
        set_error("matrix too large for the reduction workspace");
        return SPARSH_ERR_INVALID;
    }
    if (d.dist)
        csr_dict_kernel<THREADS, RPT, EPI, true><<<grid, THREADS, smem, c.stream>>>(A->view(), A->dict(), x, y, args, d.rr, cap, c.partials, d.hs);
    else
        csr_dict_kernel<THREADS, RPT, EPI, false><<<grid, THREADS, smem, c.stream>>>(A->view(), A->dict(), x, y, args, d.rr, cap, c.partials, d.hs);
    return finish_launch<EPI>(grid, args);
}

// 4 rows per thread: measured best of 2 / 4 / 8 on B200 (256^3 Jacobi sweep: 0.180 ms)
template <int THREADS, int EPI>
static int launch_dict(const sparsh_matrix_s *A, const double *x, double *y, const EpiArgs &args, const LaunchDesc &d) {
    return launch_dict_rpt<THREADS, 4, EPI>(A, x, y, args, d);
}

template <int THREADS, int RPT, int JB, int EPI>
static int launch_pattern_cfg(const sparsh_matrix_s *A, const double *x, double *y, const EpiArgs &args, LaunchDesc d) {
    Context &c = ctx();
    const int grid = grid_for(d, THREADS * RPT);
    if (grid > RED_MAX_BLOCKS) {
        set_error("matrix too large for the reduction workspace");
        return SPARSH_ERR_INVALID;
    }
    const PatView P = A->pattern(args.d != nullptr && args.d == A->diag);
    // table: n_ent values + offsets, n_pat diagonals, n_pat + 1 starts: at most 27 KB (PAT_MAX_ENT), under the 48 KB
    // a kernel may use without opting in
    const size_t smem = (size_t)A->n_pent * 12 + (size_t)A->n_pat * 8 + (size_t)(A->n_pat + 1) * 4;
    if (d.dist)
        csr_pattern_kernel<THREADS, RPT, JB, EPI, true><<<grid, THREADS, smem, c.stream>>>(A->view(), P, x, y, args, d.rr, c.partials, d.hs);
    else
        csr_pattern_kernel<THREADS, RPT, JB, EPI, false><<<grid, THREADS, smem, c.stream>>>(A->view(), P, x, y, args, d.rr, c.partials, d.hs);
    return finish_launch<EPI>(grid, args);
}

template <int THREADS, int EPI>
static int launch_pattern(const sparsh_matrix_s *A, const double *x, double *y, const EpiArgs &args, const LaunchDesc &d) {
    // lean variant (spmv_pattern.cu): one dominant pattern, gathers issued before the pattern byte is known
    if (pattern_lean_applies(A)) return launch_pattern_lean(A, EPI, x, y, args, d);
    // every other csr-pattern8 matrix (pattern 0 not 5 or 7 entries long, or carried by fewer than half the rows): the
    // table kernel, 4 rows x 2 entries in flight per thread, the best of the shapes swept in round 2
    // (profiles/r02_pattern_sweep_256cubed.log)
    return launch_pattern_cfg<THREADS, 4, 2, EPI>(A, x, y, args, d);
}

template <int EPI>
static int launch_scalar(const sparsh_matrix_s *A, const double *x, double *y, const EpiArgs &args, LaunchDesc d) {
    Context &c = ctx();
    const int grid = grid_for(d, 256);
    if (grid > RED_MAX_BLOCKS) {
        set_error("matrix too large for the reduction workspace");
        return SPARSH_ERR_INVALID;
    }
    if constexpr (EPI == EPI_SPMV || EPI == EPI_PROLONG) {
        // one entry per row (HEM's P): rowptr is not read, nor val when it holds one value.  Single-GPU launches only:
        // the distributed operators keep the kernel with the halo handshake.
        if (A->agg && !d.dist) {
            if (A->uniform_val)
                csr_agg_kernel<EPI, true><<<grid, 256, 0, c.stream>>>(A->col, A->val, A->uval, x, y, d.rr);
            else
                csr_agg_kernel<EPI, false><<<grid, 256, 0, c.stream>>>(A->col, A->val, 0.0, x, y, d.rr);
            return finish_launch<EPI>(grid, args);
        }
    }
    if (d.dist)
        csr_scalar_kernel<256, EPI, true><<<grid, 256, 0, c.stream>>>(A->view(), x, y, args, d.rr, c.partials, d.hs);
    else
        csr_scalar_kernel<256, EPI, false><<<grid, 256, 0, c.stream>>>(A->view(), x, y, args, d.rr, c.partials, d.hs);
    return finish_launch<EPI>(grid, args);
}

template <int LANES, int EPI>
static int launch_vector(const sparsh_matrix_s *A, const double *x, double *y, const EpiArgs &args, LaunchDesc d) {
    Context &c = ctx();
    const int grid = grid_for(d, 256 / LANES);
    if (grid > RED_MAX_BLOCKS) {
        set_error("matrix too large for the reduction workspace");
        return SPARSH_ERR_INVALID;
    }
    if (d.dist)
        csr_vector_kernel<LANES, EPI, true><<<grid, 256, 0, c.stream>>>(A->view(), x, y, args, d.rr, c.partials, d.hs);
    else
        csr_vector_kernel<LANES, EPI, false><<<grid, 256, 0, c.stream>>>(A->view(), x, y, args, d.rr, c.partials, d.hs);
    return finish_launch<EPI>(grid, args);
}

template <int EPI>
static int launch_epi(const sparsh_matrix_s *A, const double *x, double *y, const EpiArgs &args, const LaunchDesc &d) {
    if (d.rows1 + d.rows2 + d.rows3 <= 0) {
        if (EpiTraits<EPI>::reduces) SP_CUDA(cudaMemsetAsync(args.red_out, 0, sizeof(double), ctx().stream));
        return SPARSH_OK;
    }
    switch (A->kind) {
        case KIND_SCALAR:
            return launch_scalar<EPI>(A, x, y, args, d);
        case KIND_STREAM:
            return A->threads == 128 ? launch_stream<128, EPI>(A, x, y, args, d) : launch_stream<256, EPI>(A, x, y, args, d);
        case KIND_DICT:
            return A->threads == 128 ? launch_dict<128, EPI>(A, x, y, args, d) : launch_dict<256, EPI>(A, x, y, args, d);
        case KIND_PATTERN:
            return A->threads == 128 ? launch_pattern<128, EPI>(A, x, y, args, d) : launch_pattern<256, EPI>(A, x, y, args, d);
        default:
            switch (A->lanes) {
                case 2:
                    return launch_vector<2, EPI>(A, x, y, args, d);
                case 4:
                    return launch_vector<4, EPI>(A, x, y, args, d);
                case 8:
                    return launch_vector<8, EPI>(A, x, y, args, d);
                case 16:
                    return launch_vector<16, EPI>(A, x, y, args, d);
                default:
                    return launch_vector<32, EPI>(A, x, y, args, d);
            }
    }
}

int launch_csr3(const sparsh_matrix_s *A, int epi, const double *x, double *y, const EpiArgs &args, int b1, int e1,
                int b2, int e2, int b3, int e3, const HaloSync *hs) {
    LaunchDesc d;
    d.rr = RowRange{b1, e1, b2, e2, b3, e3, 0, 0};
    d.rows1 = e1 > b1 ? e1 - b1 : 0;
    d.rows2 = e2 > b2 ? e2 - b2 : 0;
    d.rows3 = e3 > b3 ? e3 - b3 : 0;
    if (hs) d.hs = *hs;
    d.dist = d.hs.nnbr > 0 || d.hs.nsend > 0;
    if (d.hs.nnbr > 0 && d.rows1 + d.rows2 <= 0) {
        set_error("halo handshake attached to an empty launch");
        return SPARSH_ERR_INVALID;
    }
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

int launch_csr(const sparsh_matrix_s *A, int epi, const double *x, double *y, const EpiArgs &args, int row_begin,
               int row_end) {
    return launch_csr3(A, epi, x, y, args, row_begin, row_end, 0, 0, 0, 0, nullptr);
}

}  // namespace sparsh

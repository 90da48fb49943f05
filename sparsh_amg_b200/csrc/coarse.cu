// coarse.cu — K7 of SURVEY §8a: the coarsest-level solve, entirely on the device.
//
// The reference factors the coarsest matrix with host PARDISO (src/AMG_coarse_level_solver.cpp:9-62) and, in both GPU
// variants, ships B down and X up over PCIe every cycle (src/AMG_gpu_phases_2.cu:131-141,192-203).  Here the coarsest
// level (<= limit_upper = 4000 rows, include/AMG.hpp:19) is inverted ONCE at setup by in-place Gauss-Jordan with
// partial pivoting on the device (fp64), and every solve is one dense GEMV  x = A^{-1} b  — 8 n^2 bytes, HBM/L2-bound,
// no host round trip, deterministic.
#include <cooperative_groups.h>

#include <cmath>
#include <vector>

#include "internal.cuh"

namespace sparsh {

constexpr int GJ_T = 1024;
constexpr int GJ_MAX_ROWS = 512;  // rows of the matrix one CTA owns at most (n <= 16384 on >= 32 SMs)

// In-place-equivalent Gauss-Jordan with partial pivoting as ONE cooperative kernel (one CTA per SM, a grid barrier per
// elimination step) instead of two launches per pivot column: 2 launches per hierarchy instead of 2 n_L.  The matrix is
// double-buffered (step k reads Ma, writes Mb, then the roles swap), so a step has no intra-step hazard and needs a
// single barrier.  Step k, every CTA:
//   pivot search in column k of the current matrix (largest |a_ik|, i >= k, ties -> smallest i; done redundantly by
//   every CTA: 148 x n strided reads out of L2 are cheaper than a second barrier), then for its rows i
//     row k    <- (row p)/pivot with a_kk = 1/pivot                    (p = pivot row: the interchange is folded in)
//     row i!=k <- row i' - f_i * (row p)/pivot, column k treated as the unit vector   (i' = k if i == p, else i)
// — exactly the arithmetic of the textbook in-place update after swapping rows k and p.
__global__ void __launch_bounds__(GJ_T) gj_coop_kernel(double *Ma, double *Mb, int n, int *piv, double *minpiv) {
    cooperative_groups::grid_group grid = cooperative_groups::this_grid();
    __shared__ double sv[GJ_T / 32];
    __shared__ int si[GJ_T / 32];
    __shared__ int s_p;
    __shared__ int s_src[GJ_MAX_ROWS];
    __shared__ double s_f[GJ_MAX_ROWS];
    const int rows_per = (n + gridDim.x - 1) / gridDim.x;
    const int i_begin = blockIdx.x * rows_per, i_end = min(n, i_begin + rows_per);
    double worst = 1e300;
    for (int k = 0; k < n; k++) {
        const double *M = (k & 1) ? Mb : Ma;
        double *W = (k & 1) ? Ma : Mb;
        double best = -1.0;
        int bi = n;
        for (int i = k + threadIdx.x; i < n; i += GJ_T) {
            const double a = fabs(__ldcg(M + (size_t)i * n + k));
            if (a > best) {  // strictly greater: keeps the smallest index per thread
                best = a;
                bi = i;
            }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const double ob = __shfl_xor_sync(0xffffffffu, best, off);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
            if (ob > best || (ob == best && oi < bi)) {
                best = ob;
                bi = oi;
            }
        }
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
        if (lane == 0) {
            sv[warp] = best;
            si[warp] = bi;
        }
        __syncthreads();
        if (warp == 0) {
            best = sv[lane];
            bi = si[lane];
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                const double ob = __shfl_xor_sync(0xffffffffu, best, off);
                const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
                if (ob > best || (ob == best && oi < bi)) {
                    best = ob;
                    bi = oi;
                }
            }
            if (lane == 0) {
                s_p = bi < n ? bi : k;
                if (blockIdx.x == 0) piv[k] = s_p;
                worst = fmin(worst, best);
            }
        }
        __syncthreads();
        const int p = s_p;
        const double *prow = M + (size_t)p * n;
        const double pinv = 1.0 / __ldcg(prow + k);
        // source row (the interchange k <-> p folded in) and multiplier of each of this CTA's rows, once per step
        for (int r = threadIdx.x; r < i_end - i_begin; r += GJ_T) {
            const int i = i_begin + r;
            const int src = (i == k) ? p : (i == p) ? k : i;
            s_src[r] = src;
            s_f[r] = __ldcg(M + (size_t)src * n + k);
        }
        __syncthreads();
        for (int j = threadIdx.x; j < n; j += GJ_T) {
            const double pj = (j == k ? 1.0 : __ldcg(prow + j)) * pinv;
            for (int r = 0; r < i_end - i_begin; r++) {
                const int i = i_begin + r;
                double *w = W + (size_t)i * n + j;
                if (i == k) {
                    *w = pj;
                } else {
                    const double a = (j == k) ? 0.0 : __ldcg(M + (size_t)s_src[r] * n + j);
                    *w = a - s_f[r] * pj;
                }
            }
        }
        grid.sync();
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *minpiv = worst;
}

// undo the row interchanges: columns swapped in reverse pivot order; one CTA per row, row staged in shared memory
__global__ void __launch_bounds__(256) gj_unscramble_kernel(double *M, int n, const int *piv) {
    extern __shared__ double srow[];
    double *row = M + (size_t)blockIdx.x * n;
    for (int j = threadIdx.x; j < n; j += 256) srow[j] = row[j];
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = n - 1; k >= 0; k--) {
            const int p = piv[k];
            if (p != k) {
                double t = srow[k];
                srow[k] = srow[p];
                srow[p] = t;
            }
        }
    }
    __syncthreads();
    for (int j = threadIdx.x; j < n; j += 256) row[j] = srow[j];
}

// x = Ainv b: one warp per row, fixed lane-strided accumulation + shuffle tree (deterministic)
__global__ void __launch_bounds__(256) dense_gemv_kernel(const double *__restrict__ Minv, int n, const double *__restrict__ b, double *x) {
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= n) return;
    const double *m = Minv + (size_t)row * n;
    double s0 = 0.0, s1 = 0.0;
    int j = lane * 2;
    if ((n & 1) == 0 && (reinterpret_cast<uintptr_t>(b) & 15) == 0) {  // 16-byte loads need an aligned b
        for (; j + 1 < n; j += 64) {
            const double2 a = *reinterpret_cast<const double2 *>(m + j);
            const double2 v = *reinterpret_cast<const double2 *>(b + j);
            s0 = fma(a.x, v.x, s0);
            s1 = fma(a.y, v.y, s1);
        }
    } else {
        for (j = lane; j < n; j += 32) s0 = fma(m[j], b[j], s0);
    }
    double s = s0 + s1;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    if (lane == 0) x[row] = s;
}

// Gauss-Jordan of the dense n x n matrix in M, M2 the second buffer of the double-buffered elimination: on success
// *result is the buffer holding the inverse.  SPARSH_ERR_INVALID for a singular matrix.
static int gauss_jordan(double *M, double *M2, int n, int *piv, double *d_min, double **result) {
    Context &c = ctx();
    // one CTA per SM, all co-resident (cooperative launch): the elimination steps are separated by grid barriers
    int per_sm = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, gj_coop_kernel, GJ_T, 0);
    int grid = c.sm_count * (per_sm > 0 ? 1 : 0);
    if (grid > n) grid = n;
    if (e == cudaSuccess && (grid < 1 || (n + grid - 1) / grid > GJ_MAX_ROWS)) {
        set_error("coarse solver: the cooperative Gauss-Jordan kernel does not fit on this device");
        return SPARSH_ERR_CUDA;
    }
    if (e == cudaSuccess) {
        int nn = n;
        void *kargs[] = {&M, &M2, &nn, &piv, &d_min};
        e = cudaLaunchCooperativeKernel((const void *)gj_coop_kernel, dim3(grid), dim3(GJ_T), kargs, 0, c.stream);
        count_launch();
    }
    double *R = (n & 1) ? M2 : M;  // buffer written by the last step
    static bool attr = false;
    if (e == cudaSuccess && !attr) {
        e = cudaFuncSetAttribute(gj_unscramble_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 16384 * 8);
        attr = true;
    }
    if (e == cudaSuccess) {
        gj_unscramble_kernel<<<n, 256, sizeof(double) * (size_t)n, c.stream>>>(R, n, piv);
        count_launch();
        e = cudaGetLastError();
    }
    double h_min = 0.0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&h_min, d_min, sizeof(double), cudaMemcpyDeviceToHost, c.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c.stream);
    if (e != cudaSuccess) {
        set_error(std::string("coarse solver: ") + cudaGetErrorString(e));
        return SPARSH_ERR_CUDA;
    }
    // the reference aborts on a PARDISO error for a singular coarsest matrix (src/AMG_coarse_level_solver.cpp:52-60)
    if (!(h_min > 0.0) || !std::isfinite(h_min)) {
        set_error("coarsest-level matrix is singular (zero pivot in the dense factorisation): e.g. a pure-Neumann problem");
        return SPARSH_ERR_INVALID;
    }
    *result = R;
    return SPARSH_OK;
}

int coarse_build_inverse(int n, const int *rp, const int *ci, const double *v, CoarseInverse *out) {
    Context &c = ctx();
    NvtxRange nvtx("sparsh:coarse-inverse");
    if (n > 16384) {
        set_error("coarsest level too large for the dense device solve (n > 16384): coarsen further (raise level1)");
        return SPARSH_ERR_INVALID;
    }
    out->n = n;
    if (n == 0) return SPARSH_OK;
    std::vector<double> dense((size_t)n * n, 0.0);
    for (int i = 0; i < n; i++)
        for (int j = rp[i]; j < rp[i + 1]; j++) dense[(size_t)i * n + ci[j]] += v[j];
    double *M = nullptr, *M2 = nullptr, *d_min = nullptr;
    int *piv = nullptr;
    auto fail = [&](int rc) {
        cudaFree(M);
        cudaFree(M2);
        cudaFree(d_min);
        cudaFree(piv);
        out->n = 0;
        return rc;
    };
    if (cudaMalloc(&M, sizeof(double) * (size_t)n * n) != cudaSuccess || cudaMalloc(&M2, sizeof(double) * (size_t)n * n) != cudaSuccess ||
        cudaMalloc(&d_min, sizeof(double)) != cudaSuccess || cudaMalloc(&piv, sizeof(int) * (size_t)n) != cudaSuccess) {
        set_error(std::string("coarse solver: ") + cudaGetErrorString(cudaGetLastError()));
        return fail(SPARSH_ERR_CUDA);
    }
    const cudaError_t e = cudaMemcpyAsync(M, dense.data(), sizeof(double) * (size_t)n * n, cudaMemcpyHostToDevice, c.stream);
    if (e != cudaSuccess) {
        set_error(std::string("coarse solver: ") + cudaGetErrorString(e));
        return fail(SPARSH_ERR_CUDA);
    }
    double *R = nullptr;
    const int rc = gauss_jordan(M, M2, n, piv, d_min, &R);
    if (rc != SPARSH_OK) return fail(rc);
    cudaFree(R == M ? M2 : M);
    cudaFree(d_min);
    cudaFree(piv);
    out->inv = R;
    return SPARSH_OK;
}

// dense row i = the stored entries of row i added in stored order onto zeros (coarse_build_inverse's += on the host)
__global__ void __launch_bounds__(256)
    csr_to_dense_kernel(int n, const int *__restrict__ rp, const int *__restrict__ ci, const double *__restrict__ v, double *M) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    double *row = M + (size_t)i * n;
    for (int j = rp[i]; j < rp[i + 1]; j++) row[ci[j]] = __dadd_rn(row[ci[j]], v[j]);
}

int coarse_refactor(CoarseInverse *ci, const sparsh_matrix_s *A, double *spare, int *piv, double *d_min) {
    NvtxRange nvtx("sparsh:coarse-refactor");
    const int n = ci->n;
    if (n == 0) return SPARSH_OK;
    cudaStream_t st = ctx().stream;
    double *M = ci->inv;
    SP_CUDA(cudaMemsetAsync(M, 0, sizeof(double) * (size_t)n * n, st));
    csr_to_dense_kernel<<<(n + 255) / 256, 256, 0, st>>>(n, A->rowptr, A->col, A->val, M);
    count_launch();
    SP_CUDA(cudaGetLastError());
    double *R = nullptr;
    SP_TRY(gauss_jordan(M, spare, n, piv, d_min, &R));
    // the inverse stays at its address (odd n ends the elimination in the spare buffer: copied back, n^2 doubles), so a
    // coarse solve captured into a caller's graph before the refresh reads the new inverse
    if (R != M) SP_CUDA(cudaMemcpyAsync(M, R, sizeof(double) * (size_t)n * n, cudaMemcpyDeviceToDevice, st));
    return SPARSH_OK;
}

int coarse_apply(const CoarseInverse &ci, const double *b, double *x) {
    if (ci.n == 0) return SPARSH_OK;
    dense_gemv_kernel<<<(ci.n + 7) / 8, 256, 0, ctx().stream>>>(ci.inv, ci.n, b, x);
    count_launch();
    SP_CUDA(cudaGetLastError());
    return SPARSH_OK;
}

void coarse_free(CoarseInverse *ci) {
    if (ci->inv) cudaFree(ci->inv);
    ci->inv = nullptr;
    ci->n = 0;
}

}  // namespace sparsh

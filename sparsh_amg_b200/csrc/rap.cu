// rap.cu — Galerkin product A_c = P^T (A P) on the device (SURVEY §8f.1; replaces, for the setup, what the reference does
// with two mkl_sparse_spmm calls on the host: parallel::coarsen_matrix, src/AMG_cycle_utilities.cpp:126-146).
//
// The product is a pair of row-wise (Gustavson) sparse products, one thread per output row, written so that its result
// is the one host/setup.cpp computes BIT FOR BIT: the entries of a row appear in first-touch order and each is
// accumulated in traversal order with unfused multiply/add, then the columns are sorted (sp_matrix_fill).  Integer
// output (row pointers, sorted column indices) equals the reference's; the coarsening decisions that follow on the host
// (HEM / Beck are sequential greedy sweeps) therefore see identical matrices.
//   transpose   R = P^T, stable (a coarse row lists its fine rows ascending): count, scan, scatter, per-row sort
//   spgemm      two passes (count distinct columns per row -> scan -> fill), rows longer than RAP_MAX_ROW entries make the
//               call report "not applicable" and the host product runs instead (never a silent difference)
//   transfers   host arrays go through pinned staging buffers on up to four host threads (run_copies); a product can be the
//               fine matrix of the next one without leaving the device (sparsh_galerkin_rap_next)
// No cuSPARSE / thrust: the scans and sorts are the few kernels below.
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "internal.cuh"

namespace sparsh {

namespace {

constexpr int SCAN_T = 1024, SCAN_ITEMS = 4;

struct DevCsr {
    int nrow = 0, ncol = 0, nnz = 0;
    int *rp = nullptr, *ci = nullptr;
    double *v = nullptr;
    void release() {
        cudaFree(rp);
        cudaFree(ci);
        cudaFree(v);
        rp = ci = nullptr;
        v = nullptr;
    }
};

// device scratch that is released on every return path
template <typename T>
struct Scratch {
    T *p = nullptr;
    ~Scratch() { cudaFree(p); }
    cudaError_t alloc(size_t n) { return cudaMalloc(&p, sizeof(T) * std::max<size_t>(n, 1)); }
};

// ---- exclusive scan: out[0] = 0, out[i + 1] = in[0] + ... + in[i] ------------------------------------------------------
__global__ void __launch_bounds__(SCAN_T) scan_block_kernel(const int *__restrict__ in, int n, int *out, int *block_sum) {
    __shared__ int warp_tot[SCAN_T / 32];
    const int base = blockIdx.x * SCAN_T * SCAN_ITEMS + threadIdx.x * SCAN_ITEMS;
    int v[SCAN_ITEMS], run = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) {
        v[k] = base + k < n ? in[base + k] : 0;
        run += v[k];
    }
    int incl = run;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += t;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = warp_tot[lane];
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, w, off);
            if (lane >= off) w += t;
        }
        warp_tot[lane] = w;
    }
    __syncthreads();
    int excl = incl - run + (warp > 0 ? warp_tot[warp - 1] : 0);
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) {
        excl += v[k];
        if (base + k < n) out[base + k + 1] = excl;  // inclusive value at position +1: exclusive scan shifted by one
    }
    if (threadIdx.x == SCAN_T - 1) block_sum[blockIdx.x] = excl;
}
__global__ void __launch_bounds__(SCAN_T) scan_sums_kernel(int *block_sum, int nblocks) {  // one CTA: exclusive scan in place
    __shared__ int carry_s;
    __shared__ int warp_tot[SCAN_T / 32];
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int start = 0; start < nblocks; start += SCAN_T) {
        const int i = start + threadIdx.x;
        const int x = i < nblocks ? block_sum[i] : 0;
        int incl = x;
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, off);
            if (lane >= off) incl += t;
        }
        if (lane == 31) warp_tot[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            int w = warp_tot[lane];
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, w, off);
                if (lane >= off) w += t;
            }
            warp_tot[lane] = w;
        }
        __syncthreads();
        const int carry = carry_s;
        const int excl = carry + incl - x + (warp > 0 ? warp_tot[warp - 1] : 0);
        if (i < nblocks) block_sum[i] = excl;
        __syncthreads();
        if (threadIdx.x == SCAN_T - 1) carry_s = excl + x;
        __syncthreads();
    }
}
__global__ void __launch_bounds__(SCAN_T) scan_add_kernel(int *out, int n, const int *__restrict__ block_off) {
    const int base = blockIdx.x * SCAN_T * SCAN_ITEMS + threadIdx.x * SCAN_ITEMS;
    const int off = block_off[blockIdx.x];
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++)
        if (base + k < n) out[base + k + 1] += off;
    if (blockIdx.x == 0 && threadIdx.x == 0) out[0] = 0;
}
int exclusive_scan(const int *in, int n, int *out, cudaStream_t st) {
    if (n == 0) {
        SP_CUDA(cudaMemsetAsync(out, 0, sizeof(int), st));
        return SPARSH_OK;
    }
    const int nblocks = (n + SCAN_T * SCAN_ITEMS - 1) / (SCAN_T * SCAN_ITEMS);
    Scratch<int> sums;
    SP_CUDA(sums.alloc((size_t)nblocks));
    scan_block_kernel<<<nblocks, SCAN_T, 0, st>>>(in, n, out, sums.p);
    scan_sums_kernel<<<1, SCAN_T, 0, st>>>(sums.p, nblocks);
    scan_add_kernel<<<nblocks, SCAN_T, 0, st>>>(out, n, sums.p);
    SP_CUDA(cudaStreamSynchronize(st));  // the scratch is freed on return: the kernels must be done with it
    SP_CUDA(cudaGetLastError());
    return SPARSH_OK;
}

// ---- per-row insertion sort by column (rows are short) ----------------------------------------------------------------
__global__ void __launch_bounds__(256) sort_rows_kernel(int nrow, const int *__restrict__ rp, int *ci, double *v) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= nrow) return;
    const int lo = rp[i], hi = rp[i + 1];
    for (int a = lo + 1; a < hi; a++) {
        const int c = ci[a];
        const double x = v[a];
        int b = a - 1;
        while (b >= lo && ci[b] > c) {
            ci[b + 1] = ci[b];
            v[b + 1] = v[b];
            b--;
        }
        ci[b + 1] = c;
        v[b + 1] = x;
    }
}

// ---- transpose ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) count_cols_kernel(int nnz, const int *__restrict__ ci, int *count) {
    const int j = blockIdx.x * 256 + threadIdx.x;
    if (j < nnz) atomicAdd(&count[ci[j]], 1);
}
__global__ void __launch_bounds__(256)
    scatter_T_kernel(int nrow, const int *__restrict__ rp, const int *__restrict__ ci, const double *__restrict__ v,
                     const int *__restrict__ trp, int *cursor, int *tci, double *tv) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= nrow) return;
    for (int j = rp[i]; j < rp[i + 1]; j++) {
        const int c = ci[j];
        const int d = trp[c] + atomicAdd(&cursor[c], 1);
        tci[d] = i;  // the order inside a row of T is fixed afterwards by sort_rows_kernel (ascending source row)
        tv[d] = v[j];
    }
}
int transpose(const DevCsr &M, DevCsr *T, cudaStream_t st) {
    T->nrow = M.ncol;
    T->ncol = M.nrow;
    T->nnz = M.nnz;
    Scratch<int> count;  // T's arrays belong to the caller's DevCsr, which releases them on every path
    SP_CUDA(cudaMalloc(&T->rp, sizeof(int) * ((size_t)M.ncol + 1)));
    SP_CUDA(cudaMalloc(&T->ci, sizeof(int) * (size_t)std::max(M.nnz, 1)));
    SP_CUDA(cudaMalloc(&T->v, sizeof(double) * (size_t)std::max(M.nnz, 1)));
    SP_CUDA(count.alloc((size_t)M.ncol));
    SP_CUDA(cudaMemsetAsync(count.p, 0, sizeof(int) * (size_t)std::max(M.ncol, 1), st));
    if (M.nnz > 0) count_cols_kernel<<<(M.nnz + 255) / 256, 256, 0, st>>>(M.nnz, M.ci, count.p);
    SP_TRY(exclusive_scan(count.p, M.ncol, T->rp, st));
    SP_CUDA(cudaMemsetAsync(count.p, 0, sizeof(int) * (size_t)std::max(M.ncol, 1), st));
    if (M.nrow > 0) scatter_T_kernel<<<(M.nrow + 255) / 256, 256, 0, st>>>(M.nrow, M.rp, M.ci, M.v, T->rp, count.p, T->ci, T->v);
    if (T->nrow > 0) sort_rows_kernel<<<(T->nrow + 255) / 256, 256, 0, st>>>(T->nrow, T->rp, T->ci, T->v);
    SP_CUDA(cudaStreamSynchronize(st));
    SP_CUDA(cudaGetLastError());
    return SPARSH_OK;
}

// ---- C = A * B, Gustavson, one thread per row ---------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
    spgemm_count_kernel(int arow, const int *__restrict__ arp, const int *__restrict__ aci, const int *__restrict__ brp,
                        const int *__restrict__ bci, int *count, int *too_long) {
    const int i = blockIdx.x * 128 + threadIdx.x;
    if (i >= arow) return;
    int list[RAP_MAX_ROW];
    int cnt = 0;
    for (int ja = arp[i]; ja < arp[i + 1]; ja++) {
        const int k = aci[ja];
        for (int jb = brp[k]; jb < brp[k + 1]; jb++) {
            const int c = bci[jb];
            int t = 0;
            while (t < cnt && list[t] != c) t++;
            if (t == cnt) {
                if (cnt == RAP_MAX_ROW) {
                    atomicExch(too_long, 1);
                    count[i] = 0;
                    return;
                }
                list[cnt++] = c;
            }
        }
    }
    count[i] = cnt;
}
// entries of row i of C in first-touch order, each accumulated in traversal order with separate multiply and add:
// the host product's arithmetic (host/setup.cpp: spgemm), hence its bits
__global__ void __launch_bounds__(128)
    spgemm_fill_kernel(int arow, const int *__restrict__ arp, const int *__restrict__ aci, const double *__restrict__ av,
                       const int *__restrict__ brp, const int *__restrict__ bci, const double *__restrict__ bv,
                       const int *__restrict__ crp, int *cci, double *cv) {
    const int i = blockIdx.x * 128 + threadIdx.x;
    if (i >= arow) return;
    const int base = crp[i];
    int *cc = cci + base;
    double *cx = cv + base;
    int o = 0;
    for (int ja = arp[i]; ja < arp[i + 1]; ja++) {
        const int k = aci[ja];
        const double a = av[ja];
        for (int jb = brp[k]; jb < brp[k + 1]; jb++) {
            const int c = bci[jb];
            const double prod = __dmul_rn(a, bv[jb]);
            int t = 0;
            while (t < o && cc[t] != c) t++;
            if (t == o) {
                cc[o] = c;
                cx[o] = prod;
                o++;
            } else {
                cx[t] = __dadd_rn(cx[t], prod);
            }
        }
    }
}
// returns SPARSH_OK with *applicable = false when a row of the product has more than RAP_MAX_ROW entries
int spgemm(const DevCsr &A, const DevCsr &B, DevCsr *C, bool *applicable, cudaStream_t st) {
    *applicable = true;
    C->nrow = A.nrow;
    C->ncol = B.ncol;
    Scratch<int> count, flag;
    SP_CUDA(count.alloc((size_t)A.nrow));
    SP_CUDA(flag.alloc(1));
    SP_CUDA(cudaMalloc(&C->rp, sizeof(int) * ((size_t)A.nrow + 1)));
    SP_CUDA(cudaMemsetAsync(flag.p, 0, sizeof(int), st));
    const int grid = (A.nrow + 127) / 128;
    if (A.nrow > 0) spgemm_count_kernel<<<grid, 128, 0, st>>>(A.nrow, A.rp, A.ci, B.rp, B.ci, count.p, flag.p);
    SP_TRY(exclusive_scan(count.p, A.nrow, C->rp, st));
    int h_flag = 0, nnz = 0;
    SP_CUDA(cudaMemcpyAsync(&h_flag, flag.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    SP_CUDA(cudaMemcpyAsync(&nnz, C->rp + A.nrow, sizeof(int), cudaMemcpyDeviceToHost, st));
    SP_CUDA(cudaStreamSynchronize(st));
    if (h_flag) {
        *applicable = false;
        return SPARSH_OK;
    }
    C->nnz = nnz;
    SP_CUDA(cudaMalloc(&C->ci, sizeof(int) * (size_t)std::max(nnz, 1)));
    SP_CUDA(cudaMalloc(&C->v, sizeof(double) * (size_t)std::max(nnz, 1)));
    if (A.nrow > 0) spgemm_fill_kernel<<<grid, 128, 0, st>>>(A.nrow, A.rp, A.ci, A.v, B.rp, B.ci, B.v, C->rp, C->ci, C->v);
    SP_CUDA(cudaGetLastError());
    return SPARSH_OK;
}

// ---- pageable host arrays <-> device, a few arrays at a time ------------------------------------------------------------
// Each job is one contiguous copy through the pinned staging buffers of the thread that runs it (matrix.cu); up to four
// host threads, each on a stream of its own, share the jobs — one thread's memcpy into (out of) its staging buffer
// overlaps the DMA of the others, which is what a single pageable cudaMemcpy cannot do.
struct CopyJob {
    void *dst;
    const void *src;
    size_t bytes;
    bool to_device;
};
int run_copies(std::vector<CopyJob> jobs, cudaStream_t main_stream) {
    // split large jobs so that the threads end together
    constexpr size_t PIECE = (size_t)96 << 20;
    std::vector<CopyJob> pieces;
    for (const CopyJob &j : jobs)
        for (size_t off = 0; off < j.bytes; off += PIECE)
            pieces.push_back(CopyJob{static_cast<char *>(j.dst) + off, static_cast<const char *>(j.src) + off,
                                     std::min(PIECE, j.bytes - off), j.to_device});
    if (pieces.empty()) return SPARSH_OK;
    size_t total = 0;
    for (const CopyJob &j : pieces) total += j.bytes;
    int nthreads = total < ((size_t)32 << 20) ? 1 : (int)std::min<size_t>(pieces.size(), 4);
    if (const char *e = getenv("SPARSH_RAP_COPY_THREADS")) nthreads = std::max(1, std::min(atoi(e), 16));
    SP_CUDA(cudaStreamSynchronize(main_stream));  // the device side of every job is complete / free to overwrite
    std::atomic<size_t> next{0};
    std::atomic<int> first_rc{SPARSH_OK};
    std::mutex err_mutex;
    std::string err_msg;
    const int device = ctx().device;
    auto worker = [&](bool own_thread) {
        cudaStream_t st = main_stream;
        cudaStream_t mine = nullptr;
        if (own_thread) {
            cudaSetDevice(device);
            if (cudaStreamCreateWithFlags(&mine, cudaStreamNonBlocking) == cudaSuccess) st = mine;
        }
        for (size_t i = next++; i < pieces.size(); i = next++) {
            if (first_rc.load() != SPARSH_OK) break;
            const CopyJob &j = pieces[i];
            const int rc = j.to_device ? copy_h2d_staged(j.dst, j.src, j.bytes, st) : copy_d2h_staged(j.dst, j.src, j.bytes, st);
            if (rc != SPARSH_OK) {
                std::lock_guard<std::mutex> g(err_mutex);
                int expect = SPARSH_OK;
                if (first_rc.compare_exchange_strong(expect, rc)) err_msg = sparsh_last_error();
            }
        }
        if (cudaStreamSynchronize(st) != cudaSuccess) {
            int expect = SPARSH_OK;
            first_rc.compare_exchange_strong(expect, (int)SPARSH_ERR_CUDA);
        }
        if (mine) cudaStreamDestroy(mine);
        if (own_thread) release_upload_stage();
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < nthreads; t++) pool.emplace_back(worker, true);
    worker(false);
    for (auto &th : pool) th.join();
    if (first_rc.load() != SPARSH_OK) {
        set_error(err_msg.empty() ? "device Galerkin product: a copy failed" : err_msg);
        return first_rc.load();
    }
    return SPARSH_OK;
}

int alloc_csr(int nrow, int ncol, int nnz, DevCsr *M) {
    M->nrow = nrow;
    M->ncol = ncol;
    M->nnz = nnz;
    SP_CUDA(cudaMalloc(&M->rp, sizeof(int) * ((size_t)nrow + 1)));
    SP_CUDA(cudaMalloc(&M->ci, sizeof(int) * (size_t)std::max(nnz, 1)));
    SP_CUDA(cudaMalloc(&M->v, sizeof(double) * (size_t)std::max(nnz, 1)));
    return SPARSH_OK;
}
void upload_jobs(const DevCsr &M, const int *rp, const int *ci, const double *v, std::vector<CopyJob> *jobs) {
    jobs->push_back(CopyJob{M.rp, rp, sizeof(int) * ((size_t)M.nrow + 1), true});
    if (M.nnz > 0) {
        jobs->push_back(CopyJob{M.ci, ci, sizeof(int) * (size_t)M.nnz, true});
        jobs->push_back(CopyJob{M.v, v, sizeof(double) * (size_t)M.nnz, true});
    }
}

}  // namespace

int spgemm_structure(int arow, const int *arp, const int *aci, const int *brp, const int *bci, int **crp, int *nnz,
                     bool *fits, cudaStream_t st) {
    *crp = nullptr;
    *nnz = 0;
    *fits = true;
    Scratch<int> count, flag;
    SP_CUDA(count.alloc((size_t)arow));
    SP_CUDA(flag.alloc(1));
    SP_CUDA(cudaMemsetAsync(flag.p, 0, sizeof(int), st));
    if (arow > 0) spgemm_count_kernel<<<(arow + 127) / 128, 128, 0, st>>>(arow, arp, aci, brp, bci, count.p, flag.p);
    int h_flag = 0;
    SP_CUDA(cudaMemcpyAsync(&h_flag, flag.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    SP_CUDA(cudaStreamSynchronize(st));
    if (h_flag) {
        *fits = false;
        return SPARSH_OK;
    }
    SP_CUDA(cudaMalloc(crp, sizeof(int) * ((size_t)arow + 1)));
    SP_TRY(exclusive_scan(count.p, arow, *crp, st));
    SP_CUDA(cudaMemcpyAsync(nnz, *crp + arow, sizeof(int), cudaMemcpyDeviceToHost, st));
    SP_CUDA(cudaStreamSynchronize(st));
    return SPARSH_OK;
}

int spgemm_values(int arow, const int *arp, const int *aci, const double *av, const int *brp, const int *bci,
                  const double *bv, const int *crp, int *cci, double *cv, cudaStream_t st) {
    if (arow > 0) spgemm_fill_kernel<<<(arow + 127) / 128, 128, 0, st>>>(arow, arp, aci, av, brp, bci, bv, crp, cci, cv);
    count_launch();
    SP_CUDA(cudaGetLastError());
    return SPARSH_OK;
}

}  // namespace sparsh

using namespace sparsh;

struct sparsh_rap_s {
    DevCsr C;  // the Galerkin product on the device, columns sorted
};

// the product with the fine matrix taken from `fine` (on the device: a previous product) or uploaded from the host arrays
static int galerkin_product(const DevCsr *fine, int nrow, const int *h_rowptr, const int *h_colindex, const double *h_val,
                            int ncoarse, const int *h_p_rowptr, const int *h_p_colindex, const double *h_p_val,
                            sparsh_rap_t *out, int *nnz_coarse) {
    NvtxRange nvtx("sparsh:galerkin-rap");
    cudaStream_t st = ctx().stream;
    *out = nullptr;
    *nnz_coarse = -1;
    DevCsr A_up, P, R, AP;
    sparsh_rap_s *h = new sparsh_rap_s();
    bool ok1 = true, ok2 = true;
    static const bool timing = getenv("SPARSH_SETUP_TIMING") != nullptr;
    const auto t0 = std::chrono::steady_clock::now();
    auto lap = [&](const char *what) {
        if (!timing || nrow < 20000) return;
        cudaStreamSynchronize(st);
        std::fprintf(stderr, "[rap %d rows] %s at %.3f s\n", nrow, what,
                     std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
    };
    std::vector<CopyJob> jobs;
    int rc = SPARSH_OK;
    if (!fine) {
        rc = alloc_csr(nrow, nrow, h_rowptr[nrow], &A_up);
        if (rc == SPARSH_OK) upload_jobs(A_up, h_rowptr, h_colindex, h_val, &jobs);
    }
    if (rc == SPARSH_OK) rc = alloc_csr(nrow, ncoarse, h_p_rowptr[nrow], &P);
    if (rc == SPARSH_OK) upload_jobs(P, h_p_rowptr, h_p_colindex, h_p_val, &jobs);
    if (rc == SPARSH_OK) rc = run_copies(jobs, st);
    const DevCsr &A = fine ? *fine : A_up;
    lap(fine ? "P uploaded (A is on the device)" : "A, P uploaded");
    if (rc == SPARSH_OK) rc = spgemm(A, P, &AP, &ok1, st);                 // A P
    lap("A P");
    if (rc == SPARSH_OK && ok1) rc = transpose(P, &R, st);                 // R = P^T
    lap("R = P^T");
    if (rc == SPARSH_OK && ok1) rc = spgemm(R, AP, &h->C, &ok2, st);       // R (A P)
    lap("R (A P)");
    if (rc == SPARSH_OK && ok1 && ok2) {
        if (h->C.nrow > 0) sort_rows_kernel<<<(h->C.nrow + 255) / 256, 256, 0, st>>>(h->C.nrow, h->C.rp, h->C.ci, h->C.v);
        if (cudaStreamSynchronize(st) != cudaSuccess || cudaGetLastError() != cudaSuccess) {
            set_error("device Galerkin product failed");
            rc = SPARSH_ERR_CUDA;
        }
    }
    A_up.release();
    P.release();
    R.release();
    AP.release();
    if (rc != SPARSH_OK || !ok1 || !ok2) {
        h->C.release();
        delete h;
        return rc;  // SPARSH_OK with *out == NULL: a product row exceeds the per-thread list; the caller uses its host product
    }
    *nnz_coarse = h->C.nnz;
    *out = h;
    return SPARSH_OK;
}

extern "C" {

int sparsh_galerkin_rap(int nrow, const int *h_rowptr, const int *h_colindex, const double *h_val, int ncoarse,
                        const int *h_p_rowptr, const int *h_p_colindex, const double *h_p_val, sparsh_rap_t *out,
                        int *nnz_coarse) {
    SP_TRY(ensure_init());
    SP_REQUIRE(nrow >= 0 && ncoarse >= 0 && h_rowptr && h_p_rowptr && out && nnz_coarse, "bad arguments");
    return galerkin_product(nullptr, nrow, h_rowptr, h_colindex, h_val, ncoarse, h_p_rowptr, h_p_colindex, h_p_val, out,
                            nnz_coarse);
}

int sparsh_galerkin_rap_next(sparsh_rap_t fine, int ncoarse, const int *h_p_rowptr, const int *h_p_colindex,
                             const double *h_p_val, sparsh_rap_t *out, int *nnz_coarse) {
    SP_TRY(ensure_init());
    SP_REQUIRE(fine != nullptr && ncoarse >= 0 && h_p_rowptr && out && nnz_coarse, "bad arguments");
    return galerkin_product(&fine->C, fine->C.nrow, nullptr, nullptr, nullptr, ncoarse, h_p_rowptr, h_p_colindex, h_p_val,
                            out, nnz_coarse);
}

int sparsh_rap_fetch(sparsh_rap_t h, int *h_rowptr, int *h_colindex, double *h_val) {
    SP_REQUIRE(h != nullptr && h_rowptr != nullptr, "bad arguments");
    std::vector<CopyJob> jobs;
    jobs.push_back(CopyJob{h_rowptr, h->C.rp, sizeof(int) * ((size_t)h->C.nrow + 1), false});
    if (h->C.nnz > 0) {
        SP_REQUIRE(h_colindex != nullptr && h_val != nullptr, "bad arguments");
        jobs.push_back(CopyJob{h_colindex, h->C.ci, sizeof(int) * (size_t)h->C.nnz, false});
        jobs.push_back(CopyJob{h_val, h->C.v, sizeof(double) * (size_t)h->C.nnz, false});
    }
    return run_copies(jobs, ctx().stream);
}

int sparsh_rap_destroy(sparsh_rap_t h) {
    if (!h) return SPARSH_OK;
    h->C.release();
    delete h;
    return SPARSH_OK;
}

}  // extern "C"

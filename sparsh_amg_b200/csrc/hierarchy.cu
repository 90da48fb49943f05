// hierarchy.cu — hierarchy upload and the V-cycle (row V of SURVEY §8a).
//
// Replaces AMG_GPU1_solver::GPU_Allocations / AMG_Solve (reference src/AMG_gpu_phases_2.cu:13-240) and
// AMG_GPU_solver (src/AMG_gpu_phases.cu:13-459).  Cycle semantics follow AMG_solver::AMG_solve_jacobi
// (src/AMG_phases.cpp:151-230), the only runnable oracle:
//   down: Jacobi(A_l,B_l,X_l) -> R_l = B_l - A_l X_l -> B_{l+1} = P_l^T R_l -> X_{l+1} = 0
//   bottom: X_L = A_L^{-1} B_L
//   up:   X_{l-1} += P_{l-1} X_l -> Jacobi(A_{l-1},B_{l-1},X_{l-1})
// One fused kernel per Jacobi sweep (out of place, ping-pong), one for residual + restriction (two where the fused
// kernel does not apply: resid_restrict_applies), one per prolongation-correction; the first sweep after "X = 0" needs
// no matrix pass at all (A*0 = 0 exactly).
// The whole cycle is captured into a CUDA graph: a 14-level hierarchy is ~250 launches, most of them on levels too
// small to hide launch latency otherwise.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <string>
#include <thread>
#include <utility>

#include "hierarchy.cuh"

using namespace sparsh;

namespace sparsh {

static int smooth(sparsh_hierarchy_s *h, Level &L, const double *b, double *&cur, double *&other, int sweeps,
                  bool zero_guess) {
    if (sweeps == 0 || h->prm.smoother == 1) {
        if (zero_guess) SP_TRY(k_fill(cur, (size_t)L.n, 0.0));
        // multicolour SOR, in place, one launch per colour (reference src/AMG_smoothers.cpp:78-102)
        const int ncol = (int)L.color_count.size() - 1;
        for (int s = 0; s < sweeps && h->prm.smoother == 1; s++)
            for (int k = 0; k < ncol; k++) {
                EpiArgs a;
                a.b = b;
                a.d = L.A->diag;
                a.omega = h->prm.omega;
                SP_TRY(launch_csr(L.A, EPI_SOR, cur, cur, a, L.color_count[k], L.color_count[k + 1]));
            }
        return SPARSH_OK;
    }
    for (int s = 0; s < sweeps; s++) {
        if (s == 0 && zero_guess) {
            // A x = 0: x = (omega*b)/d, d read through the pattern twin when A has one (1 B per row instead of 8)
            if (jacobi_zero_pat_applies(L.A))
                SP_TRY(launch_jacobi_zero_pat(L.A, b, h->prm.omega, other));
            else
                SP_TRY(k_jacobi_zero((size_t)L.n, b, L.A->diag, h->prm.omega, other));
        } else {
            EpiArgs a;
            a.b = b;
            a.xi = cur;
            a.d = L.A->diag;
            a.omega = h->prm.omega;
            SP_TRY(launch_csr(L.A, EPI_JACOBI, cur, other, a, 0, L.n));
        }
        std::swap(cur, other);
    }
    return SPARSH_OK;
}

int enqueue_vcycle(sparsh_hierarchy_s *h, const double *b, double *x, bool x_is_zero) {
    Context &c = ctx();
    const int L = (int)h->lev.size() - 1;
    // canonical buffers at the start of every cycle (so a captured graph replays identically)
    std::vector<double *> X(L + 1), T(L + 1);
    std::vector<const double *> B(L + 1);
    for (int l = 0; l <= L; l++) {
        X[l] = l == 0 ? x : h->lev[l].xbuf;
        T[l] = h->lev[l].tbuf;
        B[l] = l == 0 ? b : h->lev[l].bbuf;
    }
    for (int l = 0; l < L; l++) {
        Level &F = h->lev[l];
        SP_TRY(smooth(h, F, B[l], X[l], T[l], h->prm.pre_sweeps, l > 0 || x_is_zero));
        if (resid_restrict_applies(F.A, F.R)) {
            // B_{l+1} = R (B_l - A X_l) in one pass: the residual is not stored (rbuf stays unwritten)
            SP_TRY(launch_resid_restrict(F.A, F.R, B[l], X[l], h->lev[l + 1].bbuf));
        } else {
            EpiArgs a;
            a.b = B[l];
            SP_TRY(launch_csr(F.A, EPI_RESID, X[l], F.rbuf, a, 0, F.n));
            SP_TRY(launch_csr(F.R, EPI_SPMV, F.rbuf, h->lev[l + 1].bbuf, EpiArgs(), 0, F.R->nrow));
        }
    }
    if (L == 0 && h->coarse.n == 0) {
        set_error("hierarchy without a coarse solver");
        return SPARSH_ERR_INVALID;
    }
    SP_TRY(coarse_apply(h->coarse, B[L], X[L]));
    for (int l = L; l > 0; l--) {
        Level &F = h->lev[l - 1];
        SP_TRY(launch_csr(F.P, EPI_PROLONG, X[l], X[l - 1], EpiArgs(), 0, F.n));
        SP_TRY(smooth(h, F, B[l - 1], X[l - 1], T[l - 1], h->prm.post_sweeps, false));
    }
    if (X[0] != x) SP_CUDA(cudaMemcpyAsync(x, X[0], sizeof(double) * (size_t)h->lev[0].n, cudaMemcpyDeviceToDevice, c.stream));
    return SPARSH_OK;
}

int krylov_workspace(sparsh_hierarchy_s *h, int nvec) {
    const size_t n = (size_t)h->lev[0].n;
    for (int i = 0; i < nvec; i++)
        if (!h->kv[i]) SP_CUDA(cudaMalloc(&h->kv[i], sizeof(double) * (n + 2)));
    return SPARSH_OK;
}

}  // namespace sparsh

extern "C" {

void sparsh_params_default(sparsh_params *p) {
    p->omega = 0.66667;  // reference include/AMG.hpp:16
    p->pre_sweeps = 7;   // smooth_iter + 1: the CPU reference's count (src/AMG_smoothers.cpp:60, SURVEY F7)
    p->post_sweeps = 7;
    p->use_graph = 1;
    p->coarse_mode = 0;
    p->smoother = 0;
    p->halo_mode = 1;
}

int sparsh_hierarchy_create(int nlevels, const sparsh_level_desc *levels, const sparsh_params *params,
                            sparsh_hierarchy_t *out) {
    SP_TRY(ensure_init());
    SP_REQUIRE(nlevels >= 1 && levels != nullptr && out != nullptr, "bad hierarchy description");
    NvtxRange nvtx("sparsh:upload");
    sparsh_hierarchy_s *h = new sparsh_hierarchy_s();
    if (params)
        h->prm = *params;
    else
        sparsh_params_default(&h->prm);
    h->lev.resize(nlevels);
    int rc = SPARSH_OK;
    // ---- validation first (sequential), then the uploads as independent tasks
    for (int l = 0; l < nlevels && rc == SPARSH_OK; l++) {
        const sparsh_level_desc &d = levels[l];
        Level &L = h->lev[l];
        L.n = d.nrow;
        if (h->prm.smoother == 1 && l < nlevels - 1) {
            if (!d.color_count || d.total_colors < 1 || d.color_count[0] != 0 || d.color_count[d.total_colors] != d.nrow) {
                set_error("multicolour smoother: level lacks a valid colour table");
                rc = SPARSH_ERR_INVALID;
                break;
            }
            L.color_count.assign(d.color_count, d.color_count + d.total_colors + 1);
        }
        if (l < nlevels - 1 && (d.p_rowptr == nullptr || d.p_ncol != levels[l + 1].nrow)) {
            set_error("prolongator missing or its column count differs from the next level's row count");
            rc = SPARSH_ERR_INVALID;
        }
    }
    // One task per operator (A_l, P_l, R_l = P_l^T incl. its host transpose), the work vectors of a level, and the
    // coarse inverse: independent, so they are spread over a few host threads, each copying on a stream of its own —
    // pageable host arrays go through the driver's staging buffers one cudaMemcpy at a time per thread, and the O(nnz)
    // host passes (validation, row statistics, transposes) overlap with the copies of the other threads.
    // SPARSH_UPLOAD_THREADS=1 restores the sequential upload.
    struct Task {
        int level, what;  // 0 A, 1 P, 2 R, 3 vectors, 4 coarse inverse
        long long weight;
    };
    std::vector<Task> tasks;
    for (int l = 0; l < nlevels; l++) {
        tasks.push_back(Task{l, 0, (long long)levels[l].nnz * 3});
        tasks.push_back(Task{l, 3, (long long)levels[l].nrow / 8});
        if (l < nlevels - 1) {
            tasks.push_back(Task{l, 1, (long long)levels[l].p_nnz * 2});
            tasks.push_back(Task{l, 2, (long long)levels[l].p_nnz * 4});
        }
    }
    tasks.push_back(Task{nlevels - 1, 4, (long long)levels[nlevels - 1].nrow * levels[nlevels - 1].nrow * 50});
    std::sort(tasks.begin(), tasks.end(), [](const Task &a, const Task &b) { return a.weight > b.weight; });
    static const bool timing = getenv("SPARSH_UPLOAD_TIMING") != nullptr;
    const auto t_begin = std::chrono::steady_clock::now();
    // One slab for everything that lives as long as the hierarchy (internal.cuh: "device memory of a hierarchy"): per CSR
    // operator the padded arrays, the diagonal, the 1-byte pattern ids and a margin for the small tables; the level
    // vectors.  A csr-dict16 twin (2 B per entry, only built where csr-pattern8 does not apply) is not counted: it and
    // anything else beyond the estimate fall through to allocations of their own.
    if (rc == SPARSH_OK) {
        auto csr_bytes = [](size_t nrow, size_t nnz) {
            return 4 * (nrow + 8) + 12 * (nnz + 16) + 8 * (nrow + 1) + (nrow + 16) + ((size_t)1 << 20) + 12 * 256;
        };
        size_t total = (size_t)1 << 20;
        for (int l = 0; l < nlevels; l++) {
            const sparsh_level_desc &d = levels[l];
            total += csr_bytes((size_t)d.nrow, (size_t)d.nnz) + 4 * (8 * ((size_t)d.nrow + 2) + 256);
            if (l < nlevels - 1) total += csr_bytes((size_t)d.nrow, (size_t)d.p_nnz) + csr_bytes((size_t)d.p_ncol, (size_t)d.p_nnz);
        }
        h->slab = slab_create(total);  // nullptr (no room for one block): individual allocations
    }
    auto run_task = [&](const Task &t) -> int {
        const sparsh_level_desc &d = levels[t.level];
        Level &L = h->lev[t.level];
        const size_t bytes = sizeof(double) * ((size_t)d.nrow + 2);
        switch (t.what) {
            case 0:
                return sparsh_matrix_create(d.nrow, d.nrow, d.nnz, d.rowptr, d.colindex, d.val, d.diag, &L.A);
            case 1:
                return sparsh_matrix_create(d.nrow, d.p_ncol, d.p_nnz, d.p_rowptr, d.p_colindex, d.p_val, nullptr, &L.P);
            case 2:
                return sparsh_matrix_create_transpose(d.nrow, d.p_ncol, d.p_nnz, d.p_rowptr, d.p_colindex, d.p_val, &L.R);
            case 3:
                SP_CUDA(dev_alloc(&L.tbuf, bytes));
                if (t.level > 0) {
                    SP_CUDA(dev_alloc(&L.xbuf, bytes));
                    SP_CUDA(dev_alloc(&L.bbuf, bytes));
                }
                if (t.level < nlevels - 1) SP_CUDA(dev_alloc(&L.rbuf, bytes));
                return SPARSH_OK;
            default:
                return coarse_build_inverse(d.nrow, d.rowptr, d.colindex, d.val, &h->coarse);
        }
    };
    if (rc == SPARSH_OK) {
        int nthreads = (int)std::min<size_t>({tasks.size(), (size_t)std::max(1u, std::thread::hardware_concurrency()), (size_t)8});
        if (const char *e = getenv("SPARSH_UPLOAD_THREADS")) nthreads = std::max(1, std::min(atoi(e), 64));
        std::atomic<size_t> next{0};
        std::atomic<int> first_rc{SPARSH_OK};
        std::mutex err_mutex;
        std::string err_msg;
        const int device = ctx().device;
        auto worker = [&](bool own_stream) {
            slab_bind(h->slab);
            cudaStream_t s = nullptr;
            if (own_stream) {
                cudaSetDevice(device);  // the runtime's current device is per host thread
                if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) == cudaSuccess) set_upload_stream(s);
            }
            for (size_t i = next++; i < tasks.size(); i = next++) {
                if (first_rc.load() != SPARSH_OK) break;
                const int trc = run_task(tasks[i]);
                if (trc != SPARSH_OK) {
                    std::lock_guard<std::mutex> g(err_mutex);
                    int expect = SPARSH_OK;
                    if (first_rc.compare_exchange_strong(expect, trc)) err_msg = sparsh_last_error();  // this thread's message
                }
            }
            if (s) {
                cudaStreamSynchronize(s);
                set_upload_stream(nullptr);
                cudaStreamDestroy(s);
            }
            if (own_stream) release_upload_stage();
            release_thread_scratch();
            slab_bind(nullptr);
        };
        std::vector<std::thread> pool;
        for (int t = 1; t < nthreads; t++) pool.emplace_back(worker, true);
        worker(nthreads > 1);  // the calling thread works too (on a stream of its own when it has company)
        for (auto &th : pool) th.join();
        rc = first_rc.load();
        if (rc != SPARSH_OK) set_error(err_msg);
        if (timing)
            std::fprintf(stderr, "[upload] %zu tasks on %d host threads: %.3f s\n", tasks.size(), nthreads,
                         std::chrono::duration<double>(std::chrono::steady_clock::now() - t_begin).count());
    }
    if (rc == SPARSH_OK && cudaMalloc(&h->d_sc, sizeof(double) * 16) != cudaSuccess) rc = SPARSH_ERR_CUDA;
    if (rc == SPARSH_OK && cudaMallocHost(&h->h_sc, sizeof(double) * 16) != cudaSuccess) rc = SPARSH_ERR_CUDA;
    if (rc != SPARSH_OK) {
        if (rc == SPARSH_ERR_CUDA) set_error(std::string("hierarchy allocation failed: ") + cudaGetErrorString(cudaGetLastError()));
        sparsh_hierarchy_destroy(h);
        return rc;
    }
    *out = h;
    return SPARSH_OK;
}

int sparsh_hierarchy_destroy(sparsh_hierarchy_t h) {
    if (!h) return SPARSH_OK;
    if (ctx().ready) cudaStreamSynchronize(ctx().stream);
    for (auto &g : h->graphs)
        if (g.exec) cudaGraphExecDestroy(g.exec);
    drop_solve_graphs(h);
    for (cudaStream_t s : h->solve_stream)
        if (s) cudaStreamDestroy(s);
    cudaFree(h->d_ctl);
    for (auto &L : h->lev) {
        sparsh_matrix_destroy(L.A);
        sparsh_matrix_destroy(L.P);
        sparsh_matrix_destroy(L.R);
        dev_free(L.xbuf);
        dev_free(L.tbuf);
        dev_free(L.bbuf);
        dev_free(L.rbuf);
    }
    coarse_free(&h->coarse);
    refresh_plan_free(h->refresh);
    for (int i = 0; i < 8; i++) cudaFree(h->kv[i]);
    cudaFree(h->d_sc);
    cudaFreeHost(h->h_sc);
    cudaFree(h->hb);
    cudaFree(h->hx);
    cudaFree(h->gm_V);
    cudaFree(h->gm_d);
    cudaFreeHost(h->gm_h);
    slab_destroy(h->slab);  // last: the matrices and level vectors above were carved from it
    delete h;
    return SPARSH_OK;
}

int sparsh_hierarchy_nlevels(sparsh_hierarchy_t h) { return h ? (int)h->lev.size() : 0; }

int sparsh_hierarchy_level(sparsh_hierarchy_t h, int level, sparsh_matrix_t *A, sparsh_matrix_t *P, sparsh_matrix_t *R) {
    SP_REQUIRE(h != nullptr && level >= 0 && level < (int)h->lev.size(), "bad level");
    if (A) *A = h->lev[level].A;
    if (P) *P = h->lev[level].P;
    if (R) *R = h->lev[level].R;
    return SPARSH_OK;
}

int sparsh_hierarchy_coarse_solve(sparsh_hierarchy_t h, const double *d_b, double *d_x) {
    SP_REQUIRE(h != nullptr, "hierarchy is NULL");
    SP_TRY(require_fresh(h));
    return coarse_apply(h->coarse, d_b, d_x);
}

int sparsh_hierarchy_vcycle(sparsh_hierarchy_t h, const double *d_b, double *d_x, int cycles, int x_is_zero) {
    SP_REQUIRE(h != nullptr && cycles >= 0, "bad arguments");
    SP_TRY(require_fresh(h));
    for (int k = 0; k < cycles; k++) {
        const bool zero = x_is_zero && k == 0;
        SP_TRY(run_graphed(h, d_b, d_x, zero ? 1 : 0, [&]() { return enqueue_vcycle(h, d_b, d_x, zero); }));
    }
    return SPARSH_OK;
}

int sparsh_hierarchy_amg_solve(sparsh_hierarchy_t h, const double *d_b, double *d_x, double tol, int max_cycles,
                               double *h_hist, int *cycles_out) {
    SP_REQUIRE(h != nullptr, "hierarchy is NULL");
    SP_TRY(require_fresh(h));
    sparsh_matrix_s *A = h->lev[0].A;
    double r1 = 0.0;
    NvtxRange nvtx("sparsh:amg-solve");
    SP_TRY(sparsh_residual_norm(A, d_b, d_x, &r1));  // reference src/AMG_phases.cpp:159
    if (h_hist) h_hist[0] = r1;
    int cycles = 0;
    while (solve_continues(cycles, max_cycles, r1, tol)) {  // :196 (the reference has no cap: SURVEY F6)
        SP_TRY(sparsh_hierarchy_vcycle(h, d_b, d_x, 1, 0));
        cycles++;
        SP_TRY(sparsh_residual_norm(A, d_b, d_x, &r1));  // :219
        if (h_hist) h_hist[cycles] = r1;
    }
    if (cycles_out) *cycles_out = cycles;
    return solve_status(r1, tol);
}

double sparsh_hierarchy_vcycle_bytes(sparsh_hierarchy_t h, int x_is_zero) {
    if (!h) return 0.0;
    const int L = (int)h->lev.size() - 1;
    double total = 0.0;
    for (int l = 0; l < L; l++) {
        const Level &F = h->lev[l];
        const double m = F.n, z = F.A->nnz, zp = F.P->nnz, mc = h->lev[l + 1].n;
        const double jac = 12.0 * z + 4.0 * (m + 1) + 32.0 * m;            // SURVEY §8d
        const double res = 12.0 * z + 4.0 * (m + 1) + 8.0 * m + 16.0 * m;
        const double rst = 12.0 * zp + 4.0 * (mc + 1) + 8.0 * m + 8.0 * mc;
        const double pro = 12.0 * zp + 4.0 * (m + 1) + 16.0 * m + 8.0 * mc;
        const bool zero = l > 0 || x_is_zero;
        double pre = h->prm.pre_sweeps * jac;
        if (zero && h->prm.pre_sweeps > 0) pre += -jac + 24.0 * m;  // first sweep is x = (omega*b)/d
        total += pre + res + rst + pro + h->prm.post_sweeps * jac;
    }
    const double nl = h->coarse.n;
    total += 8.0 * nl * nl + 16.0 * nl;
    return total;
}

}  // extern "C"

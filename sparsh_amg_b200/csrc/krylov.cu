// krylov.cu — device Krylov drivers (rows S1/S2 of SURVEY §8a).
//
// Replace Solver_CG_2, Solver_PCG_3/4 and Solver_PBiCG_3/4 (reference src/AMG_main_solvers.cu:35-763).  The arithmetic
// is that of the CPU twins Solver_CG_1, Solver_PCG_1, Solver_BiCG_1, Solver_PBiCG_1 (src/AMG_main_solvers.cpp:47-458):
// they are the runnable oracle, and the GPU twins of BiCGStab are defective (SURVEY Appendix B).
//
// Differences in mechanism, not in arithmetic:
//  * every scalar (alpha, beta, omega, dots) stays in device memory; kernels derive alpha/beta themselves, so the host
//    is synchronised once per iteration (to read ||r||) instead of once per cuBLAS dot/nrm2 call;
//  * p.Ap is fused into the SpMV, x/r updates and ||r||^2 into one pass, BiCGStab's vector triples into one pass each;
//  * r.z needed for alpha is the value already computed for the previous beta (same operands, same summation tree,
//    so bit-identical to recomputing it as the reference does, src/AMG_main_solvers.cpp:141 vs :149);
//  * the preconditioner is called with a zero initial guess, which the reference establishes with fill(z,0)
//    (src/AMG_main_solvers.cpp:146) — the fill and the first Jacobi matrix pass disappear;
//  * one iteration = one CUDA graph launch.
#include <algorithm>
#include <cmath>
#include <vector>

#include "hierarchy.cuh"

using namespace sparsh;

namespace {

// device scalar slots
// (S_RES: ||b - A x||^2 of the device-driven AMG solve)
enum { S_PAP = 0, S_RZ = 1, S_RZNEW = 2, S_RR = 3, S_A1 = 4, S_APR0 = 5, S_ASS = 6, S_ASAS = 7, S_RR0 = 8, S_RRN = 9, S_RROLD = 10,
       S_RES = 11 };

int read_scalars(sparsh_hierarchy_s *h, int first, int count) {
    Context &c = ctx();
    SP_CUDA(cudaMemcpyAsync(h->h_sc + first, h->d_sc + first, sizeof(double) * count, cudaMemcpyDeviceToHost, c.stream));
    return SPARSH_OK;
}
int sync_stream() {
    SP_CUDA(cudaStreamSynchronize(ctx().stream));
    return SPARSH_OK;
}

// A temporary hierarchy wrapper so the unpreconditioned solvers reuse the same workspace/graph machinery
struct TmpHier {
    sparsh_hierarchy_s h;
    explicit TmpHier(sparsh_matrix_s *A) {
        h.lev.resize(1);
        h.lev[0].A = A;
        h.lev[0].n = A->nrow;
        sparsh_params_default(&h.prm);
    }
    int init() {
        SP_CUDA(cudaMalloc(&h.d_sc, sizeof(double) * 16));
        SP_CUDA(cudaMallocHost(&h.h_sc, sizeof(double) * 16));
        return SPARSH_OK;
    }
    ~TmpHier() {
        if (ctx().ready) cudaStreamSynchronize(ctx().stream);
        for (auto &g : h.graphs)
            if (g.exec) cudaGraphExecDestroy(g.exec);
        for (int i = 0; i < 8; i++) cudaFree(h.kv[i]);
        cudaFree(h.d_sc);
        cudaFreeHost(h.h_sc);
        cudaFree(h.gm_V);
        cudaFree(h.gm_d);
        cudaFreeHost(h.gm_h);
        h.lev.clear();
    }
};

// ---- (P)CG -------------------------------------------------------------------------------------------------
// precond = true : Solver_PCG_1, src/AMG_main_solvers.cpp:107-167
// precond = false: Solver_CG_1,  src/AMG_main_solvers.cpp:47-103 (r = b: assumes x0 = 0, kept as in the reference)
// The work before the loop and one iteration are shared with the device-driven loop (pcg_enqueue below); `graphed`
// runs the first V-cycle through run_graphed (host loop) instead of enqueuing it into a capture already under way.
int cg_start(sparsh_hierarchy_s *h, bool precond, const double *b, double *x, bool graphed) {
    sparsh_matrix_s *A = h->lev[0].A;
    const size_t n = (size_t)A->nrow;
    double *r = h->kv[0], *z = h->kv[1], *p = h->kv[2];
    double *sc = h->d_sc;
    Context &c = ctx();
    if (precond) {
        EpiArgs a;
        a.b = b;
        SP_TRY(launch_csr(A, EPI_RESID, x, r, a, 0, A->nrow));  // :124-125
    } else {
        SP_CUDA(cudaMemcpyAsync(r, b, sizeof(double) * n, cudaMemcpyDeviceToDevice, c.stream));  // :64
    }
    SP_TRY(k_dot(n, r, r, sc + S_RR));  // :127
    if (precond) {
        if (graphed)
            SP_TRY(run_graphed(h, r, z, 1, [&]() { return enqueue_vcycle(h, r, z, true); }));  // :132 (z0 zeroed, Appendix B)
        else
            SP_TRY(enqueue_vcycle(h, r, z, true));
        SP_CUDA(cudaMemcpyAsync(p, z, sizeof(double) * n, cudaMemcpyDeviceToDevice, c.stream));  // :134
        SP_TRY(k_dot(n, r, z, sc + S_RZ));                                                       // :141 (first iteration)
    } else {
        SP_CUDA(cudaMemcpyAsync(p, r, sizeof(double) * n, cudaMemcpyDeviceToDevice, c.stream));  // :65
        SP_TRY(k_scalar_copy(sc + S_RZ, sc + S_RR));                                             // s = r.r (:76)
    }
    return SPARSH_OK;
}

// one iteration; ||r||^2 ends in sc[S_RR].  mirror: copy the scalars of the host's stopping test to h->h_sc
int cg_step(sparsh_hierarchy_s *h, bool precond, double *x, bool mirror) {
    sparsh_matrix_s *A = h->lev[0].A;
    const size_t n = (size_t)A->nrow;
    double *r = h->kv[0], *z = h->kv[1], *p = h->kv[2], *Ap = h->kv[3];
    double *sc = h->d_sc;
    EpiArgs a;
    a.xi = p;
    a.red_out = sc + S_PAP;
    SP_TRY(launch_csr(A, EPI_SPMV_DOT, p, Ap, a, 0, A->nrow));                      // :138,:140  (:73,:75)
    SP_TRY(k_pcg_update_xr(n, p, Ap, x, r, sc + S_RZ, sc + S_PAP, sc + S_RR));      // :142-145,:152
    if (precond) {
        SP_TRY(enqueue_vcycle(h, r, z, true));                                      // :146-147
        SP_TRY(k_dot(n, z, r, sc + S_RZNEW));                                       // :149
        SP_TRY(k_pcg_update_p(n, z, p, sc + S_RZNEW, sc + S_RZ));                   // :150
    } else {
        SP_TRY(k_scalar_copy(sc + S_RZNEW, sc + S_RR));                             // :82 numerator
        SP_TRY(k_cg_update_p(n, r, p, sc + S_RZNEW, sc + S_RZ));                    // :83
    }
    SP_TRY(k_scalar_copy(sc + S_RROLD, sc + S_RZ));
    SP_TRY(k_scalar_copy(sc + S_RZ, sc + S_RZNEW));
    if (mirror) {
        SP_TRY(read_scalars(h, S_RR, 1));
        SP_TRY(read_scalars(h, S_RROLD, 1));
    }
    return SPARSH_OK;
}

int cg_impl(sparsh_hierarchy_s *h, bool precond, const double *b, double *x, double tol, int max_iter, double *hist,
            int *iters_out) {
    NvtxRange nvtx(precond ? "sparsh:pcg" : "sparsh:cg");
    const size_t n = (size_t)h->lev[0].A->nrow;
    SP_TRY(krylov_workspace(h, 4));
    SP_TRY(cg_start(h, precond, b, x, true));
    SP_TRY(read_scalars(h, S_RR, 1));
    SP_TRY(sync_stream());
    double r1 = solve_residual(h->h_sc[S_RR]);
    if (hist) hist[0] = r1;

    auto body = [&]() -> int { return cg_step(h, precond, x, true); };

    const int cap = std::min((int)n, max_iter);
    int count = 0;
    while (solve_continues(count, cap, r1, tol)) {  // :136 (:70)
        count++;
        SP_TRY(run_graphed(h, x, b, precond ? 10 : 11, body));
        SP_TRY(sync_stream());
        if (precond) {
            r1 = solve_residual(h->h_sc[S_RR]);  // :152
        } else {
            const double s = h->h_sc[S_RROLD];
            const double beta = h->h_sc[S_RR] / s;  // :82
            r1 = std::sqrt(s * beta);               // :85
        }
        if (hist) hist[count] = r1;
    }
    if (iters_out) *iters_out = count;
    return solve_status(r1, tol);
}

// ---- (P)BiCGStab -----------------------------------------------------------------------------------------
// precond = true : Solver_PBiCG_1, src/AMG_main_solvers.cpp:358-458
// precond = false: Solver_BiCG_1,  src/AMG_main_solvers.cpp:271-355
// As for (P)CG, the work before the loop and one iteration are shared with the device-driven loop.
int bicg_start(sparsh_hierarchy_s *h, const double *b, double *x) {
    sparsh_matrix_s *A = h->lev[0].A;
    const size_t n = (size_t)A->nrow;
    double *r0 = h->kv[0], *r = h->kv[1], *p = h->kv[2];
    Context &c = ctx();
    EpiArgs a;
    a.b = b;
    SP_TRY(launch_csr(A, EPI_RESID, x, r0, a, 0, A->nrow));                                       // :383-384
    SP_CUDA(cudaMemcpyAsync(r, r0, sizeof(double) * n, cudaMemcpyDeviceToDevice, c.stream));      // :387
    SP_CUDA(cudaMemcpyAsync(p, r0, sizeof(double) * n, cudaMemcpyDeviceToDevice, c.stream));      // :388
    SP_TRY(k_dot(n, r0, r0, h->d_sc + S_RRN));                                                    // :390
    return SPARSH_OK;
}

// one iteration; ||r||^2 ends in sc[S_RRN].  mirror: copy it to h->h_sc
int bicg_step(sparsh_hierarchy_s *h, bool precond, double *x, bool mirror) {
    sparsh_matrix_s *A = h->lev[0].A;
    const size_t n = (size_t)A->nrow;
    double *r0 = h->kv[0], *r = h->kv[1], *p = h->kv[2], *Ap = h->kv[3], *s = h->kv[4], *As = h->kv[5];
    double *ph = precond ? h->kv[6] : p, *sh = precond ? h->kv[7] : s;
    double *sc = h->d_sc;
    if (precond) SP_TRY(enqueue_vcycle(h, p, ph, true));                     // :399-400
    SP_TRY(k_dot(n, r, r0, sc + S_A1));                                      // :402
    SP_TRY(launch_csr(A, EPI_SPMV, ph, Ap, EpiArgs(), 0, A->nrow));          // :403
    SP_TRY(k_dot(n, Ap, r0, sc + S_APR0));                                   // :404
    SP_TRY(k_bicg_s(n, r, Ap, s, sc + S_A1, sc + S_APR0));                   // :406-411
    if (precond) SP_TRY(enqueue_vcycle(h, s, sh, true));                     // :414-415
    SP_TRY(launch_csr(A, EPI_SPMV, sh, As, EpiArgs(), 0, A->nrow));          // :416
    SP_TRY(k_dot2(n, As, s, As, sc + S_ASS));                                // :418-419 (S_ASS, S_ASAS adjacent)
    SP_TRY(k_bicg_xr(n, x, ph, sh, s, As, r, sc + S_A1, sc + S_APR0, sc + S_ASS, sc + S_ASAS, r0,
                     sc + S_RR0));                                            // :424-425, dots for :428,:437
    SP_TRY(k_bicg_p(n, r, p, Ap, sc + S_A1));                                // :428-434 (slots S_A1..S_RR0 contiguous)
    if (mirror) SP_TRY(read_scalars(h, S_RRN, 1));
    return SPARSH_OK;
}

int bicg_impl(sparsh_hierarchy_s *h, bool precond, const double *b, double *x, double tol, int max_iter, double *hist,
              int *iters_out) {
    NvtxRange nvtx(precond ? "sparsh:pbicgstab" : "sparsh:bicgstab");
    SP_TRY(krylov_workspace(h, 8));
    SP_TRY(bicg_start(h, b, x));
    SP_TRY(read_scalars(h, S_RRN, 1));
    SP_TRY(sync_stream());
    double res = solve_residual(h->h_sc[S_RRN]);
    if (hist) hist[0] = res;

    auto body = [&]() -> int { return bicg_step(h, precond, x, true); };

    int count = 0;
    while (solve_continues(count, max_iter, res, tol)) {  // :397 (no cap in the reference)
        SP_TRY(run_graphed(h, x, b, precond ? 20 : 21, body));
        SP_TRY(sync_stream());
        res = solve_residual(h->h_sc[S_RRN]);     // :437
        count++;
        if (hist) hist[count] = res;
    }
    if (iters_out) *iters_out = count;
    return solve_status(res, tol);
}

// ---- GMRES(m) ----------------------------------------------------------------------------------------------
// Not in the reference (SURVEY F3: README.md:13 advertises it, no code) — SURVEY §8f.2.  Restarted GMRES, right-
// preconditioned by one V-cycle (precond) or plain; the arithmetic is the oracle's so_gmres: Arnoldi with classical
// Gram-Schmidt applied twice — two fused multi-dot passes (4 dots per sweep over w) and two fused multi-axpy passes
// instead of 2(j+1) separate dot/axpy pairs —, Givens rotations on the host from ONE device-to-host copy of the j+2
// scalars per inner iteration, x += M^-1 (V y) per cycle, true residual at every restart.  The V-cycle replays the same
// CUDA graph as PCG's (the basis vector is staged through a fixed input vector).
int gmres_impl(sparsh_hierarchy_s *h, bool precond, const double *b, double *x, double tol, int restart, int max_iter,
               double *hist, int *iters_out) {
    NvtxRange nvtx(precond ? "sparsh:pgmres" : "sparsh:gmres");
    sparsh_matrix_s *A = h->lev[0].A;
    const size_t n = (size_t)A->nrow;
    const size_t ld = (n + 3) & ~(size_t)3;  // basis vectors 32-byte aligned
    const int m = restart > 0 ? restart : 30;
    SP_REQUIRE(m <= 256, "GMRES restart length above 256");
    Context &c = ctx();
    SP_TRY(krylov_workspace(h, 3));
    double *vin = h->kv[0], *z = h->kv[1], *w = h->kv[2];
    const int HS = ((m + 1) + 3) & ~3;  // slots per coefficient vector (multi-dot writes whole groups of 4)
    const int NS = 2 * HS + 4 + m;      // [h | h2 | norm (+3 pad) | y]
    if (h->gm_m < m) {
        SP_CUDA(cudaStreamSynchronize(c.stream));
        cudaFree(h->gm_V);
        cudaFree(h->gm_d);
        cudaFreeHost(h->gm_h);
        h->gm_V = h->gm_d = h->gm_h = nullptr;
        h->gm_m = 0;
        SP_CUDA(cudaMalloc(&h->gm_V, sizeof(double) * ld * (size_t)(m + 1)));
        SP_CUDA(cudaMalloc(&h->gm_d, sizeof(double) * (size_t)NS));
        SP_CUDA(cudaMallocHost(&h->gm_h, sizeof(double) * (size_t)NS));
        h->gm_m = m;
    }
    double *V = h->gm_V, *d_h = h->gm_d, *d_h2 = h->gm_d + HS, *d_nrm = h->gm_d + 2 * HS, *d_y = h->gm_d + 2 * HS + 4;
    double *hh = h->gm_h;
    auto residual_norm2 = [&]() -> int {  // w = b - A x, *d_nrm = w.w, mirrored to the host
        EpiArgs a;
        a.b = b;
        SP_TRY(launch_csr(A, EPI_RESID, x, w, a, 0, A->nrow));
        SP_TRY(k_dot(n, w, w, d_nrm));
        SP_CUDA(cudaMemcpyAsync(hh + 2 * HS, d_nrm, sizeof(double), cudaMemcpyDeviceToHost, c.stream));
        return sync_stream();
    };
    auto precondition = [&](const double *in, double *out) -> int {  // out = M^-1 in
        SP_CUDA(cudaMemcpyAsync(vin, in, sizeof(double) * n, cudaMemcpyDeviceToDevice, c.stream));
        return run_graphed(h, vin, out, 1, [&]() { return enqueue_vcycle(h, vin, out, true); });
    };
    std::vector<double> H((size_t)(m + 1) * (size_t)m, 0.0), cs(m), sn(m), g(m + 1), y(m);
    SP_TRY(residual_norm2());
    double beta = std::sqrt(hh[2 * HS]);
    if (hist) hist[0] = beta;
    int it = 0;
    while (beta > tol && it < max_iter && std::isfinite(beta)) {
        SP_TRY(k_scale_inv_sqrt(n, w, d_nrm, V));
        g[0] = beta;
        int j = 0;
        while (j < m && it < max_iter) {
            double *vj = V + (size_t)j * ld, *vn = V + (size_t)(j + 1) * ld, *Hj = H.data() + (size_t)j * (size_t)(m + 1);
            if (precond) {
                SP_TRY(precondition(vj, z));
                SP_TRY(launch_csr(A, EPI_SPMV, z, w, EpiArgs(), 0, A->nrow));
            } else {
                SP_TRY(launch_csr(A, EPI_SPMV, vj, w, EpiArgs(), 0, A->nrow));
            }
            SP_TRY(k_mdot(n, V, ld, j + 1, w, d_h));
            SP_TRY(k_maxpy_sub(n, V, ld, j + 1, d_h, w));
            SP_TRY(k_mdot(n, V, ld, j + 1, w, d_h2));
            SP_TRY(k_maxpy_sub(n, V, ld, j + 1, d_h2, w));
            SP_TRY(k_dot(n, w, w, d_nrm));
            SP_TRY(k_scale_inv_sqrt(n, w, d_nrm, vn));
            SP_CUDA(cudaMemcpyAsync(hh, h->gm_d, sizeof(double) * (size_t)(2 * HS + 1), cudaMemcpyDeviceToHost, c.stream));
            SP_TRY(sync_stream());
            for (int i = 0; i <= j; i++) Hj[i] = hh[i] + hh[HS + i];
            const double hn = std::sqrt(hh[2 * HS]);
            Hj[j + 1] = hn;
            for (int i = 0; i < j; i++) {  // earlier rotations
                const double t = cs[i] * Hj[i] + sn[i] * Hj[i + 1];
                Hj[i + 1] = -sn[i] * Hj[i] + cs[i] * Hj[i + 1];
                Hj[i] = t;
            }
            const double den = std::sqrt(Hj[j] * Hj[j] + Hj[j + 1] * Hj[j + 1]);
            cs[j] = den > 0.0 ? Hj[j] / den : 1.0;
            sn[j] = den > 0.0 ? Hj[j + 1] / den : 0.0;
            Hj[j] = den;
            Hj[j + 1] = 0.0;
            g[j + 1] = -sn[j] * g[j];
            g[j] = cs[j] * g[j];
            const double est = std::fabs(g[j + 1]);
            j++;
            it++;
            if (hist) hist[it] = est;
            if (est <= tol || hn == 0.0 || !std::isfinite(est)) break;
        }
        for (int i = j - 1; i >= 0; i--) {  // back substitution
            double t = g[i];
            for (int k = i + 1; k < j; k++) t -= H[(size_t)k * (size_t)(m + 1) + (size_t)i] * y[k];
            y[i] = t / H[(size_t)i * (size_t)(m + 1) + (size_t)i];
        }
        if (j == 0) break;
        for (int i = 0; i < j; i++) hh[2 * HS + 4 + i] = y[i];
        SP_CUDA(cudaMemcpyAsync(d_y, hh + 2 * HS + 4, sizeof(double) * (size_t)j, cudaMemcpyHostToDevice, c.stream));
        SP_TRY(k_lincomb(n, V, ld, j, d_y, w));
        if (precond) {
            SP_TRY(precondition(w, z));
            SP_TRY(k_axpy(n, 1.0, z, x));
        } else {
            SP_TRY(k_axpy(n, 1.0, w, x));
        }
        SP_TRY(residual_norm2());
        beta = std::sqrt(hh[2 * HS]);
        if (hist) hist[it] = beta;
    }
    if (iters_out) *iters_out = it;
    return beta <= tol ? SPARSH_OK : SPARSH_ERR_NOT_CONVERGED;
}

}  // namespace

// ---- device-driven loops (sparsh_hierarchy_*_enqueue) -------------------------------------------------------------
// A solve becomes one stream-ordered piece of CUDA graph:
//   [work before the loop] -> solve_loop_begin -> WHILE { one iteration -> solve_loop_step } -> solve_loop_end
// The work before the loop and the iteration are the host loops' own (cg_start / cg_step, bicg_start / bicg_step, the
// V-cycle and residual norm of sparsh_hierarchy_amg_solve) without the copies to the host, so every kernel runs in the
// same order on the same data and x and the history come out bit-identical.  The control kernels evaluate the host
// loops' stopping rule (solve_continues) on the same device scalar and set the WHILE node's condition.  tol, the
// iteration cap, hist and status reach the loop through h->d_ctl, written by solve_loop_args before every solve: one
// cached graph per (method, b, x) serves any tol, max_iter, hist and status.
namespace sparsh {

__global__ void solve_loop_args_kernel(SolveCtl *ctl, double tol, int cap, double *hist, int *status) {
    ctl->tol = tol;
    ctl->cap = cap;
    ctl->count = 0;
    ctl->res = 0.0;
    ctl->hist = hist;
    ctl->status = status;
}
__global__ void solve_loop_begin_kernel(cudaGraphConditionalHandle cond, SolveCtl *ctl, const double *sq) {
    const double r = solve_residual(*sq);
    ctl->count = 0;
    ctl->res = r;
    if (ctl->hist) ctl->hist[0] = r;
    cudaGraphSetConditional(cond, solve_continues(0, ctl->cap, r, ctl->tol) ? 1u : 0u);
}
__global__ void solve_loop_step_kernel(cudaGraphConditionalHandle cond, SolveCtl *ctl, const double *sq) {
    const int count = ctl->count + 1;
    const double r = solve_residual(*sq);
    ctl->count = count;
    ctl->res = r;
    if (ctl->hist) ctl->hist[count] = r;
    cudaGraphSetConditional(cond, solve_continues(count, ctl->cap, r, ctl->tol) ? 1u : 0u);
}
__global__ void solve_loop_end_kernel(const SolveCtl *ctl, int kernels_per_iteration) {
    ctl->status[0] = ctl->count;
    ctl->status[1] = solve_status(ctl->res, ctl->tol);
    ctl->status[2] = ctl->count * kernels_per_iteration;
}

namespace {

int method_vectors(int m) { return m == SOLVE_PCG ? 4 : m == SOLVE_PBICGSTAB ? 8 : 0; }
// the device scalar holding the squared residual norm the stopping test reads
int method_slot(int m) { return m == SOLVE_PCG ? S_RR : m == SOLVE_PBICGSTAB ? S_RRN : S_RES; }

// ||b - A x||^2 into sc[S_RES]: sparsh_residual_norm's kernel (src/AMG_phases.cpp:159,219)
int amg_resnorm(sparsh_hierarchy_s *h, const double *b, const double *x) {
    sparsh_matrix_s *A = h->lev[0].A;
    EpiArgs a;
    a.b = b;
    a.red_out = h->d_sc + S_RES;
    return launch_csr(A, EPI_RESNORM, x, nullptr, a, 0, A->nrow);
}
int loop_start(sparsh_hierarchy_s *h, int m, const double *b, double *x) {
    if (m == SOLVE_PCG) return cg_start(h, true, b, x, false);
    if (m == SOLVE_PBICGSTAB) return bicg_start(h, b, x);
    return amg_resnorm(h, b, x);
}
int loop_step(sparsh_hierarchy_s *h, int m, const double *b, double *x) {
    if (m == SOLVE_PCG) return cg_step(h, true, x, false);
    if (m == SOLVE_PBICGSTAB) return bicg_step(h, true, x, false);
    SP_TRY(enqueue_vcycle(h, b, x, false));
    return amg_resnorm(h, b, x);
}

int launched(const char *what) {
    count_launch();
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? SPARSH_OK : cuda_fail(e, what, __FILE__, __LINE__);
}

// Records the solve on the current stream, which is being captured (into the caller's graph, or into the solve graph
// solve_enqueue builds).  The WHILE node is added to the capture's graph by hand and its body is captured on an
// internal stream straight into the node's body graph; the capture's dependencies then move past the node.
int record_solve(sparsh_hierarchy_s *h, int m, const double *b, double *x) {
    Context &c = ctx();
    const double *sq = h->d_sc + method_slot(m);
    SP_TRY(loop_start(h, m, b, x));
    cudaStreamCaptureStatus st;
    cudaGraph_t g = nullptr;
    const cudaGraphNode_t *deps = nullptr;
    size_t ndeps = 0;
    SP_CUDA(cudaStreamGetCaptureInfo(c.stream, &st, nullptr, &g, &deps, &ndeps));
    cudaGraphConditionalHandle cond;
    SP_CUDA(cudaGraphConditionalHandleCreate(&cond, g, 0, 0));
    solve_loop_begin_kernel<<<1, 1, 0, c.stream>>>(cond, h->d_ctl, sq);
    SP_TRY(launched("solve_loop_begin_kernel"));
    SP_CUDA(cudaStreamGetCaptureInfo(c.stream, &st, nullptr, &g, &deps, &ndeps));
    cudaGraphNodeParams np = {};
    np.type = cudaGraphNodeTypeConditional;
    np.conditional.handle = cond;
    np.conditional.type = cudaGraphCondTypeWhile;
    np.conditional.size = 1;
    cudaGraphNode_t loop = nullptr;
    SP_CUDA(cudaGraphAddNode(&loop, g, deps, ndeps, &np));

    cudaStream_t outer = c.stream;
    const bool outer_capturing = c.capturing;
    const long long outer_captured = c.captured;
    SP_CUDA(cudaStreamBeginCaptureToGraph(h->solve_stream[1], np.conditional.phGraph_out[0], nullptr, nullptr, 0,
                                          cudaStreamCaptureModeThreadLocal));
    c.stream = h->solve_stream[1];
    c.capturing = true;
    c.captured = 0;
    int rc = loop_step(h, m, b, x);
    if (rc == SPARSH_OK) {
        solve_loop_step_kernel<<<1, 1, 0, c.stream>>>(cond, h->d_ctl, sq);
        rc = launched("solve_loop_step_kernel");
    }
    const long long per_iteration = c.captured;
    c.stream = outer;
    c.capturing = outer_capturing;
    c.captured = outer_captured;
    cudaGraph_t body = nullptr;
    const cudaError_t e = cudaStreamEndCapture(h->solve_stream[1], &body);
    SP_TRY(rc);
    SP_CUDA(e);

    SP_CUDA(cudaStreamUpdateCaptureDependencies(c.stream, &loop, 1, cudaStreamSetCaptureDependencies));
    solve_loop_end_kernel<<<1, 1, 0, c.stream>>>(h->d_ctl, (int)per_iteration);
    return launched("solve_loop_end_kernel");
}

int solve_enqueue(sparsh_hierarchy_s *h, int m, const double *b, double *x, double tol, int max_iter, double *hist,
                  int *status) {
    SP_REQUIRE(h != nullptr && b != nullptr && x != nullptr && status != nullptr, "bad arguments");
    SP_TRY(require_fresh(h));
    static const char *const names[] = {"sparsh:pcg-enqueue", "sparsh:pbicgstab-enqueue", "sparsh:amg-solve-enqueue"};
    NvtxRange nvtx(names[m]);
    Context &c = ctx();
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    SP_CUDA(cudaStreamIsCapturing(c.stream, &cs));
    SP_REQUIRE(cs != cudaStreamCaptureStatusInvalidated, "the current stream's capture has been invalidated");
    const bool under_capture = cs == cudaStreamCaptureStatusActive;
    if (under_capture) {
        SP_REQUIRE(h->solve_warm[m],
                   "enqueued solve under stream capture: this method has not run on this hierarchy outside a capture "
                   "yet, and its first call allocates workspace and builds its graph; run it once before capturing");
    } else {
        SP_TRY(krylov_workspace(h, method_vectors(m)));
        if (!h->d_ctl) SP_CUDA(cudaMalloc(&h->d_ctl, sizeof(SolveCtl)));
        for (cudaStream_t &s : h->solve_stream)
            if (!s) SP_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    }
    const int cap = m == SOLVE_PCG ? std::min(h->lev[0].n, max_iter) : max_iter;
    solve_loop_args_kernel<<<1, 1, 0, c.stream>>>(h->d_ctl, tol, cap, hist, status);
    SP_TRY(launched("solve_loop_args_kernel"));
    if (under_capture) return record_solve(h, m, b, x);

    SolveGraph *ent = nullptr;
    for (auto &g : h->solves)
        if (g.method == m && g.b == b && g.x == x) ent = &g;
    if (!ent) {
        NvtxRange cap_range("sparsh:graph-capture");
        SolveGraph g;
        g.method = m;
        g.b = b;
        g.x = x;
        cudaStream_t outer = c.stream;
        SP_CUDA(cudaStreamBeginCapture(h->solve_stream[0], cudaStreamCaptureModeThreadLocal));
        c.stream = h->solve_stream[0];
        c.capturing = true;
        c.captured = 0;
        const int rc = record_solve(h, m, b, x);
        g.kernels = c.captured;
        c.stream = outer;
        c.capturing = false;
        cudaGraph_t graph = nullptr;
        cudaError_t e = cudaStreamEndCapture(h->solve_stream[0], &graph);
        if (rc == SPARSH_OK && e == cudaSuccess) e = cudaGraphInstantiate(&g.exec, graph, 0);
        if (graph) cudaGraphDestroy(graph);
        SP_TRY(rc);
        SP_CUDA(e);
        h->solves.push_back(g);
        ent = &h->solves.back();
    }
    SP_CUDA(cudaGraphLaunch(ent->exec, c.stream));
    c.launches += ent->kernels;
    h->solve_warm[m] = true;
    return SPARSH_OK;
}

}  // namespace

void drop_solve_graphs(sparsh_hierarchy_s *h) {
    for (auto &g : h->solves)
        if (g.exec) cudaGraphExecDestroy(g.exec);
    h->solves.clear();
    // a refresh can change kernel families: a kernel never launched before may need its first-use attributes, which
    // belongs outside a caller's capture, so every method needs a warm call again
    for (bool &w : h->solve_warm) w = false;
}

}  // namespace sparsh

extern "C" {

int sparsh_hierarchy_pcg(sparsh_hierarchy_t h, const double *d_b, double *d_x, double tol, int max_iter, double *h_hist,
                         int *iters) {
    SP_REQUIRE(h != nullptr, "hierarchy is NULL");
    SP_TRY(require_fresh(h));
    return cg_impl(h, true, d_b, d_x, tol, max_iter, h_hist, iters);
}

int sparsh_hierarchy_pbicgstab(sparsh_hierarchy_t h, const double *d_b, double *d_x, double tol, int max_iter,
                               double *h_hist, int *iters) {
    SP_REQUIRE(h != nullptr, "hierarchy is NULL");
    SP_TRY(require_fresh(h));
    return bicg_impl(h, true, d_b, d_x, tol, max_iter, h_hist, iters);
}

int sparsh_hierarchy_pcg_enqueue(sparsh_hierarchy_t h, const double *d_b, double *d_x, double tol, int max_iter,
                                 double *d_hist, int *d_status) {
    return solve_enqueue(h, SOLVE_PCG, d_b, d_x, tol, max_iter, d_hist, d_status);
}

int sparsh_hierarchy_pbicgstab_enqueue(sparsh_hierarchy_t h, const double *d_b, double *d_x, double tol, int max_iter,
                                       double *d_hist, int *d_status) {
    return solve_enqueue(h, SOLVE_PBICGSTAB, d_b, d_x, tol, max_iter, d_hist, d_status);
}

int sparsh_hierarchy_amg_solve_enqueue(sparsh_hierarchy_t h, const double *d_b, double *d_x, double tol, int max_cycles,
                                       double *d_hist, int *d_status) {
    return solve_enqueue(h, SOLVE_AMG, d_b, d_x, tol, max_cycles, d_hist, d_status);
}

int sparsh_hierarchy_pgmres(sparsh_hierarchy_t h, const double *d_b, double *d_x, double tol, int restart,
                            int max_iter, double *h_hist, int *iters) {
    SP_REQUIRE(h != nullptr, "hierarchy is NULL");
    SP_TRY(require_fresh(h));
    return gmres_impl(h, true, d_b, d_x, tol, restart, max_iter, h_hist, iters);
}

int sparsh_gmres(sparsh_matrix_t A, const double *d_b, double *d_x, double tol, int restart, int max_iter,
                 double *h_hist, int *iters) {
    SP_REQUIRE(A != nullptr && A->nrow == A->ncol, "gmres needs a square matrix");
    TmpHier t(A);
    SP_TRY(t.init());
    return gmres_impl(&t.h, false, d_b, d_x, tol, restart, max_iter, h_hist, iters);
}

int sparsh_cg(sparsh_matrix_t A, const double *d_b, double *d_x, double tol, int max_iter, double *h_hist, int *iters) {
    SP_REQUIRE(A != nullptr && A->nrow == A->ncol, "cg needs a square matrix");
    TmpHier t(A);
    SP_TRY(t.init());
    return cg_impl(&t.h, false, d_b, d_x, tol, max_iter, h_hist, iters);
}

int sparsh_bicgstab(sparsh_matrix_t A, const double *d_b, double *d_x, double tol, int max_iter, double *h_hist,
                    int *iters) {
    SP_REQUIRE(A != nullptr && A->nrow == A->ncol, "bicgstab needs a square matrix");
    TmpHier t(A);
    SP_TRY(t.init());
    return bicg_impl(&t.h, false, d_b, d_x, tol, max_iter, h_hist, iters);
}

int sparsh_hierarchy_solve_host(sparsh_hierarchy_t h, int method, const double *h_b, double *h_x, double tol,
                                int max_iter, double *h_hist, int *iters) {
    SP_REQUIRE(h != nullptr && h_b != nullptr && h_x != nullptr, "bad arguments");
    Context &c = ctx();
    const size_t bytes = sizeof(double) * (size_t)h->lev[0].n;
    if (!h->hb) SP_CUDA(cudaMalloc(&h->hb, bytes + 16));
    if (!h->hx) SP_CUDA(cudaMalloc(&h->hx, bytes + 16));
    // reference src/AMG_gpu_phases_2.cu:245-246 / src/AMG_main_solvers.cu:311-312
    SP_CUDA(cudaMemcpyAsync(h->hb, h_b, bytes, cudaMemcpyHostToDevice, c.stream));
    SP_CUDA(cudaMemcpyAsync(h->hx, h_x, bytes, cudaMemcpyHostToDevice, c.stream));
    int rc;
    if (method == 0)
        rc = sparsh_hierarchy_amg_solve(h, h->hb, h->hx, tol, max_iter, h_hist, iters);
    else if (method == 1)
        rc = sparsh_hierarchy_pcg(h, h->hb, h->hx, tol, max_iter, h_hist, iters);
    else if (method == 2)
        rc = sparsh_hierarchy_pbicgstab(h, h->hb, h->hx, tol, max_iter, h_hist, iters);
    else if (method == 3)
        rc = sparsh_hierarchy_pgmres(h, h->hb, h->hx, tol, 30, max_iter, h_hist, iters);
    else {
        set_error("unknown method");
        return SPARSH_ERR_INVALID;
    }
    if (rc != SPARSH_OK && rc != SPARSH_ERR_NOT_CONVERGED) return rc;
    // :259 / :392
    SP_CUDA(cudaMemcpyAsync(h_x, h->hx, bytes, cudaMemcpyDeviceToHost, c.stream));
    SP_CUDA(cudaStreamSynchronize(c.stream));
    return rc;
}

}  // extern "C"

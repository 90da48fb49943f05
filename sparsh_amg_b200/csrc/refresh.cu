// refresh.cu — new coefficients for a resident hierarchy with the same sparsity (sparsh_hierarchy_refresh).
//
// The prolongators P_l and R_l = P_l^T stay; every coarse operator A_{l+1} = P_l^T A_l P_l is recomputed on the device
// and written straight into the slots of the stored, column-sorted A_{l+1}: no product CSR is built and nothing is
// sorted.  The numbers are those of the host setup (host/setup.cpp: aggregation_rap, spgemm) and of rap.cu: the same
// products, added in the same order, with unfused multiply and add.  Each level's twins and kernel family are then
// chosen again (sparsh_matrix_update_values), the coarsest inverse is refactored and cached CUDA graphs are dropped
// (they carry pattern 0 and uniform values by value, and a kernel family fixed at capture).
//
// The first refresh builds a plan and keeps it.  It checks, before anything is written, that every stored A_{l+1} has
// exactly the structure of P_l^T A_l P_l and that every product row fits the kernels' lists.  A refresh that fails
// there returns SPARSH_ERR_INVALID and the hierarchy keeps its old values.  Later refreshes reuse the plan's workspace.
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <utility>

#include "hierarchy.cuh"

namespace sparsh {

namespace {

// host/setup.cpp aggregation_rap's list limits: fine rows of at most AGG_ROWMAX entries, coarse rows of at most
// AGG_SMALL; a level beyond them takes the general product, as on the host
constexpr int AGG_ROWMAX = 128, AGG_SMALL = 96;

// which of a product row's slots (positions in the stored sorted row, < TOUCHED_MAX) have been written: first touch
// stores the product, later touches add to it — the first-touch list of the host product, kept as bits in registers
constexpr int TOUCHED_MAX = 192;
static_assert(RAP_MAX_ROW <= TOUCHED_MAX && AGG_SMALL <= TOUCHED_MAX, "a product row must fit the touched bits");
struct Touched {
    unsigned long long w0 = 0ull, w1 = 0ull, w2 = 0ull;
    // marks slot s and returns whether it was marked before
    __device__ __forceinline__ bool test_set(int s) {
        const unsigned long long bit = 1ull << (s & 63);
        bool was;
        if (s < 64) {
            was = (w0 & bit) != 0ull;
            w0 |= bit;
        } else if (s < 128) {
            was = (w1 & bit) != 0ull;
            w1 |= bit;
        } else {
            was = (w2 & bit) != 0ull;
            w2 |= bit;
        }
        return was;
    }
    __device__ __forceinline__ int count() const { return __popcll(w0) + __popcll(w1) + __popcll(w2); }
};

// position of col in the sorted columns ci[lo, hi), or hi when absent
__device__ __forceinline__ int find_slot(const int *__restrict__ ci, int lo, int hi, int col) {
    int a = lo, b = hi;
    while (a < b) {
        const int m = (a + b) >> 1;
        if (ci[m] < col)
            a = m + 1;
        else
            b = m;
    }
    return a < hi && ci[a] == col ? a : hi;
}

// CHECK: the stored row c has strictly ascending columns, at most `limit` of them, and exactly the columns the product
// touches; any difference raises *fail and nothing is written.  Otherwise the product is written into the row's slots.
template <bool CHECK>
__device__ __forceinline__ bool row_ok(const int *__restrict__ cci, int lo, int len, int limit) {
    if (!CHECK) return true;
    if (len > limit) return false;
    for (int k = 1; k < len; k++)
        if (cci[lo + k - 1] >= cci[lo + k]) return false;
    return true;
}

// Aggregation product (P one entry per row: HEM), one thread per coarse row c.  The members of aggregate c are R's row c
// (ascending fine rows, R's values = P's).  Per member i, row i of A P is formed column by column in first-touch order:
// the sum over the entries of row i that fall into the same aggregate, in traversal order.  Each sum, times the entry of
// P^T, is added into the coarse row, first touch first: host/setup.cpp aggregation_rap's operations in its order.
template <bool CHECK>
__global__ void __launch_bounds__(128)
    agg_rap_kernel(int nc, const int *__restrict__ rrp, const int *__restrict__ rci, const double *__restrict__ rv,
                   const int *__restrict__ arp, const int *__restrict__ aci, const double *__restrict__ av,
                   const int *__restrict__ agg, const double *__restrict__ pv, const int *__restrict__ crp,
                   const int *__restrict__ cci, double *cv, int *fail) {
    const int c = blockIdx.x * 128 + threadIdx.x;
    if (c >= nc) return;
    const int lo = crp[c], len = crp[c + 1] - lo;
    if (!row_ok<CHECK>(cci, lo, len, AGG_SMALL)) {
        atomicExch(fail, 1);
        return;
    }
    Touched t;
    for (int m = rrp[c]; m < rrp[c + 1]; m++) {
        const int i = rci[m], a0 = arp[i], a1 = arp[i + 1];
        const double r = rv[m];
        if (CHECK && a1 - a0 > AGG_ROWMAX) {
            atomicExch(fail, 1);
            return;
        }
        for (int j = a0; j < a1; j++) {
            const int col = agg[aci[j]];
            bool seen = false;  // an earlier entry of row i opened this column of A P
            for (int q = a0; q < j && !seen; q++) seen = agg[aci[q]] == col;
            if (seen) continue;
            const int slot = find_slot(cci, lo, lo + len, col);
            if (CHECK && slot == lo + len) {
                atomicExch(fail, 1);
                return;
            }
            const bool was = t.test_set(slot - lo);
            if (!CHECK) {
                double s = __dmul_rn(av[j], pv[aci[j]]);
                for (int q = j + 1; q < a1; q++)
                    if (agg[aci[q]] == col) s = __dadd_rn(s, __dmul_rn(av[q], pv[aci[q]]));
                const double x = __dmul_rn(r, s);
                cv[slot] = was ? __dadd_rn(cv[slot], x) : x;
            }
        }
    }
    if (CHECK && t.count() != len) atomicExch(fail, 1);
}

// General product, second half: row c of R (A P), with A P from spgemm_values in the plan's workspace.  The entries of
// A P's rows are visited in their first-touch order and each product is added into its slot of the stored row: what
// spgemm_fill_kernel followed by the column sort computes (rap.cu), hence the host product's bits.
template <bool CHECK>
__global__ void __launch_bounds__(128)
    r_ap_kernel(int nc, const int *__restrict__ rrp, const int *__restrict__ rci, const double *__restrict__ rv,
                const int *__restrict__ qrp, const int *__restrict__ qci, const double *__restrict__ qv,
                const int *__restrict__ crp, const int *__restrict__ cci, double *cv, int *fail) {
    const int c = blockIdx.x * 128 + threadIdx.x;
    if (c >= nc) return;
    const int lo = crp[c], len = crp[c + 1] - lo;
    if (!row_ok<CHECK>(cci, lo, len, RAP_MAX_ROW)) {
        atomicExch(fail, 1);
        return;
    }
    Touched t;
    for (int m = rrp[c]; m < rrp[c + 1]; m++) {
        const int i = rci[m];
        const double r = rv[m];
        for (int q = qrp[i]; q < qrp[i + 1]; q++) {
            const int slot = find_slot(cci, lo, lo + len, qci[q]);
            if (CHECK && slot == lo + len) {
                atomicExch(fail, 1);
                return;
            }
            const bool was = t.test_set(slot - lo);
            if (!CHECK) {
                const double x = __dmul_rn(r, qv[q]);
                cv[slot] = was ? __dadd_rn(cv[slot], x) : x;
            }
        }
    }
    if (CHECK && t.count() != len) atomicExch(fail, 1);
}

}  // namespace

struct RefreshPlan {
    struct LevelPlan {
        bool agg = false;
        int *ap_rp = nullptr, *ap_ci = nullptr;  // general: A_l P_l, structure fixed by the plan
        double *ap_v = nullptr;
        int ap_nnz = 0;
    };
    std::vector<LevelPlan> lev;
    double *spare = nullptr;  // second n x n buffer of the coarse Gauss-Jordan
    int *piv = nullptr;
    double *d_min = nullptr;
    int *fail = nullptr;
};

void refresh_plan_free(RefreshPlan *p) {
    if (!p) return;
    for (auto &L : p->lev) {
        cudaFree(L.ap_rp);
        cudaFree(L.ap_ci);
        cudaFree(L.ap_v);
    }
    cudaFree(p->spare);
    cudaFree(p->piv);
    cudaFree(p->d_min);
    cudaFree(p->fail);
    delete p;
}

namespace {

int read_fail(const RefreshPlan *p, cudaStream_t st, bool *failed) {
    int h = 0;
    SP_CUDA(cudaGetLastError());
    SP_CUDA(cudaMemcpyAsync(&h, p->fail, sizeof(int), cudaMemcpyDeviceToHost, st));
    SP_CUDA(cudaStreamSynchronize(st));
    *failed = h != 0;
    return SPARSH_OK;
}

// A_l P_l into the plan's workspace (general levels)
int level_ap(const Level &F, const RefreshPlan::LevelPlan &lp, cudaStream_t st) {
    const sparsh_matrix_s *A = F.A, *P = F.P;
    return spgemm_values(A->nrow, A->rowptr, A->col, A->val, P->rowptr, P->col, P->val, lp.ap_rp, lp.ap_ci, lp.ap_v, st);
}

template <bool CHECK>
void launch_product(const Level &F, const sparsh_matrix_s *Ac, const RefreshPlan::LevelPlan &lp, int *fail, cudaStream_t st) {
    const sparsh_matrix_s *A = F.A, *P = F.P, *R = F.R;
    const int nc = Ac->nrow, grid = (nc + 127) / 128;
    if (nc == 0) return;
    if (lp.agg)
        agg_rap_kernel<CHECK><<<grid, 128, 0, st>>>(nc, R->rowptr, R->col, R->val, A->rowptr, A->col, A->val, P->col, P->val,
                                                    Ac->rowptr, Ac->col, Ac->val, fail);
    else
        r_ap_kernel<CHECK><<<grid, 128, 0, st>>>(nc, R->rowptr, R->col, R->val, lp.ap_rp, lp.ap_ci, lp.ap_v, Ac->rowptr,
                                                 Ac->col, Ac->val, fail);
    count_launch();
}

// plan of level l (product A_{l+1} = P^T A_l P); *valid = false when the stored A_{l+1} is not that product's structure
// or a row outgrows the lists.  Writes nothing but the plan's workspace.
int plan_level(sparsh_hierarchy_s *h, RefreshPlan *p, int l, bool *valid, cudaStream_t st) {
    const Level &F = h->lev[l];
    const sparsh_matrix_s *Ac = h->lev[l + 1].A;
    RefreshPlan::LevelPlan &lp = p->lev[l];
    *valid = false;
    if (!F.P || !F.R || F.P->ncol != Ac->nrow || F.R->nrow != Ac->nrow || F.P->nrow != F.A->nrow) return SPARSH_OK;
    bool failed = true;
    if (F.P->one_per_row) {
        lp.agg = true;
        SP_CUDA(cudaMemsetAsync(p->fail, 0, sizeof(int), st));
        launch_product<true>(F, Ac, lp, p->fail, st);
        SP_TRY(read_fail(p, st, &failed));
    }
    if (failed) {  // not an aggregation, or a row beyond aggregation_rap's lists: the general product
        lp.agg = false;
        const sparsh_matrix_s *A = F.A, *P = F.P;
        bool fits = false;
        SP_TRY(spgemm_structure(A->nrow, A->rowptr, A->col, P->rowptr, P->col, &lp.ap_rp, &lp.ap_nnz, &fits, st));
        if (!fits) return SPARSH_OK;
        SP_CUDA(cudaMalloc(&lp.ap_ci, sizeof(int) * (size_t)std::max(lp.ap_nnz, 1)));
        SP_CUDA(cudaMalloc(&lp.ap_v, sizeof(double) * (size_t)std::max(lp.ap_nnz, 1)));
        SP_TRY(level_ap(F, lp, st));
        SP_CUDA(cudaMemsetAsync(p->fail, 0, sizeof(int), st));
        launch_product<true>(F, Ac, lp, p->fail, st);
        SP_TRY(read_fail(p, st, &failed));
    }
    *valid = !failed;
    return SPARSH_OK;
}

int build_plan(sparsh_hierarchy_s *h, RefreshPlan **out) {
    cudaStream_t st = ctx().stream;
    RefreshPlan *p = new RefreshPlan();
    const int L = (int)h->lev.size() - 1;
    p->lev.resize((size_t)L);
    auto fail = [&](int rc) {
        refresh_plan_free(p);
        return rc;
    };
    if (cudaMalloc(&p->fail, sizeof(int)) != cudaSuccess) return fail(cuda_fail(cudaGetLastError(), "cudaMalloc", __FILE__, __LINE__));
    for (int l = 0; l < L; l++) {
        bool valid = false;
        const int rc = plan_level(h, p, l, &valid, st);
        if (rc != SPARSH_OK) return fail(rc);
        if (!valid) {
            set_error("hierarchy refresh: level " + std::to_string(l + 1) +
                      " is not the Galerkin product P^T A P of the level above (structure), or a product row is longer "
                      "than the device kernels' lists");
            return fail(SPARSH_ERR_INVALID);
        }
    }
    const size_t n = (size_t)h->coarse.n;
    if (n > 0 && (cudaMalloc(&p->spare, sizeof(double) * n * n) != cudaSuccess || cudaMalloc(&p->piv, sizeof(int) * n) != cudaSuccess ||
                  cudaMalloc(&p->d_min, sizeof(double)) != cudaSuccess))
        return fail(cuda_fail(cudaGetLastError(), "cudaMalloc", __FILE__, __LINE__));
    *out = p;
    return SPARSH_OK;
}

}  // namespace

int require_fresh(const sparsh_hierarchy_s *h) {
    SP_REQUIRE(!h->stale, "hierarchy is stale: its last refresh failed after writing (refresh it again)");
    return SPARSH_OK;
}

}  // namespace sparsh

using namespace sparsh;

extern "C" {

int sparsh_hierarchy_refresh(sparsh_hierarchy_t h, const double *d_val, const double *d_diag) {
    SP_TRY(ensure_init());
    SP_REQUIRE(h != nullptr && !h->lev.empty(), "hierarchy is NULL");
    SP_REQUIRE(d_val != nullptr || h->lev[0].A->nnz == 0, "values are NULL");
    NvtxRange nvtx("sparsh:refresh");
    cudaStream_t st = ctx().stream;
    // developer switch: per-level product / twin times and the inverse's on stderr (each phase synchronised)
    const bool timing = getenv("SPARSH_REFRESH_TIMING") != nullptr;
    auto now = [&]() {
        if (timing) cudaStreamSynchronize(st);
        return std::chrono::steady_clock::now();
    };
    auto secs = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
        return std::chrono::duration<double>(b - a).count();
    };
    SP_CUDA(cudaStreamSynchronize(st));  // the hierarchy is not in use while its coefficients change
    if (!h->refresh) SP_TRY(build_plan(h, &h->refresh));
    RefreshPlan *p = h->refresh;
    const int L = (int)h->lev.size() - 1;
    // from here on the hierarchy is written: until everything has succeeded it is stale
    h->stale = true;
    for (auto &g : h->graphs)
        if (g.exec) cudaGraphExecDestroy(g.exec);
    h->graphs.clear();
    drop_solve_graphs(h);
    auto t0 = now();
    SP_TRY(sparsh_matrix_update_values(h->lev[0].A, d_val, d_diag));
    if (timing) std::fprintf(stderr, "[refresh] level 0: twins %.6f s\n", secs(t0, now()));
    for (int l = 0; l < L; l++) {
        const Level &F = h->lev[l];
        sparsh_matrix_s *Ac = h->lev[l + 1].A;
        const auto ta = now();
        if (!p->lev[l].agg) SP_TRY(level_ap(F, p->lev[l], st));
        launch_product<false>(F, Ac, p->lev[l], nullptr, st);
        SP_CUDA(cudaGetLastError());
        const auto tb = now();
        SP_TRY(sparsh_matrix_update_values(Ac, Ac->val, nullptr));
        if (timing)
            std::fprintf(stderr, "[refresh] level %d: product %.6f s (%s) twins %.6f s\n", l + 1, secs(ta, tb),
                         p->lev[l].agg ? "aggregation" : "general", secs(tb, now()));
    }
    const auto tc = now();
    SP_TRY(coarse_refactor(&h->coarse, h->lev[L].A, p->spare, p->piv, p->d_min));
    SP_CUDA(cudaStreamSynchronize(st));
    if (timing) std::fprintf(stderr, "[refresh] coarse inverse (n = %d): %.6f s\n", h->coarse.n, secs(tc, now()));
    h->stale = false;
    return SPARSH_OK;
}

}  // extern "C"

// hierarchy.cuh — device-resident AMG hierarchy (replaces the device state of AMG_GPU1_solver, reference
// include/AMG_gpu_phases_2.hpp:9-40).  Everything lives in HBM for the lifetime of the handle: on a 180 GB B200 the
// reference's level streaming over PCIe ("CI", src/AMG_gpu_phases.cu:465-564) has no reason to exist.
#pragma once
#include <vector>

#include "internal.cuh"

namespace sparsh {

struct Level {
    sparsh_matrix_s *A = nullptr;  // n x n
    sparsh_matrix_s *P = nullptr;  // n x n_coarse      (null on the coarsest level)
    sparsh_matrix_s *R = nullptr;  // n_coarse x n = P^T (null on the coarsest level)
    int n = 0;
    double *xbuf = nullptr;  // solution       (levels >= 1; level 0 uses the caller's vector)
    double *tbuf = nullptr;  // Jacobi ping-pong partner
    double *bbuf = nullptr;  // right-hand side (levels >= 1)
    double *rbuf = nullptr;  // residual        (all but the coarsest)
    std::vector<int> color_count;  // multicolour smoother: prefix offsets per colour (host copy)
};

struct RefreshPlan;  // refresh.cu: per-level products and workspace of sparsh_hierarchy_refresh
void refresh_plan_free(RefreshPlan *p);

struct GraphEntry {
    const void *k0 = nullptr, *k1 = nullptr;
    int tag = 0;
    cudaGraphExec_t exec = nullptr;
    long long kernels = 0;
};

// device-driven solves (sparsh_hierarchy_*_enqueue, krylov.cu)
enum SolveMethod { SOLVE_PCG = 0, SOLVE_PBICGSTAB = 1, SOLVE_AMG = 2 };
// the loop state of an enqueued solve, in device memory: written by the argument kernel of each call, read and
// advanced by the loop's control kernels
struct SolveCtl {
    double tol;
    int cap;    // iteration limit (PCG: min(n, max_iter))
    int count;  // iterations done
    double res;  // last residual norm
    double *hist;
    int *status;
};
// one instantiated solve graph (setup, WHILE loop, epilogue) per (method, b, x)
struct SolveGraph {
    int method = 0;
    const void *b = nullptr, *x = nullptr;
    cudaGraphExec_t exec = nullptr;
    long long kernels = 0;  // kernels outside the loop (the loop's own are counted by PendingSolve.result())
};

}  // namespace sparsh

struct sparsh_hierarchy_s {
    std::vector<sparsh::Level> lev;
    sparsh_params prm;
    sparsh::CoarseInverse coarse;
    sparsh::DevSlab *slab = nullptr;  // the one device allocation behind the operators and level vectors (internal.cuh)
    // Krylov workspace on level 0 (allocated on first use) and device-resident scalars
    double *kv[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    double *d_sc = nullptr;  // 16 doubles
    double *h_sc = nullptr;  // pinned mirror
    double *hb = nullptr, *hx = nullptr;  // device staging for the host-buffer wrappers
    // GMRES(m) workspace (allocated on first use): basis, device scalars [h | h2 | norm | y], pinned mirror
    double *gm_V = nullptr, *gm_d = nullptr, *gm_h = nullptr;
    int gm_m = 0;
    std::vector<sparsh::GraphEntry> graphs;
    // device-driven solves: loop state, two internal streams (the solve graph's and its loop body's capture), the
    // cached solve graphs, and which methods have run once outside a caller's stream capture
    sparsh::SolveCtl *d_ctl = nullptr;
    cudaStream_t solve_stream[2] = {nullptr, nullptr};
    std::vector<sparsh::SolveGraph> solves;
    bool solve_warm[3] = {false, false, false};
    sparsh::RefreshPlan *refresh = nullptr;  // built by the first sparsh_hierarchy_refresh
    bool stale = false;  // a refresh failed after writing: solves return SPARSH_ERR_INVALID until one succeeds
};

namespace sparsh {

// SPARSH_ERR_INVALID (with the error message) when a failed refresh left h's coefficients inconsistent
int require_fresh(const sparsh_hierarchy_s *h);
// enqueue one V-cycle on the current stream (no host sync)
int enqueue_vcycle(sparsh_hierarchy_s *h, const double *b, double *x, bool x_is_zero);
// run `body` directly, or (params.use_graph) as a cached CUDA graph keyed by (k0,k1,tag)
template <class F>
int run_graphed(sparsh_hierarchy_s *h, const void *k0, const void *k1, int tag, F body);
int krylov_workspace(sparsh_hierarchy_s *h, int nvec);
// destroys the cached solve graphs of sparsh_hierarchy_*_enqueue and clears solve_warm (refresh, destroy)
void drop_solve_graphs(sparsh_hierarchy_s *h);

template <class F>
int run_graphed(sparsh_hierarchy_s *h, const void *k0, const void *k1, int tag, F body) {
    Context &c = ctx();
    if (!h->prm.use_graph) return body();
    GraphEntry *ent = nullptr;
    for (auto &g : h->graphs)
        if (g.k0 == k0 && g.k1 == k1 && g.tag == tag) ent = &g;
    if (!ent) {
        // first use: run directly (also performs the one-time cudaFuncSetAttribute calls outside any capture)
        GraphEntry g;
        g.k0 = k0;
        g.k1 = k1;
        g.tag = tag;
        h->graphs.push_back(g);
        return body();
    }
    if (!ent->exec) {
        NvtxRange nvtx("sparsh:graph-capture");
        cudaGraph_t graph = nullptr;
        SP_CUDA(cudaStreamBeginCapture(c.stream, cudaStreamCaptureModeThreadLocal));
        c.capturing = true;
        c.captured = 0;
        int rc = body();
        c.capturing = false;
        cudaError_t e = cudaStreamEndCapture(c.stream, &graph);
        if (rc == SPARSH_OK && e == cudaSuccess) e = cudaGraphInstantiate(&ent->exec, graph, 0);
        if (graph) cudaGraphDestroy(graph);
        if (rc != SPARSH_OK) return rc;
        SP_CUDA(e);
        ent->kernels = c.captured;
    }
    SP_CUDA(cudaGraphLaunch(ent->exec, c.stream));
    c.launches += ent->kernels;
    return SPARSH_OK;
}

}  // namespace sparsh

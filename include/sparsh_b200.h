/*
 * sparsh_b200.h — C-ABI of the B200-native AMG solve phase (libsparsh_b200.so).
 *
 * This is the drop-in boundary.  The reference (cmgcds/SParSH-AMG) has no FFI layer: its host C++
 * (src/AMG_main_solvers.cpp, src/AMG_main_solvers.cu, src/AMG_gpu_phases*.cu) reaches the GPU through the
 * class sp_matrix_gpu and through direct cuSPARSE/cuBLAS/thrust calls.  Every entry point below names the
 * reference interface (file:line, relative to /root/reference) it replaces.  INTEGRATION.md shows the
 * reference-side code that binds to it.
 *
 * Conventions
 *  - plain C, no C++/torch/AMG.hpp types; `int` status return (0 = SPARSH_OK), message via sparsh_last_error()
 *  - matrices are the reference's 0-based int32/fp64 CSR (include/AMG_matrix.hpp:6-32)
 *  - `const double *d_*` / `double *d_*` arguments are DEVICE pointers, `h_*` are HOST pointers
 *  - everything is stream-ordered on the library's current stream (sparsh_set_stream / sparsh_get_stream);
 *    calls that return a scalar to the host synchronise that stream
 *  - fp64 throughout, no tensor cores, no cuSPARSE/cuBLAS, no CPU fallback: a missing GPU is an error
 *  - one handle per host thread (the reference is not re-entrant either: SURVEY §8b)
 */
#ifndef SPARSH_B200_H_
#define SPARSH_B200_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPARSH_OK 0
#define SPARSH_ERR_CUDA 1
#define SPARSH_ERR_INVALID 2
#define SPARSH_ERR_NOT_CONVERGED 3
#define SPARSH_ERR_NO_DEVICE 4

typedef struct sparsh_matrix_s *sparsh_matrix_t;       /* replaces class sp_matrix_gpu (include/AMG_gpu_matrix.hpp:10-48) */
typedef struct sparsh_hierarchy_s *sparsh_hierarchy_t; /* replaces the device state of AMG_GPU1_solver / AMG_GPU_solver
                                                          (include/AMG_gpu_phases_2.hpp:9-40, AMG_gpu_phases.hpp:10-55) */

/* ------------------------------------------------------------------ runtime ---- */
int sparsh_init(int device);               /* cudaSetDevice + library stream; idempotent */
int sparsh_shutdown(void);
const char *sparsh_last_error(void);
int sparsh_set_stream(void *cuda_stream);  /* adopt a caller stream (cudaStream_t); NULL restores the library's own */
int sparsh_get_stream(void **cuda_stream);
int sparsh_sync(void);                     /* replaces the cudaStreamSynchronize/cudaDeviceSynchronize pairs, e.g.
                                              src/AMG_gpu_phases_2.cu:106-108 */
int sparsh_device_name(char *buf, size_t len, int *sm_count);
/* number of kernels this library has launched since the last reset (graph replays count their kernel nodes) */
long long sparsh_launch_count(void);
void sparsh_launch_count_reset(void);
/* adds kernels run that the library could not count without a host read: the loop of an enqueued solve (d_status[2]) */
void sparsh_launch_count_add(long long kernels);

/* ------------------------------------------------------------------ memory ----- */
/* replace cudaMalloc / cudaMemcpy / thrust::fill of src/AMG_gpu_phases_2.cu:17-29,127,245-246,259 */
int sparsh_malloc(size_t bytes, void **d_ptr);
int sparsh_free(void *d_ptr);
int sparsh_host_alloc(size_t bytes, void **h_ptr); /* pinned; replaces cudaHostRegister pinning,
                                                      src/AMG_gpu_phase_utilities.cu:11-67 */
int sparsh_host_free(void *h_ptr);
int sparsh_memcpy_h2d(void *d_dst, const void *h_src, size_t bytes);
int sparsh_memcpy_d2h(void *h_dst, const void *d_src, size_t bytes);
int sparsh_memcpy_d2d(void *d_dst, const void *d_src, size_t bytes);
int sparsh_fill(double *d_x, size_t n, double value);

/* ------------------------------------------------------------------ matrix ----- */
/* sp_matrix_gpu::sp_matrix_gpu + matrix_transfer_gpu (src/AMG_gpu_matrix.cu:26-102): upload a host CSR.
 * h_diag may be NULL: the diagonal is then extracted like sp_matrix_fill_diagonal (src/AMG_cpu_matrix.cpp:35-51). */
int sparsh_matrix_create(int nrow, int ncol, int nnz, const int *h_rowptr, const int *h_colindex,
                         const double *h_val, const double *h_diag, sparsh_matrix_t *out);
/* New values for a matrix whose sparsity is unchanged.  d_val[nnz] is on the device, in the stored entry order.
 * d_diag[nrow] may be NULL: the diagonal is then extracted like sp_matrix_fill_diagonal.  Every value-derived choice
 * is made again exactly as sparsh_matrix_create makes it for the same arrays.  That covers the diagonal, the
 * csr-pattern8 and csr-dict16 twins with Pat0 and its masks, the kernel family and the transfer flags, under every
 * SPARSH_PATTERN / SPARSH_DICT setting.  A kernel forced with sparsh_matrix_force_kernel is forgotten.  The encoders'
 * device scratch stays with the calling thread, so later updates of the same sizes allocate nothing. */
int sparsh_matrix_update_values(sparsh_matrix_t A, const double *d_val, const double *d_diag);
/* Copy a device matrix back to the host.  Any pointer may be NULL (that array is skipped).
 * Sizes: rowptr[nrow+1], colindex[nnz], val[nnz], diag[nrow]. */
int sparsh_matrix_fetch(sparsh_matrix_t A, int *h_rowptr, int *h_colindex, double *h_val, double *h_diag);
/* explicit R = P^T (stable: each R row lists fine rows ascending), built once; replaces the transposed csrmv of
 * src/AMG_gpu_phases_2.cu:125,186 / src/AMG_gpu_phases.cu:512 with a deterministic gather */
int sparsh_matrix_create_transpose(int nrow, int ncol, int nnz, const int *h_rowptr, const int *h_colindex,
                                   const double *h_val, sparsh_matrix_t *out);
int sparsh_matrix_destroy(sparsh_matrix_t A); /* sp_matrix_gpu::~sp_matrix_gpu (src/AMG_gpu_matrix.cu:131-142) */
int sparsh_matrix_dims(sparsh_matrix_t A, int *nrow, int *ncol, int *nnz);
/* kernel family chosen at upload: 0 scalar (<=2.5 nnz/row), 1 stream (TMA-staged, thread per row), 2 vector
 * (sub-warp per row), 3 dict (stream kernel over the csr-dict16 twin below, when that twin exists), 4 pattern
 * (csr-pattern8 twin below, preferred over dict when the rows repeat; SPARSH_PATTERN=0 disables it, =2 builds the twin
 * without selecting it).
 * sparsh_matrix_force_kernel overrides it (tests exercise every family). */
int sparsh_matrix_kernel(sparsh_matrix_t A, int *kind, int *threads_or_lanes, int *smem_bytes);
int sparsh_matrix_force_kernel(sparsh_matrix_t A, int kind, int threads_or_lanes);
/* name of the kernel instantiation the library launches for this matrix and epilogue (0 SpMV, 1 residual, 2 Jacobi,
 * 3 prolongation-correction, 4 SOR colour, 5 SpMV+dot, 6 residual norm): for reports */
int sparsh_matrix_kernel_name(sparsh_matrix_t A, int epilogue, char *buf, size_t len);

/* csr-dict16, the lossless storage the stream kernel prefers: entry j of row i is stored as the 16-bit code
 * (vi << 8) | oi with val[j] == dict_val[vi] (compared by bit pattern) and colindex[j] == i + dict_off[oi]; rowptr is
 * kept.  Exists iff the matrix has <= 256 distinct values and <= 256 distinct (column - row) offsets (constant-
 * coefficient stencils and their Galerkin coarse operators); otherwise plain CSR is used.  No counterpart in the
 * reference (it stores CSR only, src/AMG_gpu_matrix.cu:26-102); results are bit-identical to the CSR kernels'.
 * Host-only helper (needs no GPU), so the encoding can be checked anywhere: code[nnz], dict_val[256], dict_off[256];
 * *n_val == 0 on return means "not representable". */
int sparsh_dict_encode(int nrow, int ncol, int nnz, const int *h_rowptr, const int *h_colindex, const double *h_val,
                       unsigned short *code, double *dict_val, int *dict_off, int *n_val, int *n_off);

/* csr-pattern8, one byte per ROW: rows of stencil matrices and of their Galerkin coarse operators repeat a few
 * patterns (the ordered list of (column - row, value) pairs; 27 per level in the 7-point Poisson hierarchy).  pat[i] <
 * 255 selects entries start[p] .. start[p+1] of the table, pat[i] == 255 is the escape: the row is evaluated from the
 * CSR arrays, which stay resident.  Patterns are numbered by decreasing row count.  Same entries, same order, same
 * arithmetic: bit-identical to the CSR kernels.  h_diag (may be NULL) is the diagonal the caller smooths with; rows
 * where it differs from the tabulated diagonal become escapes.  Host-only helper (needs no GPU): pat[nrow],
 * ent_val/ent_off[2048], start[256]; *n_pat == 0 on return means "rows do not repeat" (more than 65536 distinct rows). */
int sparsh_pattern_encode(int nrow, int ncol, int nnz, const int *h_rowptr, const int *h_colindex,
                          const double *h_val, const double *h_diag, unsigned char *pat, double *ent_val,
                          int *ent_off, int *start, int *n_pat, int *n_escape);

/* what the upload built (the encoder runs on the DEVICE there; it must agree with sparsh_pattern_encode): number of
 * patterns (0: no twin), table entries, escape rows, fraction of the rows that carry pattern 0 */
int sparsh_matrix_pattern_stats(sparsh_matrix_t A, int *n_pat, int *n_ent, int *n_escape, double *cover0);

/* The row-sum kernel for matrices that mostly repeat pattern 0 (csr_pat2_kernel) evaluates a row of another pattern as
 * pattern 0 with terms left out when that pattern's (offset, value bits) list is an in-order subsequence of pattern
 * 0's and its diagonal (first offset-0 entry, else 0) has pattern 0's bits: the Dirichlet boundary rows of a stencil
 * and their Galerkin coarsenings.  Host-only helper (needs no GPU) over a table as sparsh_pattern_encode returns it:
 * mask[256] receives, per pattern id, 0x80 | (bit k set when the pattern has entry k of pattern 0), or 0 when the
 * pattern is not such a subsequence.  Pattern 0 has every bit set when it has at most 7 entries; otherwise, and for
 * ids >= n_pat, every mask is 0. */
int sparsh_pattern_masks(int n_pat, const int *start, const double *ent_val, const int *ent_off, unsigned char *mask);
/* what the upload built: patterns other than pattern 0 that run as masked pattern 0, and the fraction of the rows that
 * carry pattern 0 or one of those patterns */
int sparsh_matrix_pattern_mask_stats(sparsh_matrix_t A, int *n_masked, double *cover_masked);

/* Grid-transfer structure found at upload: *one_per_row = 1 when every row stores exactly one entry (rowptr[i] == i),
 * *uniform_val = 1 when every stored value has the same bit pattern, *value (0 otherwise).  HEM's P has both, its
 * R = P^T uniform values only.  A scalar-family matrix with one entry per row runs SpMV and prolongation with the
 * aggregation kernel (no rowptr read, no val read when uniform); forcing KIND_SCALAR selects the plain scalar kernel. */
int sparsh_matrix_transfer_info(sparsh_matrix_t A, int *one_per_row, int *uniform_val, double *value);

/* ------------------------------------------------------------------ setup ------ */
/* Galerkin product A_c = P^T (A P) on the device (SURVEY 8f.1): what parallel::coarsen_matrix does with two
 * mkl_sparse_spmm calls on the host (src/AMG_cycle_utilities.cpp:126-146).  Row-wise products with the host setup's
 * traversal order and unfused arithmetic, columns sorted: row pointers and column indices equal the reference's, values
 * equal this repository's host product bit for bit.  On return *out holds the product on the device and *nnz_coarse its
 * entry count; *out == NULL with SPARSH_OK means "not applicable" (a product row longer than the kernel's per-thread
 * list: use the host product).  sparsh_rap_fetch copies it into caller arrays (rowptr[ncoarse+1], colindex, val).
 * sparsh_galerkin_rap_next computes the next level's product with the fine matrix taken from `fine`, a product that is
 * still on the device (the coarse matrix of one level is the fine matrix of the next: only P is uploaded). */
typedef struct sparsh_rap_s *sparsh_rap_t;
int sparsh_galerkin_rap(int nrow, const int *h_rowptr, const int *h_colindex, const double *h_val, int ncoarse,
                        const int *h_p_rowptr, const int *h_p_colindex, const double *h_p_val, sparsh_rap_t *out,
                        int *nnz_coarse);
int sparsh_galerkin_rap_next(sparsh_rap_t fine, int ncoarse, const int *h_p_rowptr, const int *h_p_colindex,
                             const double *h_p_val, sparsh_rap_t *out, int *nnz_coarse);
int sparsh_rap_fetch(sparsh_rap_t h, int *h_rowptr, int *h_colindex, double *h_val);
int sparsh_rap_destroy(sparsh_rap_t h);

/* ------------------------------------------------------------------ per-op ----- */
/* K9  y = A x                              cusparseDcsrmv, e.g. src/AMG_main_solvers.cu:100,221,354 */
int sparsh_spmv(sparsh_matrix_t A, const double *d_x, double *d_y);
/* K9+K8  y = A x and *d_dot = x . y fused   csrmv + cublasDdot, src/AMG_main_solvers.cu:354-357 */
int sparsh_spmv_dot(sparsh_matrix_t A, const double *d_x, double *d_y, double *d_dot);
/* K2  r = b - A x                          csrmv(-1)+daxpy, src/AMG_gpu_phases_2.cu:181-183;
 *                                          parallel::store_residual, src/AMG_cycle_utilities.cpp:115-123 */
int sparsh_residual(sparsh_matrix_t A, const double *d_b, const double *d_x, double *d_r);
/* K3  *h_norm = ||A x - b||_2 (nothing stored)   residual(), src/AMG_gpu_phase_utilities.cu:138-167;
 *                                          parallel::residual, src/AMG_cycle_utilities.cpp:83-94 */
int sparsh_residual_norm(sparsh_matrix_t A, const double *d_b, const double *d_x, double *h_norm);
/* K1  `sweeps` fused weighted-Jacobi sweeps x <- x + (omega*(b - A x))/d, result left in d_x; d_tmp is an
 * nrow scratch vector.                     sp_matrix_gpu::smooth_jacobi + jacobi_update, src/AMG_gpu_matrix.cu:15-22,
 *                                          106-127; parallel::jacobi_smoother, src/AMG_smoothers.cpp:53-76
 * (the CPU reference runs smooth_iter+1 = 7 sweeps, the GPU reference 6: SURVEY F7 — the count is an argument) */
int sparsh_jacobi(sparsh_matrix_t A, const double *d_b, double *d_x, double *d_tmp, double omega, int sweeps);
/* K1 from x = 0: x = (omega*b)/d, d the matrix' smoothing diagonal (A x = 0 needs no matrix pass).  With the lean
 * csr-pattern8 kernel d is read through the pattern twin (1 B per row); the same bits either way. */
int sparsh_jacobi_zero(sparsh_matrix_t A, const double *d_b, double omega, double *d_x);
/* K6  multicolour SOR on a colour-permuted matrix: for each colour k, rows h_color_count[k]..[k+1] updated in
 * place, x_l -= (omega*(sum_j a_lj x_j - b_l))/d_l.   parallel::sor_smoother, src/AMG_smoothers.cpp:78-102 (no GPU
 * version exists in the reference: "SOR ... to be defined", src/AMG_gpu_matrix.cu:129) */
int sparsh_mc_sor(sparsh_matrix_t A, const int *h_color_count, int total_colors, const double *d_b, double *d_x,
                  double omega, int sweeps);
/* K4  bc = R r with R = P^T explicit       transposed csrmv, src/AMG_gpu_phases_2.cu:186;
 *                                          parallel::transfer_residual, src/AMG_cycle_utilities.cpp:97-104 */
int sparsh_restrict(sparsh_matrix_t R, const double *d_r, double *d_bc);
/* K5  xf += P xc                            csrmv beta=1, src/AMG_gpu_phases_2.cu:210;
 *                                          parallel::transfer_solution, src/AMG_cycle_utilities.cpp:107-112 */
int sparsh_prolong_add(sparsh_matrix_t P, const double *d_xc, double *d_xf);
/* K2+K4  bc = R (b - A x), the V-cycle's residual and restriction.  One fused pass when A runs the lean csr-pattern8
 * kernel and R's values are uniform (HEM): the residual is neither stored nor read back.  Otherwise sparsh_residual
 * into a temporary followed by sparsh_restrict (synchronous).  Bit-identical to the two calls either way. */
int sparsh_residual_restrict(sparsh_matrix_t A, sparsh_matrix_t R, const double *d_b, const double *d_x, double *d_bc);

/* K8  BLAS-1 (replace cublasDdot/Dnrm2/Daxpy and the kernels daxpby/daxpbyc, src/AMG_main_solvers.cu:17-33).
 * Reductions are two-stage with a fixed tree: bit-reproducible run to run. */
int sparsh_dot(size_t n, const double *d_x, const double *d_y, double *h_out);
int sparsh_nrm2(size_t n, const double *d_x, double *h_out);
/* the same reduction with the result left in DEVICE memory and no host synchronisation (cublasDdot under
 * CUBLAS_POINTER_MODE_DEVICE; the Krylov drivers use this form internally, src/AMG_main_solvers.cu:357 syncs instead) */
int sparsh_dot_device(size_t n, const double *d_x, const double *d_y, double *d_out);
int sparsh_axpy(size_t n, double a, const double *d_x, double *d_y);                 /* y += a x          */
int sparsh_axpby(size_t n, double a, const double *d_x, double b, double *d_y);      /* y = a x + b y     */
int sparsh_axpbypcz(size_t n, double a, const double *d_x, double b, const double *d_y, double c,
                    double *d_z);                                                   /* z = a x + b y + c z */

/* ------------------------------------------------------------------ hierarchy -- */
typedef struct {
    /* A_l (square) */
    int nrow, nnz;
    const int *rowptr, *colindex;
    const double *val, *diag; /* diag may be NULL */
    /* P_l : nrow x p_ncol, NULL/0 on the coarsest level */
    int p_ncol, p_nnz;
    const int *p_rowptr, *p_colindex;
    const double *p_val;
    /* multicolour smoother only (params.smoother == 1): A_l is colour-permuted, rows color_count[k]..color_count[k+1]
     * share colour k (sp_matrix_mg::color_count / total_colors, include/AMG_cpu_matrix.hpp:24-26).  NULL/0 otherwise. */
    int total_colors;
    const int *color_count;
} sparsh_level_desc;

typedef struct {
    double omega;     /* include/AMG.hpp:16   (0.66667)                                          */
    int pre_sweeps;   /* Jacobi sweeps before restriction: 7 = CPU reference, 6 = GPU reference  */
    int post_sweeps;  /* Jacobi sweeps after prolongation                                        */
    int use_graph;    /* capture V-cycle / Krylov iterations into CUDA graphs (1) or launch directly (0) */
    int coarse_mode;  /* 0: dense inverse formed on the device at setup, applied as a GEMV (K7)  */
    int smoother;     /* 0: weighted Jacobi (AMG_solve_jacobi, src/AMG_phases.cpp:151-230)
                         1: multicolour SOR  (AMG_solve_SOR,   src/AMG_phases.cpp:234-306); pre/post_sweeps then count
                            SOR sweeps (the reference hard-codes 6, src/AMG_phases.cpp:251,265) */
    int halo_mode;    /* multi-GPU only.  1 (default): boundary entries are stored straight into the neighbour's halo
                         segment over NVLink peer memory by the packing kernel, with flag handshakes in device memory
                         (no NCCL call on the exchange path); 0: grouped ncclSend/ncclRecv */
} sparsh_params;
void sparsh_params_default(sparsh_params *p);

/* AMG_GPU1_solver::GPU_Allocations (src/AMG_gpu_phases_2.cu:13-94): upload every A_l, P_l once, build R_l = P_l^T,
 * factor the coarsest level (Direct_Solver_Pardiso ctor, src/AMG_coarse_level_solver.cpp:9-62, done on the device). */
int sparsh_hierarchy_create(int nlevels, const sparsh_level_desc *levels, const sparsh_params *params,
                            sparsh_hierarchy_t *out);
/* New values for level 0 of a hierarchy, same sparsity (d_val[nnz] on the device in the stored order: for a
 * multicolour-SOR hierarchy the colour-permuted order, as at create; d_diag[nrow] may be NULL).  P_l and R_l are kept.
 * For every level, A_{l+1} = P_l^T A_l P_l is recomputed on the device, bit for bit what the host setup computes for the
 * same P.  Coarse diagonals are extracted; each level is then updated as by sparsh_matrix_update_values.  The coarsest
 * inverse is refactored (in place: it keeps its device address) and the library's cached CUDA graphs are dropped.
 * A CUDA graph of the CALLER's that holds an enqueued solve (sparsh_hierarchy_*_enqueue) or a V-cycle must be captured
 * again after a refresh, successful or not: kernel choices, by-value launch arguments and twin arrays change, and a
 * replay of the old graph computes with stale ones (wrong results, no error code).  A captured
 * sparsh_hierarchy_coarse_solve stays valid.  After a refresh each enqueued method needs one call outside a capture
 * again before it may be captured.
 * The first call builds and keeps a plan: SPARSH_ERR_INVALID, with nothing written, when a stored A_{l+1} does not have
 * exactly the structure of P_l^T A_l P_l or a product row is longer than the device kernels' lists.  When the coarsest
 * matrix turns out singular or a CUDA error occurs after writing began, that error is returned and the hierarchy is
 * stale: V-cycles, solves and coarse solves return SPARSH_ERR_INVALID until a later refresh succeeds. */
int sparsh_hierarchy_refresh(sparsh_hierarchy_t h, const double *d_val, const double *d_diag);
int sparsh_hierarchy_destroy(sparsh_hierarchy_t h); /* AMG_GPU1_solver::~AMG_GPU1_solver, src/AMG_gpu_phases_2.cu:265-338 */
int sparsh_hierarchy_nlevels(sparsh_hierarchy_t h);
/* borrow the device matrices of one level (for per-op parity tests); P and R are NULL on the coarsest level */
int sparsh_hierarchy_level(sparsh_hierarchy_t h, int level, sparsh_matrix_t *A, sparsh_matrix_t *P,
                           sparsh_matrix_t *R);
/* K7  x = A_L^{-1} b on the coarsest level   Direct_Solver_Pardiso_solve, src/AMG_coarse_level_solver.cpp:64-76 (host
 * PARDISO + 2 PCIe hops per cycle in the reference, src/AMG_gpu_phases_2.cu:192-203) */
int sparsh_hierarchy_coarse_solve(sparsh_hierarchy_t h, const double *d_b, double *d_x);
/* V  exactly `cycles` V(pre,post)-cycles on device b, x (x in/out).  AMG_GPU1_solver::AMG_Solve(b,x,iterations>0),
 * src/AMG_gpu_phases_2.cu:109-170; AMG_solver::AMG_solve_jacobi(b,x,k), src/AMG_phases.cpp:163-192.
 * x_is_zero != 0 promises x == 0 on entry (preconditioner use): the first pre-sweep then needs no matrix pass. */
int sparsh_hierarchy_vcycle(sparsh_hierarchy_t h, const double *d_b, double *d_x, int cycles, int x_is_zero);
/* AMG as a solver: V-cycles until ||A x - b||_2 <= tol (absolute, as the reference) or max_cycles.
 * AMG_Solve(b,x,-1), src/AMG_gpu_phases_2.cu:171-236; AMG_solve_jacobi(b,x,-1), src/AMG_phases.cpp:194-226.
 * h_hist (may be NULL) receives hist[0] = initial residual, hist[k] = residual after cycle k (max_cycles+1 slots). */
int sparsh_hierarchy_amg_solve(sparsh_hierarchy_t h, const double *d_b, double *d_x, double tol, int max_cycles,
                               double *h_hist, int *cycles);
/* S1  AMG-preconditioned CG on the device.  Solver_PCG_4 / Solver_PCG_3 (src/AMG_main_solvers.cu:142-413) with the
 * arithmetic of Solver_PCG_1 (src/AMG_main_solvers.cpp:107-167).  hist[0] = ||b - A x0||, hist[k] after iteration k. */
int sparsh_hierarchy_pcg(sparsh_hierarchy_t h, const double *d_b, double *d_x, double tol, int max_iter,
                         double *h_hist, int *iters);
/* S2  AMG-preconditioned BiCGStab.  Solver_PBiCG_3/4 (src/AMG_main_solvers.cu:416-763) with the arithmetic of
 * Solver_PBiCG_1 (src/AMG_main_solvers.cpp:358-458; the GPU twins are defective, SURVEY Appendix B). */
int sparsh_hierarchy_pbicgstab(sparsh_hierarchy_t h, const double *d_b, double *d_x, double tol, int max_iter,
                               double *h_hist, int *iters);
/* Unpreconditioned twins: Solver_CG_2 (src/AMG_main_solvers.cu:35-139; arithmetic of Solver_CG_1,
 * src/AMG_main_solvers.cpp:47-103, which assumes x0 = 0) and Solver_BiCG_1 (src/AMG_main_solvers.cpp:271-355). */
int sparsh_cg(sparsh_matrix_t A, const double *d_b, double *d_x, double tol, int max_iter, double *h_hist,
              int *iters);
int sparsh_bicgstab(sparsh_matrix_t A, const double *d_b, double *d_x, double tol, int max_iter, double *h_hist,
                    int *iters);
/* Restarted GMRES(restart), right-preconditioned by one V-cycle (sparsh_hierarchy_pgmres) or plain (sparsh_gmres).
 * No counterpart in the reference: README.md:13 advertises GMRES, the sources have none (SURVEY F3, §8f.2).  Arnoldi
 * with classical Gram-Schmidt applied twice (fused multi-dot / multi-axpy kernels), Givens rotations on the host.
 * restart <= 0 means 30; at most 256.  hist[0] = ||b - A x0||, hist[k] = residual-norm estimate after k inner
 * iterations, the entry of the last iteration of each cycle replaced by the true residual norm (max_iter+1 slots). */
int sparsh_hierarchy_pgmres(sparsh_hierarchy_t h, const double *d_b, double *d_x, double tol, int restart,
                            int max_iter, double *h_hist, int *iters);
int sparsh_gmres(sparsh_matrix_t A, const double *d_b, double *d_x, double tol, int restart, int max_iter,
                 double *h_hist, int *iters);
/* Host-buffer wrappers (the reference's AMG_GPU1_solver::helper, src/AMG_gpu_phases_2.cu:242-263, and the
 * cudaMemcpy prologue/epilogue of Solver_PCG_4, src/AMG_main_solvers.cu:311-312,392): H2D of b and x, solve,
 * D2H of x.  method: 0 = AMG as solver, 1 = PCG, 2 = PBiCGStab, 3 = PGMRES(30). */
int sparsh_hierarchy_solve_host(sparsh_hierarchy_t h, int method, const double *h_b, double *h_x, double tol,
                                int max_iter, double *h_hist, int *iters);
/* bytes moved by one V-cycle according to the algorithmic model of SURVEY §8d (for roofline reports) */
double sparsh_hierarchy_vcycle_bytes(sparsh_hierarchy_t h, int x_is_zero);

/* ---------------------------------------------------- device-driven hierarchy solvers -- */
/* Device-driven twins of sparsh_hierarchy_pcg / _pbicgstab / _amg_solve: the same kernels in the same order, so x and
 * the residual history are bit-identical to theirs.  The iteration loop and its stopping test run on the device (a
 * conditional WHILE node of a CUDA graph).  The call only enqueues work on the library's current stream: it never
 * synchronises, allocates or copies to the host once the hierarchy has run the same method once.  If that stream is
 * being captured by the caller, the solve is recorded into the caller's graph.
 * Results are in DEVICE memory: d_hist[max_iter+1] (may be NULL) as h_hist of the synchronous call;
 * d_status[0] = iterations (cycles), d_status[1] = SPARSH_OK or SPARSH_ERR_NOT_CONVERGED, d_status[2] = kernels the
 * loop ran (d_status has 3 slots).
 * The return code covers what the host can see: bad arguments, a stale hierarchy, CUDA errors, and SPARSH_ERR_INVALID
 * for a call under stream capture before the method has run once on this hierarchy outside a capture (that first call
 * allocates workspace and builds the solve graph, which a capture forbids).  One instantiated graph is cached per
 * (method, d_b, d_x) address pair and kept until sparsh_hierarchy_refresh or _destroy: a caller that solves every step
 * reuses its b and x buffers (new addresses each step would build and keep a graph per call).
 * A graph of the caller's into which a solve was captured is valid until the next sparsh_hierarchy_refresh of h,
 * successful or not: after it, capture the solve again (see sparsh_hierarchy_refresh), and run the method once outside
 * a capture first.  b, x, the workspace and the device scalars are read when the work runs, not when it is enqueued:
 * do not start another solve on the same hierarchy on a different stream before this one has finished.
 * sparsh_launch_count: the kernels outside the loop count when the call enqueues them (under a caller's capture: once,
 * when captured); the loop's kernels, unknown to the host, count when the caller adds d_status[2] with
 * sparsh_launch_count_add (PendingSolve.result() in the Python package does). */
int sparsh_hierarchy_pcg_enqueue(sparsh_hierarchy_t h, const double *d_b, double *d_x, double tol, int max_iter,
                                 double *d_hist, int *d_status);
int sparsh_hierarchy_pbicgstab_enqueue(sparsh_hierarchy_t h, const double *d_b, double *d_x, double tol, int max_iter,
                                       double *d_hist, int *d_status);
int sparsh_hierarchy_amg_solve_enqueue(sparsh_hierarchy_t h, const double *d_b, double *d_x, double tol, int max_cycles,
                                       double *d_hist, int *d_status);

/* ------------------------------------------------------------------ multi-GPU -- */
/* One process per GPU, NCCL over NVLink 5 / NVSwitch (the reference has no distributed path at all: SURVEY §2.1 last
 * row; this is new work behind the same solver semantics, SURVEY §8e).  Every level's A, P and R = P^T are row-partitioned;
 * a rank stores its rows with columns relabelled to [owned | halo] positions (entry order inside a row is preserved, so
 * row sums are bit-identical to the single-GPU ones).  Before an operator is applied, the halo part of its input vector
 * is filled by grouped ncclSend/ncclRecv of packed boundary entries; Krylov scalars are combined with ncclAllReduce on
 * 1-2 doubles.  Levels at and below a size threshold are gathered once per cycle (ncclAllGather) and solved redundantly
 * on every GPU with the single-GPU hierarchy code. */
#define SPARSH_NCCL_ID_BYTES 128
int sparsh_dist_get_unique_id(char *id128);                        /* rank 0; the launcher broadcasts it */
int sparsh_dist_init(const char *id128, int nranks, int rank);     /* ncclCommInitRank on the current device */
int sparsh_dist_finalize(void);
int sparsh_dist_info(int *nranks, int *rank);

typedef struct {
    int nrow;       /* owned rows of the operator's row space                                  */
    int ncol_local; /* owned entries of its column-space vector                                */
    int nhalo;      /* remote entries appended after them: input vectors are [owned | halo]    */
    int nnz;
    const int *rowptr, *colindex; /* local CSR, columns relabelled, entry order preserved      */
    const double *val;
    const double *diag;           /* A only (NULL for P, R)                                    */
    int n_send;                   /* neighbours this rank sends to                             */
    const int *send_rank, *send_ptr, *send_idx; /* send_ptr[n_send+1] into send_idx (owned positions to pack) */
    int n_recv;                   /* neighbours it receives from                               */
    const int *recv_rank, *recv_ptr;            /* recv_ptr[n_recv+1]: offsets inside the halo segment */
    int interior_begin, interior_end;           /* rows [begin,end) reference no halo entry    */
} sparsh_dist_op_desc;

typedef struct {
    sparsh_dist_op_desc A; /* level l                      */
    sparsh_dist_op_desc P; /* level l rows x level l+1 cols */
    sparsh_dist_op_desc R; /* level l+1 rows x level l cols */
} sparsh_dist_level_desc;

typedef struct sparsh_dist_s *sparsh_dist_t;
/* lev[0..n_dist_levels) are distributed; tail[0..n_tail_levels) (global numbering, tail[0] = level n_dist_levels) are
 * replicated.  tail_counts[r] = rows of tail[0] owned by rank r, tail_rows = their global ids, rank-major. */
int sparsh_dist_hierarchy_create(int n_dist_levels, const sparsh_dist_level_desc *lev, int n_tail_levels,
                                 const sparsh_level_desc *tail, const int *tail_counts, const int *tail_rows,
                                 const sparsh_params *params, sparsh_dist_t *out);
int sparsh_dist_hierarchy_destroy(sparsh_dist_t h);
int sparsh_dist_local_rows(sparsh_dist_t h, int level, int *nrow);
/* borrow this rank's row block of A_level (columns are [owned | halo] positions) for per-kernel measurements */
int sparsh_dist_level_matrix(sparsh_dist_t h, int level, sparsh_matrix_t *A);
/* y_local = A_level x (x_local: owned entries only; the halo exchange happens inside) */
int sparsh_dist_spmv(sparsh_dist_t h, int level, const double *d_x_local, double *d_y_local);
int sparsh_dist_vcycle(sparsh_dist_t h, const double *d_b_local, double *d_x_local, int cycles, int x_is_zero);
/* distributed AMG-PCG: same arithmetic as sparsh_hierarchy_pcg, dots completed by ncclAllReduce */
int sparsh_dist_pcg(sparsh_dist_t h, const double *d_b_local, double *d_x_local, double tol, int max_iter,
                    double *h_hist, int *iters);
/* distributed twins of sparsh_hierarchy_amg_solve (AMG as a solver, AMG_solve_jacobi(b,x,-1), src/AMG_phases.cpp:194-226)
 * and of sparsh_hierarchy_pbicgstab (Solver_PBiCG_1, src/AMG_main_solvers.cpp:358-458): same arithmetic on the local
 * row blocks, residual norms and dot products completed across the ranks */
/* assemble a row-distributed HOST vector on every rank: h_full[h_rows[i]] = h_local[i] over the rows of all ranks (result
 * collection for reference-style callers that hold global b and x; setup-time collective, not on the solve path) */
int sparsh_dist_allgather_rows(const double *h_local, const int *h_rows, int n_local, double *h_full, int n_full);
int sparsh_dist_amg_solve(sparsh_dist_t h, const double *d_b_local, double *d_x_local, double tol, int max_cycles,
                          double *h_hist, int *cycles);
int sparsh_dist_pbicgstab(sparsh_dist_t h, const double *d_b_local, double *d_x_local, double tol, int max_iter,
                          double *h_hist, int *iters);

#ifdef __cplusplus
}
#endif
#endif /* SPARSH_B200_H_ */

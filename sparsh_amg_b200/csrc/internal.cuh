// internal.cuh — shared declarations of libsparsh_b200 (never includes the reference's AMG.hpp: its macros
// `th`, `omega`, ... break CUDA headers, SURVEY F8).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cmath>
#include <string>

#include <nvtx3/nvToolsExt.h>  // header-only (dlopen's the tools library when a profiler is attached; a no-op otherwise)

#include "../../include/sparsh_b200.h"

namespace sparsh {

// ---- error plumbing -------------------------------------------------------------------------------
void set_error(const std::string &msg);
int cuda_fail(cudaError_t e, const char *what, const char *file, int line);

#define SP_CUDA(call)                                                              \
    do {                                                                           \
        cudaError_t e__ = (call);                                                  \
        if (e__ != cudaSuccess) return ::sparsh::cuda_fail(e__, #call, __FILE__, __LINE__); \
    } while (0)
#define SP_TRY(call)                      \
    do {                                  \
        int rc__ = (call);                \
        if (rc__ != SPARSH_OK) return rc__; \
    } while (0)
#define SP_REQUIRE(cond, msg)             \
    do {                                  \
        if (!(cond)) {                    \
            ::sparsh::set_error(msg);     \
            return SPARSH_ERR_INVALID;    \
        }                                 \
    } while (0)

// ---- NVTX ranges (the reference links nvToolsExt without using it, CMakeLists.txt:42): phases of the solve show up by
// name in ncu / nsys timelines: sparsh:upload, sparsh:coarse-inverse, sparsh:pcg, sparsh:bicgstab, sparsh:amg-solve, ...
struct NvtxRange {
    explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange &) = delete;
    NvtxRange &operator=(const NvtxRange &) = delete;
};

// ---- runtime context --------------------------------------------------------------------------------
struct Context {
    bool ready = false;
    int device = 0;
    int sm_count = 148;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    long long launches = 0;  // kernels launched (direct) + kernel nodes replayed (graphs)
    bool capturing = false;  // launches issued while capturing are counted per replay instead
    long long captured = 0;
    // reduction workspace (two-stage deterministic reductions)
    double *partials = nullptr;  // RED_MAX_BLOCKS * RED_MAX_VALUES doubles
    unsigned int *ticket = nullptr;
    double *d_scalar = nullptr;  // small device scratch for scalar results (16 doubles)
    double *h_scalar = nullptr;  // pinned mirror
};
Context &ctx();
int ensure_init();
inline void count_launch() {
    Context &c = ctx();
    if (c.capturing)
        c.captured++;
    else
        c.launches++;
}

// ---- stopping rule of the solve loops: the host loops and the device loops' control kernels both evaluate these, so
// the two cannot drift.  Double sqrt is correctly rounded on host and device (the library is built without fast-math),
// so both sides see the same bits.
__host__ __device__ inline double solve_residual(double sq) { return sqrt(sq); }
// go on after `count` iterations with residual norm r?  No while count reaches cap or r <= tol; also no after an
// iteration that produced a non-finite r (the initial residual only meets `r > tol`: NaN stops, +inf iterates)
__host__ __device__ inline bool solve_continues(int count, int cap, double r, double tol) {
    return (count == 0 || isfinite(r)) && count < cap && r > tol;
}
__host__ __device__ inline int solve_status(double r, double tol) { return r <= tol ? SPARSH_OK : SPARSH_ERR_NOT_CONVERGED; }

constexpr int RED_MAX_BLOCKS = 1 << 20;  // partial sums per reduced value (2^28 rows at 256 rows per block)
constexpr int RED_MAX_VALUES = 4;

// ---- device CSR ---------------------------------------------------------------------------------------
enum KernelKind { KIND_SCALAR = 0, KIND_STREAM = 1, KIND_VECTOR = 2, KIND_DICT = 3, KIND_PATTERN = 4 };

// csr-dict16: lossless re-encoding of a CSR whose entries take at most 256 distinct values and 256 distinct column
// offsets (col - row) — stencil-like matrices and their Galerkin coarsenings.  One 16-bit code per entry
// (value id << 8 | offset id) replaces the 8-byte value and the 4-byte column: 2 B/nnz instead of 12.
struct DictView {
    const unsigned short *__restrict__ code;
    const double *__restrict__ val;  // n_val distinct values
    const int *__restrict__ off;     // n_off distinct col-row offsets
    int n_val, n_off;
};

// csr-pattern8: one byte per ROW.  Rows of a stencil matrix (and of its Galerkin coarsenings) repeat a handful of
// patterns — the ordered list of (col - row offset, value) pairs; the 7-point Poisson hierarchy has 27 per level.
// pat[i] < 255 selects a pattern of the table (entries start[p]..start[p+1]); pat[i] == 255 is the escape: that row is
// evaluated from the plain CSR arrays, which stay resident.  Same entries, same order, same unfused arithmetic as the
// CSR kernels: results are bit-identical.
struct PatEntry {
    double v;
    int off;
    int pad;
};
struct PatView {
    const unsigned char *__restrict__ pat;  // nrow
    const PatEntry *__restrict__ ent;       // n_ent (+8 zero entries)
    const int *__restrict__ start;          // n_pat + 1
    const double *__restrict__ pdiag;       // n_pat: the row's diagonal as sp_matrix_fill_diagonal extracts it
    int n_pat, n_ent;
    int use_pdiag;  // the epilogue's d[] is this matrix' own diagonal: take it from the table
    int far_off;    // largest positive offset of the table (0: none): the only x line of a row that rows swept earlier
                    // have not pulled into L2 yet — prefetched while the pattern byte is still on its way
};
// Pattern 0 (the most frequent row: patterns are numbered by decreasing row count) travels BY VALUE in the kernel
// parameters, so the lean kernel reads its offsets and values as constant-bank operands: no shared-memory look-up, no
// register, and — because the offsets do not depend on anything loaded — every gather of a row can be issued before
// the row's pattern byte has arrived (csr_pat2_kernel in spmv.cu).
constexpr int PAT0_MAX = 32;
// mask[p] (pattern_masks in matrix.cu): PAT_MASK_VALID set when the row of pattern p is pattern 0's row with some terms
// left out — its (offset, value bits) list is an in-order subsequence of pattern 0's and its tabulated diagonal has
// pattern 0's bits (the Dirichlet boundary rows of a stencil and their Galerkin coarsenings).  Bit k (< PAT_MASK_BITS)
// then says whether the row has entry k of pattern 0.  Pattern 0 itself has every bit; the escape id has none.
constexpr int PAT_MASK_BITS = 7;
constexpr unsigned PAT_MASK_VALID = 0x80u;
struct Pat0 {
    int len = 0;      // entries of pattern 0 (0: the lean kernel does not apply)
    int kdiag = -1;   // index of its offset-0 entry (-1: none)
    int lo = 0, hi = 0;  // smallest / largest offset
    double diag = 0.0;   // the tabulated diagonal (pdiag[0])
    double cover = 0.0;  // fraction of the rows that carry pattern 0
    double cover_masked = 0.0;  // fraction of the rows that carry pattern 0 or a pattern with a valid mask
    int off[PAT0_MAX] = {};
    double val[PAT0_MAX] = {};
    unsigned char mask[256] = {};  // per pattern id, see PAT_MASK_VALID
};
constexpr int PAT_ESCAPE = 255;    // pattern id of an escape row
constexpr int PAT_MAX_ENT = 2048;  // table entries over all patterns (32 KB)
constexpr int PAT_MAX_ROW = 64;    // longer rows are never tabulated

struct CsrView {
    int nrow, ncol, nnz;
    const int *__restrict__ rowptr;
    const int *__restrict__ col;
    const double *__restrict__ val;
};

}  // namespace sparsh

struct sparsh_matrix_s {
    int nrow = 0, ncol = 0, nnz = 0;
    int *rowptr = nullptr;  // nrow+1 (+ padding)
    int *col = nullptr;     // nnz padded to a multiple of 4, +8
    double *val = nullptr;
    double *diag = nullptr;  // nrow, or null for rectangular operators
    // kernel selection (made at upload from host-side row statistics)
    int kind = sparsh::KIND_VECTOR;
    int threads = 256;  // stream/scalar: rows per CTA == threads per CTA
    bool threads_forced = false;  // set by sparsh_matrix_force_kernel: the caller's launch shape is honoured as given
    int lanes = 8;      // vector: lanes per row
    int max_row = 0;
    double mean_row = 0.0;
    int win128 = 0, win256 = 0;  // max nnz over any window of 128 / 256 consecutive rows
    int smem_bytes = 0;          // dynamic shared memory of the stream kernel
    // choose_kernel's result before any twin or sparsh_matrix_force_kernel changed it: sparsh_matrix_update_values
    // starts its selection from here (the row statistics depend on the sparsity only)
    int base_kind = sparsh::KIND_VECTOR, base_threads = 256, base_lanes = 8, base_smem_bytes = 0;
    // csr-dict16 twin (present when the dictionaries fit; see DictView)
    unsigned short *code = nullptr;
    double *dict_val = nullptr;
    int *dict_off = nullptr;
    int n_dval = 0, n_doff = 0;
    bool has_dict = false;
    // csr-pattern8 twin (see PatView)
    unsigned char *pat = nullptr;
    sparsh::PatEntry *pat_ent = nullptr;
    int *pat_start = nullptr;
    double *pat_diag = nullptr;
    int n_pat = 0, n_pent = 0, n_escape = 0, pat_far = 0;
    int pat_cap_ent = 0, pat_cap_pat = 0;  // entries / patterns the allocated table arrays hold (reused by value updates)
    bool has_pat = false;
    sparsh::Pat0 pat0;  // len == 0: the lean (speculative-gather) variant does not apply
    // grid-transfer structure, read from the host arrays at upload (HEM: P has both, R = P^T uniform values only)
    bool one_per_row = false;  // rowptr[i] == i: exactly one stored entry per row
    bool uniform_val = false;  // every stored value has the same bits, uval
    double uval = 0.0;
    bool agg = false;  // KIND_SCALAR runs SpMV / prolongation with csr_agg_kernel (one_per_row; cleared by force_kernel)
    sparsh::PatView pattern(bool use_pdiag) const {
        return sparsh::PatView{pat, pat_ent, pat_start, pat_diag, n_pat, n_pent, use_pdiag ? 1 : 0, pat_far};
    }
    sparsh::CsrView view() const { return sparsh::CsrView{nrow, ncol, nnz, rowptr, col, val}; }
    sparsh::DictView dict() const { return sparsh::DictView{code, dict_val, dict_off, n_dval, n_doff}; }
};

namespace sparsh {

// ---- SpMV family (spmv.cu) ----------------------------------------------------------------------------
// y_i = epilogue(sum_j a_ij x_j) over rows [row_begin,row_end)
enum EpiKind {
    EPI_SPMV = 0,      // y = s
    EPI_RESID = 1,     // y = b - s
    EPI_JACOBI = 2,    // y = xi + (omega*(b - s))/d
    EPI_PROLONG = 3,   // y = s + y
    EPI_SOR = 4,       // y = y - (omega*(s - b))/d              (in place, one colour)
    EPI_SPMV_DOT = 5,  // y = s, reduce x_i*s
    EPI_RESNORM = 6    // reduce (s - b)^2, nothing stored
};
struct EpiArgs {
    const double *b = nullptr;
    const double *xi = nullptr;  // the "own" x entry stream (same array as the gathered x for Jacobi)
    const double *d = nullptr;
    double omega = 0.0;
    double *red_out = nullptr;  // device scalar receiving the reduction (EPI_SPMV_DOT / EPI_RESNORM)
    // multi-GPU, EPI_JACOBI only: rows whose new value a neighbour needs store it ALSO into that neighbour's halo
    // segment over NVLink (compute fused with the halo exchange of the next sweep).  CSR over the local rows:
    // entries pm_ptr[row]..pm_ptr[row+1] give (neighbour slot, position inside the slice sent to it).
    const int *pm_ptr = nullptr, *pm_nbr = nullptr, *pm_off = nullptr;
    double *const *pm_dst = nullptr;  // device table: per neighbour slot, the peer address of my slice (output vector)
};
int launch_csr(const sparsh_matrix_s *A, int epi, const double *x, double *y, const EpiArgs &args, int row_begin,
               int row_end);
// rows [b1,e1), [b2,e2) and [b3,e3) in ONE launch: the first nblk1 CTAs own range 1, the next nblk2 range 2, the rest
// range 3.  Multi-GPU: ranges 1 and 2 are the two boundary strips of a row block (their CTAs have the lowest block
// indices, so they are scheduled first and run the halo handshake), range 3 the interior rows.
struct RowRange {
    int b1, e1, b2, e2, b3, e3, nblk1, nblk2;
};
// multi-GPU: flag handshake fused into the consuming kernel (dist.cu).  Every CTA waits (acquire, system scope) until
// each neighbour's halo slice has landed before it gathers x; the last CTA to finish advances the sequence counter and
// stores the acks that allow the neighbours to overwrite the slices.
typedef unsigned long long sparsh_u64;
struct HaloSync {
    // consumer side: this kernel reads halo slices
    int nnbr = 0;
    const sparsh_u64 *flag_local[8];
    sparsh_u64 *ack_dst[8];
    sparsh_u64 *expect = nullptr;
    // producer side (fused Jacobi): this kernel also writes the NEXT slices into its neighbours (EpiArgs::pm_*); it
    // first makes sure they have consumed the previous ones, and the last CTA raises their flags
    int nsend = 0;
    sparsh_u64 *flag_dst[8];
    const sparsh_u64 *ack_local[8];
    sparsh_u64 *seq = nullptr;
    unsigned int *ticket = nullptr;
    int *err = nullptr;
    // CTAs [0, nstrip) take part in the handshake and in the fused push (the boundary strips); the CTAs behind them
    // own interior rows, which reference no halo entry and feed no neighbour: they neither wait nor signal.  Set by
    // the launcher.
    int nstrip = 0;
    // columns >= halo_begin of the gathered vector are halo entries, written by peers over NVLink while this grid may
    // already be resident: they are loaded through L2 (ld.global.cg), never through the non-coherent path
    int halo_begin = 0x7fffffff;
    long long timeout_ns = 10000000000ll;  // a wait that lasts longer raises *err instead of hanging the GPU
};
// rows [b1,e1) + [b2,e2) (strips: handshake CTAs when hs is given) + [b3,e3) (interior) in one launch
int launch_csr3(const sparsh_matrix_s *A, int epi, const double *x, double *y, const EpiArgs &args, int b1, int e1,
                int b2, int e2, int b3, int e3, const HaloSync *hs);
// V-cycle grid transfers (spmv_pattern.cu).  bc = R (b - A x) in one pass, one thread per row of R, the residual never
// stored: same operations in the same order as EPI_RESID followed by the restriction SpMV, so the same bits.  Applies
// when A runs the lean csr-pattern8 kernel and R's stored values are all one value (aggregation).
bool resid_restrict_applies(const sparsh_matrix_s *A, const sparsh_matrix_s *R);
int launch_resid_restrict(const sparsh_matrix_s *A, const sparsh_matrix_s *R, const double *b, const double *x, double *bc);
// x = (omega*b)/d with d = A->diag taken from A's csr-pattern8 twin (1 B per row instead of 8); applies with the lean kernel
bool jacobi_zero_pat_applies(const sparsh_matrix_s *A);
int launch_jacobi_zero_pat(const sparsh_matrix_s *A, const double *b, double omega, double *x);

inline int launch_csr2(const sparsh_matrix_s *A, int epi, const double *x, double *y, const EpiArgs &args, int b1, int e1,
                       int b2, int e2, const HaloSync *hs) {
    return launch_csr3(A, epi, x, y, args, b1, e1, b2, e2, 0, 0, hs);
}

// ---- BLAS-1 (blas1.cu) -------------------------------------------------------------------------------------
int k_fill(double *x, size_t n, double v);
int k_axpy(size_t n, double a, const double *x, double *y);
int k_axpby(size_t n, double a, const double *x, double b, double *y);
int k_axpbypcz(size_t n, double a, const double *x, double b, const double *y, double c, double *z);
int k_dot(size_t n, const double *x, const double *y, double *d_out);        // d_out[0] = x.y
int k_jacobi_zero(size_t n, const double *b, const double *d, double omega, double *x);  // x = (omega*b)/d
// Krylov fused updates; scalars live in device memory (s[] indices documented in krylov.cu)
int k_pcg_update_xr(size_t n, const double *p, const double *Ap, double *x, double *r, const double *rz,
                    const double *pAp, double *rr_out);
int k_pcg_update_p(size_t n, const double *z, double *p, const double *rz_new, const double *rz_old);
int k_scalar_copy(double *dst, const double *src);
int k_cg_update_p(size_t n, const double *r, double *p, const double *rr_new, const double *rr_old);
int k_bicg_s(size_t n, const double *r, const double *Ap, double *s, const double *alpha1, const double *apr0);
int k_bicg_xr(size_t n, double *x, const double *ph, const double *sh, const double *s, const double *As, double *r,
              const double *alpha1, const double *apr0, const double *ass, const double *asas, const double *r0,
              double *out2);
int k_bicg_p(size_t n, const double *r, double *p, const double *Ap, const double *sc);
int k_dot2(size_t n, const double *a, const double *b, const double *c, double *d_out2);  // out[0]=a.b out[1]=a.c
// GMRES(m): V holds basis vectors ld apart.  d_out[q] = V_q.w for q < k (d_out needs k rounded up to 4 slots);
// w -= sum h[q] V_q;  out = sum y[q] V_q;  out = in / sqrt(*d_nrm2)
int k_mdot(size_t n, const double *V, size_t ld, int k, const double *w, double *d_out);
int k_maxpy_sub(size_t n, const double *V, size_t ld, int k, const double *d_h, double *w);
int k_lincomb(size_t n, const double *V, size_t ld, int k, const double *d_y, double *out);
int k_scale_inv_sqrt(size_t n, const double *in, const double *d_nrm2, double *out);

// matrix uploads issued by the calling host thread go to `s` (nullptr: the library's stream) — hierarchy.cu builds the
// levels of a hierarchy with several host threads, each on a stream of its own
void set_upload_stream(cudaStream_t s);
// pageable host memory <-> device through the calling thread's pinned staging buffers (matrix.cu)
int copy_h2d_staged(void *dst, const void *src, size_t bytes, cudaStream_t st);
int copy_d2h_staged(void *dst, const void *src, size_t bytes, cudaStream_t st);  // returns when the data has arrived
void release_upload_stage();  // hands the calling thread's pinned staging buffers back to the pool (matrix.cu)

// ---- device memory of a hierarchy (runtime.cu) ------------------------------------------------------------------------------
// A device allocation or free is a call into the kernel driver: 0.6-3 ms each on the shared GPU hosts, with 0.1-1 s
// outliers (tools/alloc_probe.py) — the ~450 of them behind a 13-level hierarchy cost more than moving its 3.7 GB.  So a
// hierarchy takes ONE slab; the arrays that live as long as it does are carved from the slab by the threads bound to it
// (bump pointer, 256-byte aligned; dev_free of such a pointer is a no-op, the slab is freed as a whole), and short-lived
// temporaries come from a grow-only per-thread scratch buffer.  Without a bound slab, or once it is exhausted, dev_alloc
// is cudaMalloc and dev_free is cudaFree.
struct DevSlab;
DevSlab *slab_create(size_t bytes);  // nullptr when the allocation fails: the caller goes on without
void slab_bind(DevSlab *s);          // the calling thread's dev_alloc calls carve from s; nullptr unbinds
bool slab_bound();                   // is the calling thread bound to a slab?
void slab_destroy(DevSlab *s);       // everything carved from the slab dies with it
cudaError_t dev_alloc_bytes(void **p, size_t bytes);
template <typename T>
inline cudaError_t dev_alloc(T **p, size_t bytes) {
    return dev_alloc_bytes(reinterpret_cast<void **>(p), bytes);
}
void dev_free(void *p);
// at least `bytes` of device memory owned by the calling thread, valid until its next thread_scratch call; the caller
// synchronises its stream before it lets go of the buffer.  nullptr when the allocation fails.
void *thread_scratch(size_t bytes);
void release_thread_scratch();

// ---- Galerkin products with a kept prolongator (rap.cu, refresh.cu) ----------------------------------------------------
constexpr int RAP_MAX_ROW = 192;  // distinct columns per product row handled by the device kernels' per-thread lists
// C = A B, structure only: *crp (allocated, arow + 1) and *nnz; *fits = false when a row of C has more than RAP_MAX_ROW
// entries (nothing allocated then).  Synchronises st.
int spgemm_structure(int arow, const int *arp, const int *aci, const int *brp, const int *bci, int **crp, int *nnz,
                     bool *fits, cudaStream_t st);
// C = A B into a structure from spgemm_structure: first-touch order, unfused multiply / add (the host product's bits)
int spgemm_values(int arow, const int *arp, const int *aci, const double *av, const int *brp, const int *bci,
                  const double *bv, const int *crp, int *cci, double *cv, cudaStream_t st);

// ---- dense coarse solve (coarse.cu) ----------------------------------------------------------------------
struct CoarseInverse {
    int n = 0;
    double *inv = nullptr;  // n x n row-major
};
int coarse_build_inverse(int n, const int *h_rowptr, const int *h_col, const double *h_val, CoarseInverse *out);
// the inverse of the device CSR A (n x n, n == ci->n) in place of ci->inv: dense scatter in stored order, then the same
// Gauss-Jordan as coarse_build_inverse.  spare (n x n), piv (n) and d_min (1) are caller workspace; ci->inv keeps its
// address.  SPARSH_ERR_INVALID when A is singular.
int coarse_refactor(CoarseInverse *ci, const sparsh_matrix_s *A, double *spare, int *piv, double *d_min);
int coarse_apply(const CoarseInverse &ci, const double *b, double *x);
void coarse_free(CoarseInverse *ci);

}  // namespace sparsh

// matrix.cu — device CSR upload, kernel-family selection, and the per-op entry points of the C-ABI.
// Replaces class sp_matrix_gpu (reference include/AMG_gpu_matrix.hpp:10-48, src/AMG_gpu_matrix.cu:26-142).
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <thread>
#include <unordered_map>
#include <vector>

#include <cstdio>

#include "spmv_common.cuh"

using namespace sparsh;

namespace {

// Row statistics drive the kernel family (spmv.cu).  Computed on the host from the arrays being uploaded.
void choose_kernel(sparsh_matrix_s *A, const int *rp) {
    const int n = A->nrow;
    int max_row = 0, w128 = 0, w256 = 0;
    for (int i = 0; i < n; i++) {
        max_row = std::max(max_row, rp[i + 1] - rp[i]);
        w128 = std::max(w128, rp[std::min(i + 128, n)] - rp[i]);
        w256 = std::max(w256, rp[std::min(i + 256, n)] - rp[i]);
    }
    A->max_row = max_row;
    A->win128 = w128;
    A->win256 = w256;
    A->mean_row = n > 0 ? (double)A->nnz / n : 0.0;
    const double mean = A->mean_row;
    // lanes for the vector family: smallest power of two >= mean/2, in [2,32]
    int lanes = 2;
    while (lanes < 32 && lanes * 2 <= mean) lanes *= 2;
    A->lanes = lanes;
    A->threads = mean <= 12.0 ? 256 : 128;
    const int win = A->threads == 256 ? w256 : w128;
    A->smem_bytes = (((win + 8) + 3) & ~3) * 12;
    if (mean <= 2.5 && max_row <= 8) {
        A->kind = KIND_SCALAR;
        A->threads = 256;
    } else if (A->smem_bytes <= 96 * 1024 && max_row <= 8 * mean + 16) {
        A->kind = KIND_STREAM;  // >= 2 CTAs per SM, rows regular enough for thread-per-row
    } else {
        A->kind = KIND_VECTOR;
    }
    A->base_kind = A->kind;
    A->base_threads = A->threads;
    A->base_lanes = A->lanes;
    A->base_smem_bytes = A->smem_bytes;
}

// Aggregation operators (HEM: P has one 1.0 per row, R = P^T rows of one or two 1.0) are recognised from the host
// arrays: one entry per row, and / or one value (bit pattern) throughout.  Both scans stop at the first counterexample,
// so on any other matrix they cost a few entries.  One entry per row selects csr_agg_kernel for SpMV and prolongation.
void transfer_structure(sparsh_matrix_s *A, const int *rp, const double *v) {
    const int n = A->nrow;
    bool one = n > 0 && A->nnz == n;
    for (int i = 1; one && i <= n; i++) one = rp[i] == i;
    bool uni = A->nnz > 0;
    uint64_t u0 = 0;
    if (uni) std::memcpy(&u0, v, sizeof u0);
    for (int k = 1; uni && k < A->nnz; k++) {
        uint64_t u;
        std::memcpy(&u, v + k, sizeof u);
        uni = u == u0;
    }
    A->one_per_row = one;
    A->uniform_val = uni;
    std::memcpy(&A->uval, &u0, sizeof u0);
    A->agg = one && A->kind == KIND_SCALAR;
}

// uploads run on the library's stream, or on the calling thread's own stream while sparsh_hierarchy_create builds the
// levels with several host threads (set_upload_stream)
thread_local cudaStream_t t_upload_stream = nullptr;
struct UpStream {
    cudaStream_t stream;
};
UpStream up() { return UpStream{t_upload_stream ? t_upload_stream : ctx().stream}; }

// Pageable host arrays reach the device through this thread's pair of pinned staging buffers: the host thread copies
// chunk k+1 into one buffer while the DMA engine drains the other.  A cudaMemcpy straight from pageable memory does
// the same inside the driver, but one chunk at a time behind a lock that the upload threads of sparsh_hierarchy_create
// would share: 3.7 GB took 1.15 s (3.2 GB/s) on 8 threads.
constexpr size_t STAGE_BYTES = (size_t)8 << 20;
struct Stage {
    char *buf[2] = {nullptr, nullptr};
    cudaEvent_t ev[2] = {nullptr, nullptr};
    bool used[2] = {false, false};
    int next = 0;
    bool ready = false;
};
// The buffers are expensive to pin, so a thread borrows a pair from a process-wide pool and hands it back when it ends
// (release_upload_stage): the upload threads of successive calls reuse the same few pairs.
std::mutex g_stage_mutex;
std::vector<Stage *> g_stage_pool;  // idle pairs, every copy out of them complete
constexpr size_t STAGE_POOL_KEEP = 8;
thread_local Stage *t_stage = nullptr;
void stage_destroy(Stage *s) {
    for (int k = 0; k < 2; k++) {
        if (s->buf[k]) cudaFreeHost(s->buf[k]);
        if (s->ev[k]) cudaEventDestroy(s->ev[k]);
    }
    delete s;
}
bool stage_init() {
    if (t_stage) return true;
    {
        std::lock_guard<std::mutex> g(g_stage_mutex);
        if (!g_stage_pool.empty()) {
            t_stage = g_stage_pool.back();
            g_stage_pool.pop_back();
            return true;
        }
    }
    Stage *s = new Stage();
    for (int k = 0; k < 2; k++)
        if (cudaHostAlloc(&s->buf[k], STAGE_BYTES, cudaHostAllocDefault) != cudaSuccess ||
            cudaEventCreateWithFlags(&s->ev[k], cudaEventDisableTiming) != cudaSuccess) {
            cudaGetLastError();
            stage_destroy(s);
            return false;
        }
    s->ready = true;
    t_stage = s;
    return true;
}
int staged_h2d(void *dst, const void *src, size_t bytes, cudaStream_t st) {
    if (bytes < ((size_t)1 << 20) || !stage_init()) {
        SP_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
        return SPARSH_OK;
    }
    Stage &s = *t_stage;
    for (size_t off = 0; off < bytes; off += STAGE_BYTES) {
        const size_t n = std::min(STAGE_BYTES, bytes - off);
        const int k = s.next;
        s.next ^= 1;
        if (s.used[k]) SP_CUDA(cudaEventSynchronize(s.ev[k]));  // the DMA that last read this buffer has finished
        std::memcpy(s.buf[k], static_cast<const char *>(src) + off, n);
        SP_CUDA(cudaMemcpyAsync(static_cast<char *>(dst) + off, s.buf[k], n, cudaMemcpyHostToDevice, st));
        SP_CUDA(cudaEventRecord(s.ev[k], st));
        s.used[k] = true;
    }
    return SPARSH_OK;
}

// device -> pageable host array through the same pair of buffers (chunk k is copied out of its buffer while chunk k+1
// is on its way); the call returns when everything has arrived
int staged_d2h(void *dst, const void *src, size_t bytes, cudaStream_t st) {
    if (bytes < ((size_t)1 << 20) || !stage_init()) {
        SP_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st));
        SP_CUDA(cudaStreamSynchronize(st));
        return SPARSH_OK;
    }
    Stage &s = *t_stage;
    for (int k = 0; k < 2; k++)
        if (s.used[k]) SP_CUDA(cudaEventSynchronize(s.ev[k]));  // no upload of this thread still reads the buffers
    size_t issued = 0, drained = 0;
    int kin = 0, kout = 0;
    size_t len[2] = {0, 0};
    while (drained < bytes) {
        while (issued < bytes && issued - drained < 2 * STAGE_BYTES) {
            const size_t n = std::min(STAGE_BYTES, bytes - issued);
            SP_CUDA(cudaMemcpyAsync(s.buf[kin], static_cast<const char *>(src) + issued, n, cudaMemcpyDeviceToHost, st));
            SP_CUDA(cudaEventRecord(s.ev[kin], st));
            s.used[kin] = true;
            len[kin] = n;
            issued += n;
            kin ^= 1;
        }
        SP_CUDA(cudaEventSynchronize(s.ev[kout]));
        std::memcpy(static_cast<char *>(dst) + drained, s.buf[kout], len[kout]);
        drained += len[kout];
        kout ^= 1;
    }
    return SPARSH_OK;
}

int upload(sparsh_matrix_s *A, const int *rp, const int *ci, const double *v, const double *diag) {
    const UpStream c = up();
    const int n = A->nrow, nnz = A->nnz;
    // padding: the stream kernel's bulk copies round the slice [rowptr[r0], rowptr[r1]) outwards to multiples of 4
    const size_t pad_nnz = (((size_t)nnz + 3) & ~(size_t)3) + 8;
    SP_CUDA(dev_alloc(&A->rowptr, sizeof(int) * ((size_t)n + 8)));
    SP_CUDA(dev_alloc(&A->col, sizeof(int) * pad_nnz));
    SP_CUDA(dev_alloc(&A->val, sizeof(double) * pad_nnz));
    SP_CUDA(cudaMemsetAsync(A->col + (nnz & ~3), 0, sizeof(int) * (pad_nnz - (size_t)(nnz & ~3)), c.stream));
    SP_CUDA(cudaMemsetAsync(A->val + (nnz & ~3), 0, sizeof(double) * (pad_nnz - (size_t)(nnz & ~3)), c.stream));
    SP_TRY(staged_h2d(A->rowptr, rp, sizeof(int) * ((size_t)n + 1), c.stream));
    if (nnz > 0) {
        SP_TRY(staged_h2d(A->col, ci, sizeof(int) * (size_t)nnz, c.stream));
        SP_TRY(staged_h2d(A->val, v, sizeof(double) * (size_t)nnz, c.stream));
    }
    std::vector<double> dtmp;
    if (A->nrow == A->ncol || diag) {
        if (!diag) {
            // sp_matrix_fill_diagonal (reference src/AMG_cpu_matrix.cpp:35-51): first stored entry with col == row
            dtmp.assign((size_t)n, 0.0);
            for (int i = 0; i < n; i++)
                for (int j = rp[i]; j < rp[i + 1]; j++)
                    if (ci[j] == i) {
                        dtmp[i] = v[j];
                        break;
                    }
            diag = dtmp.data();
        }
        SP_CUDA(dev_alloc(&A->diag, sizeof(double) * ((size_t)n + 1)));
        SP_TRY(staged_h2d(A->diag, diag, sizeof(double) * (size_t)n, c.stream));
    }
    SP_CUDA(cudaStreamSynchronize(c.stream));  // host arrays may be pageable / temporary
    return SPARSH_OK;
}

// csr-dict16 twin: dictionaries of the distinct values and of the distinct (col - row) offsets, one 16-bit code per
// entry.  The encoder is host-only; false when either dictionary would need more than 256 entries.  Row chunks are
// scanned by a few threads: local dictionaries in order of first appearance, merged in chunk order (so the result is
// the one a sequential scan produces), then the codes are written in parallel.
struct LocalDict {
    std::vector<double> val;
    std::vector<int> off;
    bool overflow = false;
};
inline int find_bits(const std::vector<double> &d, double x, int hint) {
    if (hint < (int)d.size() && std::memcmp(&d[hint], &x, sizeof x) == 0) return hint;
    for (int k = 0; k < (int)d.size(); k++)
        if (std::memcmp(&d[k], &x, sizeof x) == 0) return k;  // bit pattern: -0.0 and NaNs stay themselves
    return -1;
}
inline int find_int(const std::vector<int> &d, int x, int hint) {
    if (hint < (int)d.size() && d[hint] == x) return hint;
    for (int k = 0; k < (int)d.size(); k++)
        if (d[k] == x) return k;
    return -1;
}
bool dict_encode(int n, const int *rp, const int *ci, const double *v, unsigned short *code, std::vector<double> &dv,
                 std::vector<int> &dof) {
    const size_t nnz = (size_t)rp[n];
    int nt = (int)std::min<size_t>(std::max(1u, std::thread::hardware_concurrency()), 16);
    if (nnz < (size_t)1 << 20) nt = 1;
    auto row_begin = [&](int t) { return (int)((long long)n * t / nt); };
    std::vector<LocalDict> loc((size_t)nt);
    auto scan = [&](int t) {
        LocalDict &L = loc[t];
        int hv = 0, ho = 0;
        for (int i = row_begin(t); i < row_begin(t + 1) && !L.overflow; i++)
            for (int j = rp[i]; j < rp[i + 1]; j++) {
                int vi = find_bits(L.val, v[j], hv), oi = find_int(L.off, ci[j] - i, ho);
                if (vi < 0) {
                    if (L.val.size() == 256) {
                        L.overflow = true;
                        break;
                    }
                    L.val.push_back(v[j]);
                    vi = (int)L.val.size() - 1;
                }
                if (oi < 0) {
                    if (L.off.size() == 256) {
                        L.overflow = true;
                        break;
                    }
                    L.off.push_back(ci[j] - i);
                    oi = (int)L.off.size() - 1;
                }
                hv = vi;
                ho = oi;
            }
    };
    auto run = [&](auto fn) {
        std::vector<std::thread> th;
        for (int t = 1; t < nt; t++) th.emplace_back(fn, t);
        fn(0);
        for (auto &x : th) x.join();
    };
    run(scan);
    dv.clear();
    dof.clear();
    for (const LocalDict &L : loc) {
        if (L.overflow) return false;
        for (double x : L.val)
            if (find_bits(dv, x, 0) < 0) {
                if (dv.size() == 256) return false;
                dv.push_back(x);
            }
        for (int x : L.off)
            if (find_int(dof, x, 0) < 0) {
                if (dof.size() == 256) return false;
                dof.push_back(x);
            }
    }
    auto write = [&](int t) {
        int hv = 0, ho = 0;
        for (int i = row_begin(t); i < row_begin(t + 1); i++)
            for (int j = rp[i]; j < rp[i + 1]; j++) {
                hv = find_bits(dv, v[j], hv);
                ho = find_int(dof, ci[j] - i, ho);
                code[j] = (unsigned short)((hv << 8) | ho);
            }
    };
    run(write);
    return true;
}

// encodes and uploads; false (nothing uploaded) when the matrix is not representable or SPARSH_DICT=0
bool build_dict(sparsh_matrix_s *A, const int *rp, const int *ci, const double *v) {
    const int n = A->nrow;
    const size_t nnz = (size_t)A->nnz;
    if (nnz == 0) return false;
    std::vector<double> dv;
    std::vector<int> dof;
    std::vector<unsigned short> code(nnz);
    if (!dict_encode(n, rp, ci, v, code.data(), dv, dof)) return false;
    const size_t pad = ((nnz + 7) & ~(size_t)7) + 16;  // bulk copies round the slice outwards to multiples of 8 codes
    cudaStream_t st = up().stream;
    // a value update reuses the arrays of an earlier twin: their sizes depend on nnz only
    if (!A->code && dev_alloc(&A->code, sizeof(unsigned short) * pad) != cudaSuccess) return false;
    if (!A->dict_val) dev_alloc(&A->dict_val, sizeof(double) * 256);
    if (!A->dict_off) dev_alloc(&A->dict_off, sizeof(int) * 256);
    cudaMemsetAsync(A->code, 0, sizeof(unsigned short) * pad, st);
    cudaMemcpyAsync(A->code, code.data(), sizeof(unsigned short) * nnz, cudaMemcpyHostToDevice, st);
    cudaMemcpyAsync(A->dict_val, dv.data(), sizeof(double) * dv.size(), cudaMemcpyHostToDevice, st);
    cudaMemcpyAsync(A->dict_off, dof.data(), sizeof(int) * dof.size(), cudaMemcpyHostToDevice, st);
    if (cudaStreamSynchronize(st) != cudaSuccess) return false;
    A->n_dval = (int)dv.size();
    A->n_doff = (int)dof.size();
    A->has_dict = true;
    return true;
}

// ---- csr-pattern8 (PatView in internal.cuh) ------------------------------------------------------------------
struct PatternTable {
    std::vector<int> start;  // n_pat + 1
    std::vector<double> val;
    std::vector<int> off;
    std::vector<double> diag;  // per pattern: first entry with offset 0 (what sp_matrix_fill_diagonal extracts), else 0
    int n_escape = 0;
};

inline bool same_bits(double a, double b) { return std::memcmp(&a, &b, sizeof a) == 0; }

// do rows ra and rb list the same (col - row, value bits) pairs in the same order?
inline bool same_row_pattern(const int *rp, const int *ci, const double *v, int ra, int rb) {
    const int la = rp[ra + 1] - rp[ra];
    if (la != rp[rb + 1] - rp[rb]) return false;
    const int a = rp[ra], b = rp[rb];
    for (int k = 0; k < la; k++)
        if (ci[a + k] - ra != ci[b + k] - rb || !same_bits(v[a + k], v[b + k])) return false;
    return true;
}

inline uint64_t row_pattern_hash(const int *rp, const int *ci, const double *v, int row) {
    uint64_t h = 0x9E3779B97F4A7C15ull ^ (uint64_t)(rp[row + 1] - rp[row]);
    for (int k = rp[row]; k < rp[row + 1]; k++) {
        uint64_t bits;
        std::memcpy(&bits, &v[k], sizeof bits);
        h = (h ^ bits) * 0x100000001B3ull;
        h = (h ^ (uint64_t)(uint32_t)(ci[k] - row)) * 0xC2B2AE3D27D4EB4Full;
        h ^= h >> 29;
    }
    return h;
}

// distinct rows beyond which a matrix is declared not stencil-like, by both encoders
constexpr int PAT_MAX_CAND = 1 << 15;

// Host-only encoder.  pat[i] receives the pattern id of row i (PAT_ESCAPE for rows left to the CSR arrays).  Patterns
// are numbered by decreasing row count (ties: first occurrence).  h_diag, when given, is the diagonal the caller will
// smooth with: rows where it differs from the tabulated one become escapes.  Returns false when the matrix is not
// stencil-like (more than PAT_MAX_CAND distinct rows, or fewer than min_cover of the rows tabulated).
bool pattern_encode(int n, const int *rp, const int *ci, const double *v, const double *h_diag, unsigned char *pat,
                    PatternTable &T, double min_cover) {
    struct Cand {
        int rep, count;
    };
    std::vector<Cand> cand;
    std::unordered_map<uint64_t, int> by_hash;
    std::vector<int> cand_of((size_t)n, -1);
    int prev = -1;
    for (int i = 0; i < n; i++) {
        if (rp[i + 1] - rp[i] > PAT_MAX_ROW) {
            prev = -1;
            continue;
        }
        int c = -1;
        if (prev >= 0 && same_row_pattern(rp, ci, v, i, cand[prev].rep)) {
            c = prev;  // neighbouring rows of a stencil matrix mostly repeat the pattern
        } else {
            const uint64_t h = row_pattern_hash(rp, ci, v, i);
            auto it = by_hash.find(h);
            if (it == by_hash.end()) {
                if (cand.size() >= (size_t)PAT_MAX_CAND) return false;  // not stencil-like: stop before the map grows with n
                c = (int)cand.size();
                cand.push_back(Cand{i, 0});
                by_hash.emplace(h, c);
            } else if (same_row_pattern(rp, ci, v, i, cand[it->second].rep)) {
                c = it->second;
            }  // else: a hash collision between different rows; this one stays an escape
        }
        if (c >= 0) cand[c].count++;
        cand_of[i] = c;
        prev = c;
    }
    std::vector<int> order(cand.size());
    for (size_t k = 0; k < order.size(); k++) order[k] = (int)k;
    std::sort(order.begin(), order.end(), [&](int a, int b) {
        return cand[a].count != cand[b].count ? cand[a].count > cand[b].count : cand[a].rep < cand[b].rep;
    });
    std::vector<int> id_of(cand.size(), -1);
    T = PatternTable();
    T.start.push_back(0);
    for (int c : order) {
        const int r = cand[c].rep, len = rp[r + 1] - rp[r];
        if ((int)T.diag.size() == PAT_ESCAPE) break;
        if ((int)T.val.size() + len > PAT_MAX_ENT) continue;
        id_of[c] = (int)T.diag.size();
        double d = 0.0;
        bool found = false;
        for (int k = rp[r]; k < rp[r + 1]; k++) {
            T.val.push_back(v[k]);
            T.off.push_back(ci[k] - r);
            if (!found && ci[k] == r) {
                d = v[k];
                found = true;
            }
        }
        T.diag.push_back(d);
        T.start.push_back((int)T.val.size());
    }
    long long covered = 0;
    for (int i = 0; i < n; i++) {
        int id = cand_of[i] >= 0 ? id_of[cand_of[i]] : -1;
        if (id >= 0 && h_diag && !same_bits(h_diag[i], T.diag[id])) id = -1;
        pat[i] = (unsigned char)(id >= 0 ? id : PAT_ESCAPE);
        covered += id >= 0;
    }
    T.n_escape = n - (int)covered;
    return n > 0 && !T.diag.empty() && (double)covered >= min_cover * (double)n;
}

// The lean kernel's masks (Pat0::mask in internal.cuh).  A pattern whose (offset, value bits) list is an in-order
// subsequence of pattern 0's, with pattern 0's diagonal, is evaluated as pattern 0 with the missing terms skipped: the
// same products added in the same order, so the same bits as the table walk and the CSR kernels.  Greedy leftmost
// matching decides the subsequence; where pattern 0 repeats an (offset, value) pair, any match adds the same terms.
void pattern_masks(const PatternTable &T, unsigned char mask[256]) {
    std::fill(mask, mask + 256, (unsigned char)0);
    const int n_pat = std::min((int)T.diag.size(), PAT_ESCAPE);
    if (n_pat == 0) return;
    const int len0 = T.start[1] - T.start[0];
    if (len0 > PAT_MASK_BITS) return;
    for (int p = 0; p < n_pat; p++) {
        if (!same_bits(T.diag[p], T.diag[0])) continue;
        unsigned m = 0;
        int k = 0;
        bool sub = true;
        for (int j = T.start[p]; sub && j < T.start[p + 1]; j++) {
            while (k < len0 && !(T.off[k] == T.off[j] && same_bits(T.val[k], T.val[j]))) k++;
            sub = k < len0;
            if (sub) m |= 1u << k++;
        }
        if (sub) mask[p] = (unsigned char)(PAT_MASK_VALID | m);
    }
}

// ---- csr-pattern8 encoder on the device -----------------------------------------------------------------------
// The host encoder above (kept as the CPU-checkable statement of the format, sparsh_pattern_encode) walks every row
// with a hash map on one core: 0.5 s for 3D Poisson 256^3, a quarter of the whole upload.  The matrix is on the device
// anyway by then, so: (1) one kernel hashes every row (same hash as row_pattern_hash) and registers it in a small
// open-addressing table — key = hash, representative = smallest row index (atomicMin: the first occurrence, as on the
// host), count —; (2) the host reads the few candidates back, orders them exactly like the host encoder (count
// descending, first occurrence ascending) and builds the table from the representatives' rows; (3) a second kernel
// gives every row its pattern id after comparing it ENTRY BY ENTRY with the tabulated pattern (a hash collision or a
// differing smoothing diagonal makes the row an escape).  The result equals the host encoder's, including the decision:
// both give up past PAT_MAX_CAND distinct rows.
constexpr int PAT_SLOTS = 1 << 17;  // open addressing: load factor <= 1/4 at PAT_MAX_CAND keys
struct PatSlot {
    unsigned long long key;  // 0 = empty
    int rep, count;
};

__device__ __forceinline__ unsigned long long device_row_hash(const int *rp, const int *ci, const double *v, int row) {
    unsigned long long h = 0x9E3779B97F4A7C15ull ^ (unsigned long long)(rp[row + 1] - rp[row]);
    for (int k = rp[row]; k < rp[row + 1]; k++) {
        const unsigned long long bits = (unsigned long long)__double_as_longlong(v[k]);
        h = (h ^ bits) * 0x100000001B3ull;
        h = (h ^ (unsigned long long)(unsigned int)(ci[k] - row)) * 0xC2B2AE3D27D4EB4Full;
        h ^= h >> 29;
    }
    return h ? h : 1ull;
}

__global__ void __launch_bounds__(256)
    pat_hash_kernel(int n, const int *__restrict__ rp, const int *__restrict__ ci, const double *__restrict__ v, PatSlot *table,
                    int *slot_of, int *overflow) {
    // overflow[0]: "rows do not repeat" (too many distinct rows) — everybody stops as soon as somebody finds out;
    // overflow[1]: distinct rows registered so far
    const int row = blockIdx.x * 256 + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const bool valid = row < n && rp[row + 1] - rp[row] <= PAT_MAX_ROW && *reinterpret_cast<volatile int *>(overflow) == 0;
    // Almost every row of a stencil matrix carries the same hash: three atomics per row on ONE slot serialise in the L2
    // atomic unit (measured: 45 ms for 16.8 M rows).  The lanes of a warp that share a hash elect their lowest lane (=
    // their smallest row) to register the whole group once.  (All 32 lanes take part in the vote; a lane without a
    // row votes with a key of its own.)
    const unsigned long long h = valid ? device_row_hash(rp, ci, v, row) : (0xFFFFFFFFFFFFFF00ull | (unsigned long long)lane);
    const unsigned int peers = __match_any_sync(0xffffffffu, h);
    const int leader = __ffs(peers) - 1;
    int slot = -1;
    if (valid && lane == leader) {
        unsigned int s = (unsigned int)(h >> 20) & (PAT_SLOTS - 1);
        bool failed = true;
        for (int probe = 0; probe < 256; probe++, s = (s + 1) & (PAT_SLOTS - 1)) {  // load factor <= 1/4: probes are short
            const unsigned long long seen = atomicCAS(&table[s].key, 0ull, h);
            if (seen == 0ull && atomicAdd(overflow + 1, 1) >= PAT_MAX_CAND) break;
            if (seen == 0ull || seen == h) {
                atomicMin(&table[s].rep, row);
                atomicAdd(&table[s].count, __popc(peers));
                slot = (int)s;
                failed = false;
                break;
            }
        }
        if (failed) atomicExch(overflow, 1);
    }
    slot = __shfl_sync(0xffffffffu, slot, leader);
    if (row < n) slot_of[row] = valid ? slot : -1;
}

// pat[i] = id of row i's pattern if the row equals the tabulated pattern entry by entry (and, when `diag` is given, its
// smoothing diagonal equals the tabulated one bit for bit), PAT_ESCAPE otherwise; counts[0] += covered rows, counts[1] += rows
// of pattern 0, counts[2] += rows of pattern 0 or of a pattern with a valid mask in Z
__global__ void __launch_bounds__(256)
    pat_assign_kernel(int n, const int *__restrict__ rp, const int *__restrict__ ci, const double *__restrict__ v,
                      const double *__restrict__ diag, const int *__restrict__ slot_of, const int *__restrict__ id_of_slot,
                      const PatEntry *__restrict__ ent, const int *__restrict__ start, const double *__restrict__ pdiag,
                      const __grid_constant__ Pat0 Z, unsigned char *pat, unsigned long long *counts) {
    const int row = blockIdx.x * 256 + threadIdx.x;
    int id = -1;
    if (row < n) {
        const int s = slot_of[row];
        if (s >= 0) id = id_of_slot[s];
        if (id >= 0) {
            const int lo = rp[row], len = rp[row + 1] - lo, st = start[id];
            bool same = len == start[id + 1] - st;
            for (int k = 0; same && k < len; k++)
                same = ci[lo + k] - row == ent[st + k].off && __double_as_longlong(v[lo + k]) == __double_as_longlong(ent[st + k].v);
            if (same && diag) same = __double_as_longlong(diag[row]) == __double_as_longlong(pdiag[id]);
            if (!same) id = -1;
        }
        pat[row] = (unsigned char)(id >= 0 ? id : PAT_ESCAPE);
    }
    const unsigned int covered = __ballot_sync(0xffffffffu, id >= 0), zero = __ballot_sync(0xffffffffu, id == 0);
    const unsigned int masked = __ballot_sync(0xffffffffu, id == 0 || (id > 0 && (Z.mask[id] & PAT_MASK_VALID)));
    if ((threadIdx.x & 31) == 0) {
        if (covered) atomicAdd(&counts[0], (unsigned long long)__popc(covered));
        if (zero) atomicAdd(&counts[1], (unsigned long long)__popc(zero));
        if (masked) atomicAdd(&counts[2], (unsigned long long)__popc(masked));
    }
}

// SPARSH_PATTERN: 1 (default) build the twin and run the pattern kernel wherever it applies (measured on B200: fused
// Jacobi sweep on 3D Poisson 256^3 0.111 ms against 0.179 ms for csr-dict16 and 0.294 ms for plain CSR, whole AMG-PCG
// solve 0.157 s against 0.206 s; bit-identical results); 0 no twin; 2 build the twin but keep the dict / stream kernel
// (sparsh_matrix_force_kernel selects)
int pattern_mode() {
    const char *env = getenv("SPARSH_PATTERN");
    return env ? atoi(env) : 1;
}

// lengths (dst == nullptr) or entries (col - row, value) of the rows reps[0..k): the representative rows a pattern table
// is built from when the matrix' host arrays are gone (sparsh_matrix_update_values)
__global__ void __launch_bounds__(256)
    pat_gather_kernel(int k, const int *__restrict__ reps, const int *__restrict__ rp, const int *__restrict__ ci,
                      const double *__restrict__ v, const int *__restrict__ dst, int *len, int *off, double *val) {
    const int t = blockIdx.x * 256 + threadIdx.x;
    if (t >= k) return;
    const int r = reps[t], lo = rp[r], l = rp[r + 1] - lo;
    if (!dst) {
        len[t] = l;
        return;
    }
    for (int q = 0; q < l; q++) {
        off[dst[t] + q] = ci[lo + q] - r;
        val[dst[t] + q] = v[lo + q];
    }
}

// encodes (on the device, see above) and keeps the twin; false (nothing kept) when the rows do not repeat enough.  The
// table is built from the representatives' rows: read from the HOST arrays rp, ci, v when given (the upload), else
// gathered from the device copies A->rowptr/col/val (a value update).  check_diag: A->diag is the caller's smoothing
// diagonal, and rows where it differs from the tabulated one become escapes.
bool build_pattern(sparsh_matrix_s *A, const int *rp, const int *ci, const double *v, bool check_diag) {
    const int n = A->nrow;
    if (n == 0 || A->nnz == 0) return false;
    cudaStream_t st = up().stream;
    bool kept = false;
    auto cleanup = [&]() {  // the temporaries live in this thread's scratch buffer; every path here has synchronised st
        if (!kept) {
            dev_free(A->pat);
            dev_free(A->pat_ent);
            dev_free(A->pat_start);
            dev_free(A->pat_diag);
            A->pat = nullptr;
            A->pat_ent = nullptr;
            A->pat_start = nullptr;
            A->pat_diag = nullptr;
            A->pat_cap_ent = A->pat_cap_pat = 0;
        }
        cudaGetLastError();
    };
    // temporaries: [table | id_of | slot_of | counts | overflow | gather: reps, lengths, destinations, offsets, values],
    // each 256-byte aligned, in one scratch block
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t o_table = 0, o_id = o_table + al(sizeof(PatSlot) * PAT_SLOTS), o_slot = o_id + al(sizeof(int) * PAT_SLOTS),
                 o_counts = o_slot + al(sizeof(int) * (size_t)n), o_over = o_counts + 256, o_reps = o_over + 256,
                 o_len = o_reps + al(sizeof(int) * PAT_MAX_CAND), o_dst = o_len + al(sizeof(int) * PAT_MAX_CAND),
                 o_goff = o_dst + al(sizeof(int) * PAT_ESCAPE), o_gval = o_goff + al(sizeof(int) * PAT_MAX_ENT),
                 scratch_bytes = o_gval + al(sizeof(double) * PAT_MAX_ENT);
    char *scratch = static_cast<char *>(thread_scratch(scratch_bytes));
    if (!scratch) return false;
    PatSlot *d_table = reinterpret_cast<PatSlot *>(scratch + o_table);
    int *d_id_of = reinterpret_cast<int *>(scratch + o_id), *d_slot_of = reinterpret_cast<int *>(scratch + o_slot);
    unsigned long long *d_counts = reinterpret_cast<unsigned long long *>(scratch + o_counts);
    int *d_overflow = reinterpret_cast<int *>(scratch + o_over);
    bool ok = true;
    std::vector<PatSlot> table(PAT_SLOTS, PatSlot{0ull, 0x7fffffff, 0});
    cudaMemcpyAsync(d_table, table.data(), sizeof(PatSlot) * PAT_SLOTS, cudaMemcpyHostToDevice, st);
    cudaMemsetAsync(d_overflow, 0, sizeof(int) * 2, st);
    cudaMemsetAsync(d_counts, 0, sizeof(unsigned long long) * 3, st);
    const int grid = (n + 255) / 256;
    pat_hash_kernel<<<grid, 256, 0, st>>>(n, A->rowptr, A->col, A->val, d_table, d_slot_of, d_overflow);
    int overflow = 0;
    cudaMemcpyAsync(&overflow, d_overflow, sizeof(int), cudaMemcpyDeviceToHost, st);
    if (cudaStreamSynchronize(st) != cudaSuccess || overflow) {
        cleanup();
        return false;
    }
    if (cudaMemcpyAsync(table.data(), d_table, sizeof(PatSlot) * PAT_SLOTS, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess) {
        cleanup();
        return false;
    }
    // candidates in the host encoder's order: by decreasing row count, ties by first occurrence
    struct Cand {
        int rep, count, slot;
    };
    std::vector<Cand> cand;
    for (int sidx = 0; sidx < PAT_SLOTS; sidx++)
        if (table[sidx].key != 0ull) cand.push_back(Cand{table[sidx].rep, table[sidx].count, sidx});
    if (cand.empty()) {
        cleanup();
        return false;
    }
    std::sort(cand.begin(), cand.end(), [](const Cand &a, const Cand &b) { return a.count != b.count ? a.count > b.count : a.rep < b.rep; });
    // row lengths of the candidates, then the ones that enter the table (a row that would overflow it is skipped)
    const int n_cand = (int)cand.size();
    std::vector<int> len((size_t)n_cand), reps((size_t)n_cand);
    for (int k = 0; k < n_cand; k++) reps[k] = cand[k].rep;
    int *d_reps = reinterpret_cast<int *>(scratch + o_reps), *d_len = reinterpret_cast<int *>(scratch + o_len);
    if (rp) {
        for (int k = 0; k < n_cand; k++) len[k] = rp[reps[k] + 1] - rp[reps[k]];
    } else {
        cudaMemcpyAsync(d_reps, reps.data(), sizeof(int) * (size_t)n_cand, cudaMemcpyHostToDevice, st);
        pat_gather_kernel<<<(n_cand + 255) / 256, 256, 0, st>>>(n_cand, d_reps, A->rowptr, A->col, A->val, nullptr, d_len, nullptr, nullptr);
        cudaMemcpyAsync(len.data(), d_len, sizeof(int) * (size_t)n_cand, cudaMemcpyDeviceToHost, st);
        if (cudaStreamSynchronize(st) != cudaSuccess) {
            cleanup();
            return false;
        }
    }
    PatternTable T;
    T.start.push_back(0);
    std::vector<int> id_of(PAT_SLOTS, -1), sel;
    for (int k = 0; k < n_cand; k++) {
        if ((int)T.start.size() - 1 == PAT_ESCAPE) break;
        if (T.start.back() + len[k] > PAT_MAX_ENT) continue;
        id_of[cand[k].slot] = (int)T.start.size() - 1;
        sel.push_back(k);
        T.start.push_back(T.start.back() + len[k]);
    }
    const int n_pat = (int)sel.size(), n_ent = T.start.back();
    if (n_pat == 0) {
        cleanup();
        return false;
    }
    std::vector<int> g_off;
    std::vector<double> g_val;
    if (!rp) {  // the selected rows' entries, in table order
        std::vector<int> sreps((size_t)n_pat);
        for (int p = 0; p < n_pat; p++) sreps[p] = reps[sel[p]];
        g_off.resize((size_t)std::max(n_ent, 1));
        g_val.resize((size_t)std::max(n_ent, 1));
        int *d_dst = reinterpret_cast<int *>(scratch + o_dst), *d_goff = reinterpret_cast<int *>(scratch + o_goff);
        double *d_gval = reinterpret_cast<double *>(scratch + o_gval);
        cudaMemcpyAsync(d_reps, sreps.data(), sizeof(int) * (size_t)n_pat, cudaMemcpyHostToDevice, st);
        cudaMemcpyAsync(d_dst, T.start.data(), sizeof(int) * (size_t)n_pat, cudaMemcpyHostToDevice, st);
        pat_gather_kernel<<<(n_pat + 255) / 256, 256, 0, st>>>(n_pat, d_reps, A->rowptr, A->col, A->val, d_dst, nullptr, d_goff, d_gval);
        cudaMemcpyAsync(g_off.data(), d_goff, sizeof(int) * (size_t)n_ent, cudaMemcpyDeviceToHost, st);
        cudaMemcpyAsync(g_val.data(), d_gval, sizeof(double) * (size_t)n_ent, cudaMemcpyDeviceToHost, st);
        if (cudaStreamSynchronize(st) != cudaSuccess) {
            cleanup();
            return false;
        }
    }
    for (int p = 0; p < n_pat; p++) {
        const int r = reps[sel[p]];
        double d = 0.0;
        bool found = false;
        for (int q = 0; q < len[sel[p]]; q++) {
            const int off = rp ? ci[rp[r] + q] - r : g_off[T.start[p] + q];
            const double x = rp ? v[rp[r] + q] : g_val[T.start[p] + q];
            T.val.push_back(x);
            T.off.push_back(off);
            if (!found && off == 0) {
                d = x;
                found = true;
            }
        }
        T.diag.push_back(d);
    }
    std::vector<PatEntry> ent((size_t)n_ent + 8, PatEntry{0.0, 0, 0});
    for (int k = 0; k < n_ent; k++) ent[k] = PatEntry{T.val[k], T.off[k], 0};
    Pat0 z;  // pattern 0 by value for the lean kernel (spmv_pattern.cu: csr_pat2_kernel)
    const int len0 = T.start[1] - T.start[0];
    if (len0 >= 1 && len0 <= PAT0_MAX) {
        z.len = len0;
        z.diag = T.diag[0];
        z.lo = z.hi = T.off[0];
        for (int k = 0; k < len0; k++) {
            z.off[k] = T.off[k];
            z.val[k] = T.val[k];
            z.lo = std::min(z.lo, T.off[k]);
            z.hi = std::max(z.hi, T.off[k]);
            if (T.off[k] == 0 && z.kdiag < 0) z.kdiag = k;
        }
        pattern_masks(T, z.mask);
    }
    // a value update reuses the arrays of an earlier twin when the new table fits them
    if (!A->pat) ok = dev_alloc(&A->pat, (size_t)n + 16) == cudaSuccess;
    if (ok && A->pat_cap_ent < (int)ent.size()) {
        dev_free(A->pat_ent);
        A->pat_ent = nullptr;
        ok = dev_alloc(&A->pat_ent, sizeof(PatEntry) * ent.size()) == cudaSuccess;
        A->pat_cap_ent = ok ? (int)ent.size() : 0;
    }
    if (ok && A->pat_cap_pat < n_pat) {
        dev_free(A->pat_start);
        dev_free(A->pat_diag);
        A->pat_start = nullptr;
        A->pat_diag = nullptr;
        ok = dev_alloc(&A->pat_start, sizeof(int) * ((size_t)n_pat + 1)) == cudaSuccess &&
             dev_alloc(&A->pat_diag, sizeof(double) * (size_t)n_pat) == cudaSuccess;
        A->pat_cap_pat = ok ? n_pat : 0;
    }
    unsigned long long counts[3] = {0ull, 0ull, 0ull};
    if (ok) {
        cudaMemsetAsync(A->pat, PAT_ESCAPE, (size_t)n + 16, st);
        cudaMemcpyAsync(A->pat_ent, ent.data(), sizeof(PatEntry) * ent.size(), cudaMemcpyHostToDevice, st);
        cudaMemcpyAsync(A->pat_start, T.start.data(), sizeof(int) * ((size_t)n_pat + 1), cudaMemcpyHostToDevice, st);
        cudaMemcpyAsync(A->pat_diag, T.diag.data(), sizeof(double) * (size_t)n_pat, cudaMemcpyHostToDevice, st);
        cudaMemcpyAsync(d_id_of, id_of.data(), sizeof(int) * PAT_SLOTS, cudaMemcpyHostToDevice, st);
        // rows whose smoothing diagonal (A->diag, the caller's) differs from the tabulated one become escapes
        pat_assign_kernel<<<grid, 256, 0, st>>>(n, A->rowptr, A->col, A->val, check_diag ? A->diag : nullptr, d_slot_of, d_id_of,
                                                A->pat_ent, A->pat_start, A->pat_diag, z, A->pat, d_counts);
        cudaMemcpyAsync(counts, d_counts, sizeof counts, cudaMemcpyDeviceToHost, st);
        ok = cudaStreamSynchronize(st) == cudaSuccess;
    }
    if (!ok || (double)counts[0] < 0.75 * (double)n) {  // min_cover of the host encoder's upload path
        cleanup();
        return false;
    }
    A->n_pat = n_pat;
    A->n_pent = n_ent;
    A->n_escape = n - (int)counts[0];
    A->pat_far = 0;
    for (int k = 0; k < n_ent; k++) A->pat_far = std::max(A->pat_far, T.off[k]);
    // the shares are statistics of the table (sparsh_matrix_pattern_stats), also when pattern 0 is too long to travel
    // by value (z.len == 0: the lean kernel does not apply whatever they are)
    z.cover = (double)counts[1] / (double)n;
    z.cover_masked = (double)counts[2] / (double)n;
    A->pat0 = z;
    A->has_pat = true;
    kept = true;
    cleanup();
    return true;
}

// ---- value updates on the device (sparsh_matrix_update_values) ----------------------------------------------------
// differs[0] = 1 when some stored value's bits differ from v[0]'s (transfer_structure's scan)
__global__ void __launch_bounds__(256) uniform_bits_kernel(size_t nnz, const double *__restrict__ v, int *differs) {
    const long long u0 = __double_as_longlong(v[0]);
    for (size_t k = (size_t)blockIdx.x * 256 + threadIdx.x; k < nnz; k += (size_t)gridDim.x * 256)
        if (__double_as_longlong(v[k]) != u0) {
            *differs = 1;
            return;
        }
}

// sp_matrix_fill_diagonal: the first stored entry with col == row, else 0
__global__ void __launch_bounds__(256)
    diag_extract_kernel(int n, const int *__restrict__ rp, const int *__restrict__ ci, const double *__restrict__ v, double *d) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    double x = 0.0;
    for (int j = rp[i]; j < rp[i + 1]; j++)
        if (ci[j] == i) {
            x = v[j];
            break;
        }
    d[i] = x;
}

// Can the csr-dict16 twin exist?  Distinct value bit patterns and distinct (col - row) offsets are registered in two
// small open-addressing sets; count[0] / count[1] receive their sizes, over[0] = 1 as soon as either passes 256 (every
// thread then stops).  An empty slot holds ~0; a value with exactly those bits is recorded in count[2] instead.
constexpr int DICT_SLOTS = 1024;
constexpr unsigned long long DICT_EMPTY = ~0ull;
__device__ __forceinline__ void dict_insert(unsigned long long *set, unsigned long long key, int *count, int *over) {
    unsigned int s = (unsigned int)((key * 0x9E3779B97F4A7C15ull) >> 54);
    for (int probe = 0; probe < DICT_SLOTS; probe++, s = (s + 1) & (DICT_SLOTS - 1)) {
        unsigned long long seen = *reinterpret_cast<volatile unsigned long long *>(set + s);
        if (seen == DICT_EMPTY) seen = atomicCAS(set + s, DICT_EMPTY, key);
        if (seen == DICT_EMPTY) {
            if (atomicAdd(count, 1) >= 256) atomicExch(over, 1);
            return;
        }
        if (seen == key) return;
    }
    atomicExch(over, 1);
}
__global__ void __launch_bounds__(256)
    dict_fits_kernel(int n, const int *__restrict__ rp, const int *__restrict__ ci, const double *__restrict__ v,
                     unsigned long long *vset, unsigned long long *oset, int *count, int *over) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n || *reinterpret_cast<volatile int *>(over)) return;
    for (int j = rp[i]; j < rp[i + 1]; j++) {
        const unsigned long long bits = (unsigned long long)__double_as_longlong(v[j]);
        if (bits == DICT_EMPTY)
            atomicExch(count + 2, 1);
        else
            dict_insert(vset, bits, count, over);
        dict_insert(oset, (unsigned long long)(unsigned int)(ci[j] - i), count + 1, over);
    }
}

// build_dict from the device arrays: the host encoder runs only when the device found the twin possible
bool build_dict_device(sparsh_matrix_s *A) {
    const int n = A->nrow, nnz = A->nnz;
    if (nnz == 0) return false;
    cudaStream_t st = up().stream;
    char *scratch = static_cast<char *>(thread_scratch(2 * sizeof(unsigned long long) * DICT_SLOTS + 256));
    if (!scratch) return false;
    unsigned long long *vset = reinterpret_cast<unsigned long long *>(scratch), *oset = vset + DICT_SLOTS;
    int *d_count = reinterpret_cast<int *>(oset + DICT_SLOTS), *d_over = d_count + 3;
    int h[4] = {0, 0, 0, 0};
    cudaMemsetAsync(vset, 0xff, 2 * sizeof(unsigned long long) * DICT_SLOTS, st);
    cudaMemsetAsync(d_count, 0, sizeof(int) * 4, st);
    dict_fits_kernel<<<(n + 255) / 256, 256, 0, st>>>(n, A->rowptr, A->col, A->val, vset, oset, d_count, d_over);
    cudaMemcpyAsync(h, d_count, sizeof h, cudaMemcpyDeviceToHost, st);
    if (cudaStreamSynchronize(st) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    if (h[3] || h[0] + h[2] > 256 || h[1] > 256) return false;
    std::vector<int> rp((size_t)n + 1), ci((size_t)nnz);
    std::vector<double> v((size_t)nnz);
    if (staged_d2h(rp.data(), A->rowptr, sizeof(int) * ((size_t)n + 1), st) != SPARSH_OK ||
        staged_d2h(ci.data(), A->col, sizeof(int) * (size_t)nnz, st) != SPARSH_OK ||
        staged_d2h(v.data(), A->val, sizeof(double) * (size_t)nnz, st) != SPARSH_OK) {
        cudaGetLastError();
        return false;
    }
    return build_dict(A, rp.data(), ci.data(), v.data());
}

// The compressed twins and the kernel family, from A's kind as choose_kernel left it.  rp, ci, v: the host arrays of
// the upload, or nullptr to work from the device arrays (a value update).  check_diag: A->diag is the caller's.
void choose_twins(sparsh_matrix_s *A, const int *rp, const int *ci, const double *v, bool check_diag) {
    // Matrices that would run the stream kernel get a lossless compressed twin when they are stencil-like.
    // csr-pattern8 first (1 B per row, encoded on the device): when the rows repeat it wins, and the csr-dict16 twin
    // (2 B per entry, encoded by the host: 0.5 s per 10^8 entries) is not even built unless SPARSH_DICT=2 asks for both.
    const int pmode = pattern_mode();
    const char *denv = getenv("SPARSH_DICT");
    const int dmode = denv ? atoi(denv) : 1;  // 0: never, 1: when csr-pattern8 is not selected, 2: always (tests, A/B runs)
    // (rectangular operators qualify too: the multi-GPU local blocks are nrow x (owned + halo) with a diagonal)
    bool pattern_selected = false;
    if (pmode > 0 && A->kind == KIND_STREAM && build_pattern(A, rp, ci, v, check_diag)) pattern_selected = pmode == 1;
    if (A->kind == KIND_STREAM && dmode > 0 && (!pattern_selected || dmode == 2) &&
        (rp ? build_dict(A, rp, ci, v) : build_dict_device(A))) {
        A->kind = KIND_DICT;
        A->threads = 128;  // measured on B200 (256^3 Jacobi): 128-thread CTAs x 4 rows per thread 0.180 ms, 256 x 4 0.199 ms
    }
    if (pattern_selected) {
        A->kind = KIND_PATTERN;
        A->threads = 128;
    }
}

int validate(int nrow, int ncol, int nnz, const int *rp, const int *ci) {
    SP_REQUIRE(nrow >= 0 && ncol >= 0 && nnz >= 0, "negative matrix dimension");
    SP_REQUIRE(rp != nullptr, "rowptr is NULL");
    SP_REQUIRE(rp[0] == 0 && rp[nrow] == nnz, "rowptr[0] != 0 or rowptr[nrow] != nnz");
    for (int i = 0; i < nrow; i++) SP_REQUIRE(rp[i] <= rp[i + 1], "rowptr not monotone");
    for (int j = 0; j < nnz; j++) SP_REQUIRE(ci[j] >= 0 && ci[j] < ncol, "column index out of range");
    return SPARSH_OK;
}

}  // namespace

namespace sparsh {
void set_upload_stream(cudaStream_t s) { t_upload_stream = s; }
int copy_h2d_staged(void *dst, const void *src, size_t bytes, cudaStream_t st) { return staged_h2d(dst, src, bytes, st); }
int copy_d2h_staged(void *dst, const void *src, size_t bytes, cudaStream_t st) { return staged_d2h(dst, src, bytes, st); }
// give this thread's pinned staging buffers back (upload worker threads call it before they end)
void release_upload_stage() {
    Stage *s = t_stage;
    if (!s) return;
    t_stage = nullptr;
    for (int k = 0; k < 2; k++)
        if (s->used[k]) {
            cudaEventSynchronize(s->ev[k]);  // the pool holds idle pairs only
            s->used[k] = false;
        }
    s->next = 0;
    {
        std::lock_guard<std::mutex> g(g_stage_mutex);
        if (g_stage_pool.size() < STAGE_POOL_KEEP) {
            g_stage_pool.push_back(s);
            return;
        }
    }
    stage_destroy(s);
}
}  // namespace sparsh

extern "C" {

int sparsh_matrix_create(int nrow, int ncol, int nnz, const int *h_rowptr, const int *h_colindex,
                         const double *h_val, const double *h_diag, sparsh_matrix_t *out) {
    SP_TRY(ensure_init());
    SP_REQUIRE(out != nullptr, "out is NULL");
    static const bool timing = getenv("SPARSH_UPLOAD_TIMING") != nullptr;  // developer switch: where does the upload go?
    const auto t0 = std::chrono::steady_clock::now();
    SP_TRY(validate(nrow, ncol, nnz, h_rowptr, h_colindex));
    sparsh_matrix_s *A = new sparsh_matrix_s();
    A->nrow = nrow;
    A->ncol = ncol;
    A->nnz = nnz;
    auto lap = [&](const char *what) {
        if (timing && nnz > 1000000)
            std::fprintf(stderr, "[upload %d x %d, %d nnz] %s at %.3f s\n", nrow, ncol, nnz, what,
                         std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
    };
    lap("validated");
    choose_kernel(A, h_rowptr);
    transfer_structure(A, h_rowptr, h_val);
    lap("row statistics");
    int rc = upload(A, h_rowptr, h_colindex, h_val, h_diag);
    if (rc != SPARSH_OK) {
        sparsh_matrix_destroy(A);
        return rc;
    }
    lap("CSR copied");
    choose_twins(A, h_rowptr, h_colindex, h_val, h_diag != nullptr);
    lap("twins built");
    if (!slab_bound()) release_thread_scratch();  // a hierarchy build keeps the encoder's scratch until its thread ends
    *out = A;
    return SPARSH_OK;
}

int sparsh_matrix_update_values(sparsh_matrix_t A, const double *d_val, const double *d_diag) {
    SP_TRY(ensure_init());
    SP_REQUIRE(A != nullptr, "matrix is NULL");
    SP_REQUIRE(d_val != nullptr || A->nnz == 0, "values are NULL");
    NvtxRange nvtx("sparsh:update-values");
    cudaStream_t st = up().stream;
    const int n = A->nrow;
    const size_t nnz = (size_t)A->nnz;
    if (nnz > 0 && d_val != A->val) SP_CUDA(cudaMemcpyAsync(A->val, d_val, sizeof(double) * nnz, cudaMemcpyDeviceToDevice, st));
    // the selection starts again from the row statistics; a forced kernel is forgotten
    A->kind = A->base_kind;
    A->threads = A->base_threads;
    A->lanes = A->base_lanes;
    A->smem_bytes = A->base_smem_bytes;
    A->threads_forced = false;
    // transfer_structure's value scan (one entry per row depends on the sparsity only and is kept)
    if (nnz > 0) {
        struct {
            int differs;
            int pad;
            double v0;
        } h = {0, 0, 0.0};
        int *d_flag = static_cast<int *>(thread_scratch(256));
        SP_REQUIRE(d_flag != nullptr, "value update: no device scratch");
        SP_CUDA(cudaMemsetAsync(d_flag, 0, sizeof(int), st));
        const int grid = (int)std::min<size_t>((nnz + 255) / 256, (size_t)ctx().sm_count * 8);
        uniform_bits_kernel<<<grid, 256, 0, st>>>(nnz, A->val, d_flag);
        count_launch();
        SP_CUDA(cudaMemcpyAsync(&h.differs, d_flag, sizeof(int), cudaMemcpyDeviceToHost, st));
        SP_CUDA(cudaMemcpyAsync(&h.v0, A->val, sizeof(double), cudaMemcpyDeviceToHost, st));
        SP_CUDA(cudaStreamSynchronize(st));
        A->uniform_val = h.differs == 0;
        A->uval = h.v0;
    } else {
        A->uniform_val = false;
        A->uval = 0.0;
    }
    A->agg = A->one_per_row && A->kind == KIND_SCALAR;
    // the smoothing diagonal: the caller's, or extracted as sparsh_matrix_create extracts it
    if (d_diag || n == A->ncol) {
        if (!A->diag) SP_CUDA(dev_alloc(&A->diag, sizeof(double) * ((size_t)n + 1)));
        if (d_diag && d_diag != A->diag && n > 0)
            SP_CUDA(cudaMemcpyAsync(A->diag, d_diag, sizeof(double) * (size_t)n, cudaMemcpyDeviceToDevice, st));
        if (!d_diag && n > 0) {
            diag_extract_kernel<<<(n + 255) / 256, 256, 0, st>>>(n, A->rowptr, A->col, A->val, A->diag);
            count_launch();
            SP_CUDA(cudaGetLastError());
        }
    } else {
        dev_free(A->diag);  // a rectangular matrix has a diagonal only when one is given
        A->diag = nullptr;
    }
    A->has_pat = A->has_dict = false;
    A->n_pat = A->n_pent = A->n_escape = A->pat_far = 0;
    A->n_dval = A->n_doff = 0;
    A->pat0 = Pat0();
    // the encoders' device scratch stays with this thread (grow-only): later updates of the same sizes allocate nothing
    choose_twins(A, nullptr, nullptr, nullptr, d_diag != nullptr);
    SP_CUDA(cudaStreamSynchronize(st));
    SP_CUDA(cudaGetLastError());
    return SPARSH_OK;
}

int sparsh_matrix_fetch(sparsh_matrix_t A, int *h_rowptr, int *h_colindex, double *h_val, double *h_diag) {
    SP_REQUIRE(A != nullptr, "matrix is NULL");
    SP_REQUIRE(!h_diag || A->diag, "matrix has no diagonal");
    cudaStream_t st = ctx().stream;
    SP_CUDA(cudaStreamSynchronize(st));
    if (h_rowptr) SP_TRY(staged_d2h(h_rowptr, A->rowptr, sizeof(int) * ((size_t)A->nrow + 1), st));
    if (h_colindex && A->nnz > 0) SP_TRY(staged_d2h(h_colindex, A->col, sizeof(int) * (size_t)A->nnz, st));
    if (h_val && A->nnz > 0) SP_TRY(staged_d2h(h_val, A->val, sizeof(double) * (size_t)A->nnz, st));
    if (h_diag && A->nrow > 0) SP_TRY(staged_d2h(h_diag, A->diag, sizeof(double) * (size_t)A->nrow, st));
    return SPARSH_OK;
}

int sparsh_dict_encode(int nrow, int ncol, int nnz, const int *rp, const int *ci, const double *v,
                       unsigned short *code, double *dict_val, int *dict_off, int *n_val, int *n_off) {
    SP_TRY(validate(nrow, ncol, nnz, rp, ci));
    SP_REQUIRE(code && dict_val && dict_off && n_val && n_off, "output pointer is NULL");
    std::vector<double> dv;
    std::vector<int> dof;
    *n_val = *n_off = 0;
    if (!dict_encode(nrow, rp, ci, v, code, dv, dof)) return SPARSH_OK;  // not representable: plain CSR is used
    std::copy(dv.begin(), dv.end(), dict_val);
    std::copy(dof.begin(), dof.end(), dict_off);
    *n_val = (int)dv.size();
    *n_off = (int)dof.size();
    return SPARSH_OK;
}

int sparsh_pattern_encode(int nrow, int ncol, int nnz, const int *rp, const int *ci, const double *v,
                          const double *h_diag, unsigned char *pat, double *ent_val, int *ent_off, int *start,
                          int *n_pat, int *n_escape) {
    SP_TRY(validate(nrow, ncol, nnz, rp, ci));
    SP_REQUIRE(pat && ent_val && ent_off && start && n_pat && n_escape, "output pointer is NULL");
    PatternTable T;
    *n_pat = 0;
    *n_escape = nrow;
    if (!pattern_encode(nrow, rp, ci, v, h_diag, pat, T, 0.0)) return SPARSH_OK;  // rows do not repeat: CSR / dict
    std::copy(T.val.begin(), T.val.end(), ent_val);
    std::copy(T.off.begin(), T.off.end(), ent_off);
    std::copy(T.start.begin(), T.start.end(), start);
    *n_pat = (int)T.diag.size();
    *n_escape = T.n_escape;
    return SPARSH_OK;
}

int sparsh_pattern_masks(int n_pat, const int *start, const double *ent_val, const int *ent_off, unsigned char *mask) {
    SP_REQUIRE(start && ent_val && ent_off && mask, "pointer is NULL");
    SP_REQUIRE(n_pat >= 0 && n_pat <= PAT_ESCAPE, "n_pat out of range");  // ids 0..254; 255 is the escape
    SP_REQUIRE(n_pat == 0 || start[0] == 0, "start[0] != 0");
    for (int p = 0; p < n_pat; p++) SP_REQUIRE(start[p] <= start[p + 1], "start not monotone");
    SP_REQUIRE(n_pat == 0 || start[n_pat] <= PAT_MAX_ENT, "more table entries than a pattern table holds");
    PatternTable T;
    if (n_pat > 0) {
        T.start.assign(start, start + n_pat + 1);
        T.val.assign(ent_val, ent_val + start[n_pat]);
        T.off.assign(ent_off, ent_off + start[n_pat]);
    }
    for (int p = 0; p < n_pat; p++) {  // the tabulated diagonal: the pattern's first offset-0 entry, else 0
        double d = 0.0;
        for (int k = start[p]; k < start[p + 1]; k++)
            if (ent_off[k] == 0) {
                d = ent_val[k];
                break;
            }
        T.diag.push_back(d);
    }
    pattern_masks(T, mask);
    return SPARSH_OK;
}

int sparsh_matrix_create_transpose(int nrow, int ncol, int nnz, const int *rp, const int *ci, const double *v,
                                   sparsh_matrix_t *out) {
    SP_TRY(ensure_init());
    SP_TRY(validate(nrow, ncol, nnz, rp, ci));
    // stable counting sort: row c of the transpose lists the source rows in ascending order, which is the order
    // in which the reference's transposed product scatters into b_c[c] (src/AMG_cycle_utilities.cpp:102)
    std::vector<int> trp((size_t)ncol + 1, 0), tci((size_t)std::max(nnz, 1));
    std::vector<double> tv((size_t)std::max(nnz, 1));
    for (int j = 0; j < nnz; j++) trp[ci[j] + 1]++;
    for (int c = 0; c < ncol; c++) trp[c + 1] += trp[c];
    std::vector<int> cur(trp.begin(), trp.end() - 1);
    for (int i = 0; i < nrow; i++)
        for (int j = rp[i]; j < rp[i + 1]; j++) {
            int d = cur[ci[j]]++;
            tci[d] = i;
            tv[d] = v[j];
        }
    return sparsh_matrix_create(ncol, nrow, nnz, trp.data(), tci.data(), tv.data(), nullptr, out);
}

int sparsh_matrix_destroy(sparsh_matrix_t A) {
    if (!A) return SPARSH_OK;
    dev_free(A->rowptr);
    dev_free(A->col);
    dev_free(A->val);
    dev_free(A->diag);
    dev_free(A->code);
    dev_free(A->dict_val);
    dev_free(A->dict_off);
    dev_free(A->pat);
    dev_free(A->pat_ent);
    dev_free(A->pat_start);
    dev_free(A->pat_diag);
    delete A;
    return SPARSH_OK;
}

int sparsh_matrix_dims(sparsh_matrix_t A, int *nrow, int *ncol, int *nnz) {
    SP_REQUIRE(A != nullptr, "matrix is NULL");
    if (nrow) *nrow = A->nrow;
    if (ncol) *ncol = A->ncol;
    if (nnz) *nnz = A->nnz;
    return SPARSH_OK;
}

int sparsh_matrix_kernel(sparsh_matrix_t A, int *kind, int *threads_or_lanes, int *smem_bytes) {
    SP_REQUIRE(A != nullptr, "matrix is NULL");
    if (kind) *kind = A->kind;
    if (threads_or_lanes) *threads_or_lanes = A->kind == KIND_VECTOR ? A->lanes : A->threads;
    if (smem_bytes) *smem_bytes = A->kind == KIND_STREAM ? A->smem_bytes : 0;
    if (smem_bytes && A->kind == KIND_DICT)
        *smem_bytes = ((((A->threads == 256 ? A->win256 : A->win128) + 16) + 7) & ~7) * 2 + A->n_dval * 8 + A->n_doff * 4;
    return SPARSH_OK;
}

// statistics of the csr-pattern8 twin as the device encoder built it (n_pat == 0: no twin)
int sparsh_matrix_pattern_stats(sparsh_matrix_t A, int *n_pat, int *n_ent, int *n_escape, double *cover0) {
    SP_REQUIRE(A != nullptr, "matrix is NULL");
    if (n_pat) *n_pat = A->has_pat ? A->n_pat : 0;
    if (n_ent) *n_ent = A->has_pat ? A->n_pent : 0;
    if (n_escape) *n_escape = A->has_pat ? A->n_escape : A->nrow;
    if (cover0) *cover0 = A->has_pat ? A->pat0.cover : 0.0;
    return SPARSH_OK;
}

int sparsh_matrix_pattern_mask_stats(sparsh_matrix_t A, int *n_masked, double *cover_masked) {
    SP_REQUIRE(A != nullptr, "matrix is NULL");
    int m = 0;
    if (A->has_pat)
        for (int p = 1; p < A->n_pat; p++) m += (A->pat0.mask[p] & PAT_MASK_VALID) != 0;
    if (n_masked) *n_masked = m;
    if (cover_masked) *cover_masked = A->has_pat ? A->pat0.cover_masked : 0.0;
    return SPARSH_OK;
}

int sparsh_matrix_transfer_info(sparsh_matrix_t A, int *one_per_row, int *uniform_val, double *value) {
    SP_REQUIRE(A != nullptr, "matrix is NULL");
    if (one_per_row) *one_per_row = A->one_per_row ? 1 : 0;
    if (uniform_val) *uniform_val = A->uniform_val ? 1 : 0;
    if (value) *value = A->uniform_val ? A->uval : 0.0;
    return SPARSH_OK;
}

// name of the kernel instantiation launch_csr picks for this matrix and epilogue (reports: bench.py's roofline / kernel
// table must name what really ran)
int sparsh_matrix_kernel_name(sparsh_matrix_t A, int epi, char *buf, size_t len) {
    SP_REQUIRE(A != nullptr && buf != nullptr && len > 0, "bad arguments");
    static const char *epis[] = {"EPI_SPMV", "EPI_RESID", "EPI_JACOBI", "EPI_PROLONG", "EPI_SOR", "EPI_SPMV_DOT", "EPI_RESNORM"};
    SP_REQUIRE(epi >= 0 && epi < 7, "unknown epilogue");
    char tmp[160];
    switch (A->kind) {
        case KIND_SCALAR:
            if (A->agg && (epi == EPI_SPMV || epi == EPI_PROLONG))
                std::snprintf(tmp, sizeof tmp, "csr_agg_kernel<%s,%s>", epis[epi], A->uniform_val ? "true" : "false");
            else
                std::snprintf(tmp, sizeof tmp, "csr_scalar_kernel<256,%s>", epis[epi]);
            break;
        case KIND_STREAM:
            std::snprintf(tmp, sizeof tmp, "csr_stream_kernel<%d,%s>", A->threads, epis[epi]);
            break;
        case KIND_DICT:
            std::snprintf(tmp, sizeof tmp, "csr_dict_kernel<%d,4,%s>", A->threads, epis[epi]);
            break;
        case KIND_PATTERN:
            if (pattern_lean_applies(A)) {
                const bool div = epi == EPI_JACOBI || epi == EPI_SOR;
                const bool one_row = A->threads_forced ? A->threads == 256 : div;
                std::snprintf(tmp, sizeof tmp, "csr_pat2_kernel<%d,%d,%d,%s>", one_row ? 256 : 128, one_row ? 1 : 2, A->pat0.len, epis[epi]);
            } else {
                std::snprintf(tmp, sizeof tmp, "csr_pattern_kernel<%d,4,2,%s>", A->threads, epis[epi]);
            }
            break;
        default:
            std::snprintf(tmp, sizeof tmp, "csr_vector_kernel<%d,%s>", A->lanes, epis[epi]);
    }
    std::snprintf(buf, len, "%s", tmp);
    return SPARSH_OK;
}

int sparsh_matrix_force_kernel(sparsh_matrix_t A, int kind, int tl) {
    SP_REQUIRE(A != nullptr, "matrix is NULL");
    A->agg = false;  // a forced kind runs that family's kernel: KIND_SCALAR is csr_scalar_kernel even for one entry per row
    if (kind == KIND_SCALAR) {
        A->kind = kind;
        A->threads = 256;
    } else if (kind == KIND_STREAM) {
        SP_REQUIRE(tl == 128 || tl == 256, "stream kernel: threads must be 128 or 256");
        const int win = tl == 256 ? A->win256 : A->win128;
        const int smem = (((win + 8) + 3) & ~3) * 12;
        SP_REQUIRE(smem <= 200 * 1024, "stream kernel: row window does not fit in shared memory");
        A->kind = kind;
        A->threads = tl;
        A->smem_bytes = smem;
    } else if (kind == KIND_DICT) {
        SP_REQUIRE(A->has_dict, "dict kernel: this matrix has no csr-dict16 twin (more than 256 distinct values or offsets)");
        SP_REQUIRE(tl == 128 || tl == 256, "dict kernel: threads must be 128 or 256");
        A->kind = kind;
        A->threads = tl;
    } else if (kind == KIND_PATTERN) {
        SP_REQUIRE(A->has_pat, "pattern kernel: this matrix has no csr-pattern8 twin (SPARSH_PATTERN unset, or rows do not repeat)");
        SP_REQUIRE(tl == 128 || tl == 256, "pattern kernel: threads must be 128 or 256");
        A->kind = kind;
        A->threads = tl;
        A->threads_forced = true;
    } else if (kind == KIND_VECTOR) {
        SP_REQUIRE(tl == 2 || tl == 4 || tl == 8 || tl == 16 || tl == 32, "vector kernel: lanes must be 2..32");
        A->kind = kind;
        A->lanes = tl;
    } else {
        SP_REQUIRE(false, "unknown kernel kind");
    }
    return SPARSH_OK;
}

// ---- per-op entry points -------------------------------------------------------------------------------------
int sparsh_spmv(sparsh_matrix_t A, const double *d_x, double *d_y) {
    SP_REQUIRE(A != nullptr, "matrix is NULL");
    return launch_csr(A, EPI_SPMV, d_x, d_y, EpiArgs(), 0, A->nrow);
}

int sparsh_spmv_dot(sparsh_matrix_t A, const double *d_x, double *d_y, double *d_dot) {
    SP_REQUIRE(A != nullptr && A->nrow == A->ncol, "spmv_dot needs a square matrix");
    EpiArgs a;
    a.xi = d_x;
    a.red_out = d_dot;
    return launch_csr(A, EPI_SPMV_DOT, d_x, d_y, a, 0, A->nrow);
}

int sparsh_residual(sparsh_matrix_t A, const double *d_b, const double *d_x, double *d_r) {
    SP_REQUIRE(A != nullptr, "matrix is NULL");
    EpiArgs a;
    a.b = d_b;
    return launch_csr(A, EPI_RESID, d_x, d_r, a, 0, A->nrow);
}

int sparsh_residual_norm(sparsh_matrix_t A, const double *d_b, const double *d_x, double *h_norm) {
    SP_REQUIRE(A != nullptr, "matrix is NULL");
    Context &c = ctx();
    EpiArgs a;
    a.b = d_b;
    a.red_out = c.d_scalar;
    SP_TRY(launch_csr(A, EPI_RESNORM, d_x, nullptr, a, 0, A->nrow));
    SP_CUDA(cudaMemcpyAsync(c.h_scalar, c.d_scalar, sizeof(double), cudaMemcpyDeviceToHost, c.stream));
    SP_CUDA(cudaStreamSynchronize(c.stream));
    *h_norm = solve_residual(c.h_scalar[0]);
    return SPARSH_OK;
}

int sparsh_jacobi(sparsh_matrix_t A, const double *d_b, double *d_x, double *d_tmp, double omega, int sweeps) {
    SP_REQUIRE(A != nullptr && A->diag != nullptr, "jacobi needs a square matrix with a diagonal");
    SP_REQUIRE(sweeps >= 0, "negative sweep count");
    double *cur = d_x, *other = d_tmp;
    for (int s = 0; s < sweeps; s++) {
        EpiArgs a;
        a.b = d_b;
        a.xi = cur;
        a.d = A->diag;
        a.omega = omega;
        SP_TRY(launch_csr(A, EPI_JACOBI, cur, other, a, 0, A->nrow));
        std::swap(cur, other);
    }
    if (cur != d_x) SP_CUDA(cudaMemcpyAsync(d_x, cur, sizeof(double) * (size_t)A->nrow, cudaMemcpyDeviceToDevice, ctx().stream));
    return SPARSH_OK;
}

int sparsh_jacobi_zero(sparsh_matrix_t A, const double *d_b, double omega, double *d_x) {
    SP_REQUIRE(A != nullptr && A->diag != nullptr, "jacobi needs a square matrix with a diagonal");
    if (jacobi_zero_pat_applies(A)) return launch_jacobi_zero_pat(A, d_b, omega, d_x);
    return k_jacobi_zero((size_t)A->nrow, d_b, A->diag, omega, d_x);
}

int sparsh_mc_sor(sparsh_matrix_t A, const int *h_color_count, int total_colors, const double *d_b, double *d_x,
                  double omega, int sweeps) {
    SP_REQUIRE(A != nullptr && A->diag != nullptr, "mc_sor needs a square matrix with a diagonal");
    SP_REQUIRE(h_color_count != nullptr && total_colors >= 0, "bad colour table");
    SP_REQUIRE(h_color_count[0] == 0 && h_color_count[total_colors] == A->nrow, "colour offsets do not cover the rows");
    for (int s = 0; s < sweeps; s++)
        for (int k = 0; k < total_colors; k++) {
            EpiArgs a;
            a.b = d_b;
            a.d = A->diag;
            a.omega = omega;
            SP_TRY(launch_csr(A, EPI_SOR, d_x, d_x, a, h_color_count[k], h_color_count[k + 1]));
        }
    return SPARSH_OK;
}

int sparsh_restrict(sparsh_matrix_t R, const double *d_r, double *d_bc) {
    SP_REQUIRE(R != nullptr, "matrix is NULL");
    return launch_csr(R, EPI_SPMV, d_r, d_bc, EpiArgs(), 0, R->nrow);
}

int sparsh_residual_restrict(sparsh_matrix_t A, sparsh_matrix_t R, const double *d_b, const double *d_x, double *d_bc) {
    SP_REQUIRE(A != nullptr && R != nullptr, "matrix is NULL");
    SP_REQUIRE(R->ncol == A->nrow, "R's column count differs from A's row count");
    if (resid_restrict_applies(A, R)) return launch_resid_restrict(A, R, d_b, d_x, d_bc);
    // the two launches the fused kernel replaces, through a temporary residual
    double *r = nullptr;
    SP_CUDA(cudaMalloc(&r, sizeof(double) * ((size_t)A->nrow + 1)));
    EpiArgs a;
    a.b = d_b;
    int rc = launch_csr(A, EPI_RESID, d_x, r, a, 0, A->nrow);
    if (rc == SPARSH_OK) rc = launch_csr(R, EPI_SPMV, r, d_bc, EpiArgs(), 0, R->nrow);
    const cudaError_t e = cudaStreamSynchronize(ctx().stream);
    cudaFree(r);
    SP_TRY(rc);
    SP_CUDA(e);
    return SPARSH_OK;
}

int sparsh_prolong_add(sparsh_matrix_t P, const double *d_xc, double *d_xf) {
    SP_REQUIRE(P != nullptr, "matrix is NULL");
    return launch_csr(P, EPI_PROLONG, d_xc, d_xf, EpiArgs(), 0, P->nrow);
}

}  // extern "C"

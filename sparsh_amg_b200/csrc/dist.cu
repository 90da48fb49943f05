// dist.cu — multi-GPU solve phase (SURVEY §8e): one process per GPU, NVLink 5 / NVSwitch.
//
// The reference has no distributed path (no MPI/NCCL anywhere).  This file row-partitions the same V-cycle / PCG:
//   * operators: each rank owns a row block of A_l, P_l and R_l = P_l^T with columns relabelled to [owned | halo]
//     positions (built on the host by host/dist_plan.cpp); the per-row entry order is preserved, so every row sum is
//     bit-identical to the single-GPU one and only the reductions (dot products) see a different summation tree;
//   * halo exchange, halo_mode 1 (default): every vector that can receive halo data lives in one cudaMalloc'ed ARENA per
//     rank that all ranks map through CUDA IPC.  The packing kernel stores the boundary entries STRAIGHT INTO THE
//     NEIGHBOUR'S HALO SEGMENT over NVLink (peer stores), fences, and raises a sequence flag in the neighbour's memory;
//     the consumer's boundary-strip kernel (rows that read the halo) waits on those flags at CTA start (acquire,
//     system scope) and acks from its last CTA, while the interior rows run concurrently on the main stream.  For Jacobi
//     sweeps the exchange disappears into the compute kernel altogether: the boundary-strip kernel stores each new
//     value it produces BOTH locally and into the neighbour's halo segment of the next sweep's input vector and signals
//     when done (fused compute + communication over peer memory).  Sequence counters live in device memory, so all of
//     it replays inside a CUDA graph: no NCCL call, host round trip or staging copy sits on the exchange path;
//   * halo_mode 0: pack kernel -> grouped ncclSend/ncclRecv into the halo tail on a communication stream (fallback);
//     Boundary strips run beside the interior rows (auxiliary high-priority stream; the fused reductions, which need one
//     grid, as its first CTAs): they wait for the flags and signal as soon as the last of them is done; interior rows
//     never wait;
//   * Krylov scalars: local fixed-tree partial, then a one-warp kernel stores it into a slot of every peer's arena,
//     waits for the peers' slots and adds them in rank order (deterministic, graph-replayable; ~one NVLink round trip).
//     The handshake error flag rides along, so every rank learns of a failure in the same iteration;
//   * small levels: every rank stores its part of the restricted right-hand side straight into all peers' copy of the
//     replicated vector (flags + acks as above) and the levels are solved redundantly on every GPU by the single-GPU
//     hierarchy code (levels whose halo would exceed their interior are latency-bound on a partitioned layout).
//   In halo_mode 1 no NCCL call is left on the iteration path (NCCL bootstraps the IPC handles at setup); halo_mode 0
//   keeps ncclSend/ncclRecv + ncclAllReduce + ncclAllGather as the reference point.
#include <nccl.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <utility>
#include <vector>

#include "hierarchy.cuh"

using namespace sparsh;

namespace {

constexpr int MAX_NBR = 8;
typedef unsigned long long u64;

struct Comm {
    ncclComm_t comm = nullptr;
    int nranks = 1, rank = 0;
    cudaStream_t comm_stream = nullptr;
    cudaEvent_t ev_ready = nullptr, ev_done = nullptr;
};
Comm &comm() {
    static Comm c;
    return c;
}

int nccl_fail(ncclResult_t r, const char *what, int line) {
    set_error(std::string("NCCL error at dist.cu:") + std::to_string(line) + " " + what + ": " + ncclGetErrorString(r));
    return SPARSH_ERR_CUDA;
}
#define SP_NCCL(call)                                          \
    do {                                                       \
        ncclResult_t r__ = (call);                             \
        if (r__ != ncclSuccess) return nccl_fail(r__, #call, __LINE__); \
    } while (0)

struct DistOp {
    sparsh_matrix_s *M = nullptr;
    int id = 0;  // flag slot
    int nrow = 0, ncol_local = 0, nhalo = 0, shift = 0;  // halo segment starts at ncol_local + shift
    std::vector<int> send_rank, send_ptr, recv_rank, recv_ptr;
    std::vector<long long> peer_dst_off;  // per send neighbour: element offset of my slice inside ITS input vector
    int *d_send_idx = nullptr;
    double *d_sendbuf = nullptr;  // NCCL mode only
    int *d_pm_ptr = nullptr, *d_pm_nbr = nullptr, *d_pm_off = nullptr;  // A ops: row -> (neighbour slot, position) it is sent to
    int ib = 0, ie = 0;
    bool needs_exchange() const { return !send_rank.empty() || !recv_rank.empty(); }
};

struct DistLevel {
    DistOp A, P, R;
    int n = 0;       // owned rows of this level
    int n_next = 0;  // owned rows of the next level
    double *xbuf = nullptr, *tbuf = nullptr;  // [owned | halo(A_l) | halo(P_{l-1})]
    double *bbuf = nullptr;                   // owned (levels >= 1)
    double *rbuf = nullptr;                   // [owned | halo(R_l)]
    size_t xcap = 0;
};

// ---- device-side signalling ---------------------------------------------------------------------------------------
__device__ __forceinline__ u64 ld_acquire_sys(const u64 *p) {
    u64 v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(u64 *p, u64 v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_sys(u64 *p, u64 v) {
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ long long wall_ns() {
    long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
// spin until *p >= want; gives up after timeout_ns of wall clock and raises *err so a broken handshake can never hang
// the GPU (ranks may legitimately be seconds apart: graph instantiation, lazy module loads, a profiler replay)
__device__ __forceinline__ void spin_until(const u64 *p, u64 want, int *err, long long timeout_ns) {
    if (ld_acquire_sys(p) >= want) return;
    const long long t0 = wall_ns();
    while (ld_acquire_sys(p) < want) {
        if (*reinterpret_cast<volatile int *>(err) != 0) break;
        if (wall_ns() - t0 > timeout_ns) {
            atomicExch(err, 1);
            break;
        }
        __nanosleep(64);
    }
}
__device__ __forceinline__ double ld_relaxed_sys_f64(const double *p) {
    double v;
    asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_sys_f64(double *p, double v) {
    asm volatile("st.relaxed.sys.global.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}

struct PushArgs {
    int nnbr;
    int ptr[MAX_NBR + 1];          // prefix offsets into the send list
    double *dst[MAX_NBR];          // peer address of my slice in the neighbour's halo segment
    u64 *flag_dst[MAX_NBR];        // neighbour's "data from <me> for op" flag
    const u64 *ack_local[MAX_NBR]; // my "neighbour has consumed my previous slice" flag
};

// producer: wait until the neighbours have consumed the previous slice, store the boundary entries into their halo
// segments over NVLink, fence, raise the flags (last block to finish)
__global__ void __launch_bounds__(256)
    push_kernel(const double *__restrict__ x, const int *__restrict__ send_idx, int total, PushArgs a, u64 *seq,
                unsigned int *ticket, int *err, long long timeout_ns) {
    __shared__ u64 s_prev;
    if (threadIdx.x == 0) s_prev = *reinterpret_cast<volatile u64 *>(seq);
    __syncthreads();
    const u64 prev = s_prev;
    if (threadIdx.x < a.nnbr) spin_until(a.ack_local[threadIdx.x], prev, err, timeout_ns);
    __syncthreads();
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i < total) {
        int q = 0;
#pragma unroll
        for (int k = 1; k < MAX_NBR; k++)
            if (k < a.nnbr && i >= a.ptr[k]) q = k;
        a.dst[q][i - a.ptr[q]] = x[send_idx[i]];
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int t = atomicAdd(ticket, 1u);
        if (t == gridDim.x - 1) {
            __threadfence_system();  // one fence, then the flags back to back (relaxed stores behind a fence: release)
            for (int q = 0; q < a.nnbr; q++) st_relaxed_sys(a.flag_dst[q], prev + 1);
            *reinterpret_cast<volatile u64 *>(seq) = prev + 1;
            *ticket = 0u;
            __threadfence();
        }
    }
}

struct WaitArgs {
    int nnbr;
    const u64 *flag_local[MAX_NBR];  // "data from neighbour q has landed" flags in my memory
    u64 *ack_dst[MAX_NBR];           // neighbour q's ack slot for me
};
__global__ void __launch_bounds__(256) pack_kernel(const double *__restrict__ x, const int *__restrict__ idx, int n, double *out) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i < n) out[i] = x[idx[i]];
}
// scatter the padded all-gather buffer into the replicated coarse vector: full[map[i]] = gathered[i]
__global__ void __launch_bounds__(256) scatter_map_kernel(const double *__restrict__ src, const int *__restrict__ map, int n, double *dst) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i < n) {
        const int g = map[i];
        if (g >= 0) dst[g] = src[i];
    }
}
__global__ void __launch_bounds__(256) gather_rows_kernel(const double *__restrict__ src, const int *__restrict__ rows, int n, double *dst) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i < n) dst[i] = src[rows[i]];
}

// ---- collectives over peer memory (halo_mode 1): no NCCL kernel on the iteration path -------------------------------
// Shared block at the same offset of every rank's arena.  Slots are double-buffered by the parity of the sequence number:
// a rank can be at most one collective ahead of a peer that has not read its slot yet (it needs that peer's NEXT
// contribution to get any further).
constexpr int RED_SLOTS = 4;  // up to 3 values + the error flag
struct CollArea {
    u64 red_flag[2][MAX_NBR];
    double red_val[2][MAX_NBR][RED_SLOTS];
    u64 tail_flag[MAX_NBR];  // "rank r's part of the replicated right-hand side has landed", sequence number
    u64 tail_ack[MAX_NBR];   // "rank r has finished the replicated levels of cycle k": my copy may be overwritten
};
struct PeerTab {
    int nranks, rank;
    char *base[MAX_NBR];  // mapped arena of every rank (own arena for `rank`)
};

// In-place all-reduce (sum) of `count` <= 3 device scalars; one thread per rank.  Every rank stores its values into
// slot [rank] of every peer, raises that peer's flag, waits for all flags in its own arena and adds the slots in RANK
// ORDER: every rank computes the same bits.  *err travels in the spare slot: after the call it is set on all ranks
// if it was set on any, so the host loops of all ranks leave in the same iteration.
__global__ void __launch_bounds__(32)
    peer_allreduce_kernel(double *vals, int count, PeerTab tab, size_t coll_off, u64 *seq, int *err, long long timeout_ns) {
    __shared__ double sv[MAX_NBR][RED_SLOTS];
    const int t = threadIdx.x;
    const u64 k = *reinterpret_cast<volatile u64 *>(seq) + 1;
    const int par = (int)(k & 1);
    if (t < tab.nranks) {
        CollArea *dst = reinterpret_cast<CollArea *>(tab.base[t] + coll_off);
        for (int i = 0; i < count; i++) st_relaxed_sys_f64(&dst->red_val[par][tab.rank][i], vals[i]);
        st_relaxed_sys_f64(&dst->red_val[par][tab.rank][RED_SLOTS - 1], *reinterpret_cast<volatile int *>(err) ? 1.0 : 0.0);
        __threadfence_system();
        st_release_sys(&dst->red_flag[par][tab.rank], k);
        CollArea *mine = reinterpret_cast<CollArea *>(tab.base[tab.rank] + coll_off);
        spin_until(&mine->red_flag[par][t], k, err, timeout_ns);
        for (int i = 0; i < count; i++) sv[t][i] = ld_relaxed_sys_f64(&mine->red_val[par][t][i]);
        sv[t][RED_SLOTS - 1] = ld_relaxed_sys_f64(&mine->red_val[par][t][RED_SLOTS - 1]);
    }
    __syncthreads();
    if (t == 0) {
        for (int i = 0; i < count; i++) {
            double acc = 0.0;
            for (int r = 0; r < tab.nranks; r++) acc = __dadd_rn(acc, sv[r][i]);
            vals[i] = acc;
        }
        bool bad = false;
        for (int r = 0; r < tab.nranks; r++) bad = bad || sv[r][RED_SLOTS - 1] != 0.0;
        if (bad) atomicExch(err, 1);
        *reinterpret_cast<volatile u64 *>(seq) = k;
    }
}

// Replicated right-hand side: every rank stores its owned entries (global ids `rows`) into ALL ranks' copy of the
// vector (own copy included), the last CTA raises the flags and then waits until every rank's part has landed here, so
// the kernels that follow in the stream see the complete vector.  Before overwriting, every CTA makes sure all ranks
// have finished the replicated levels of the previous cycle (acks raised by tail_ack_kernel).
__global__ void __launch_bounds__(256)
    tail_exchange_kernel(const double *__restrict__ src, const int *__restrict__ rows, int n_own, PeerTab tab, size_t vec_off,
                         size_t coll_off, u64 *seq, unsigned int *ticket, int *err, long long timeout_ns) {
    __shared__ u64 s_prev;
    __shared__ int s_last;
    if (threadIdx.x == 0) s_prev = *reinterpret_cast<volatile u64 *>(seq);
    __syncthreads();
    const u64 prev = s_prev;
    CollArea *mine = reinterpret_cast<CollArea *>(tab.base[tab.rank] + coll_off);
    if (threadIdx.x < tab.nranks) spin_until(&mine->tail_ack[threadIdx.x], prev, err, timeout_ns);
    __syncthreads();
    for (int i = blockIdx.x * 256 + threadIdx.x; i < n_own; i += gridDim.x * 256) {
        const double v = src[i];
        const int g = rows[i];
        for (int q = 0; q < tab.nranks; q++) reinterpret_cast<double *>(tab.base[q] + vec_off)[g] = v;
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (s_last) {
        if (threadIdx.x < tab.nranks) {
            __threadfence_system();
            CollArea *dst = reinterpret_cast<CollArea *>(tab.base[threadIdx.x] + coll_off);
            st_release_sys(&dst->tail_flag[tab.rank], prev + 1);
            spin_until(&mine->tail_flag[threadIdx.x], prev + 1, err, timeout_ns);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            *reinterpret_cast<volatile u64 *>(seq) = prev + 1;
            *ticket = 0u;
            __threadfence();
        }
    }
}
// the replicated levels of this cycle are done on this rank: gather the owned entries of the correction and tell every
// rank that its next right-hand side may overwrite my copy
__global__ void __launch_bounds__(256)
    tail_gather_ack_kernel(const double *__restrict__ src, const int *__restrict__ rows, int n, double *dst, PeerTab tab,
                           size_t coll_off, const u64 *seq) {
    for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) dst[i] = src[rows[i]];
    if (blockIdx.x == 0 && threadIdx.x < tab.nranks) {
        const u64 k = *reinterpret_cast<const volatile u64 *>(seq);
        CollArea *peer = reinterpret_cast<CollArea *>(tab.base[threadIdx.x] + coll_off);
        st_release_sys(&peer->tail_ack[tab.rank], k);
    }
}

}  // namespace

struct sparsh_dist_s {
    std::vector<DistLevel> lev;          // distributed levels 0..nd-1
    sparsh_hierarchy_s *tail = nullptr;  // replicated levels nd..L
    sparsh_params prm;
    int n_tail0 = 0;      // global rows of the first replicated level
    int tail_maxc = 0;    // padded per-rank count for the all-gather
    int n_own_tail0 = 0;  // rows of that level owned by this rank
    double *tail_send = nullptr, *tail_recv = nullptr, *tail_b = nullptr, *tail_x = nullptr;
    int *d_tail_map = nullptr, *d_tail_rows = nullptr;
    double *xtail_local = nullptr;  // owned part of X at level nd, [owned | halo(P_{nd-1})]
    double *btail_local = nullptr;
    // Krylov
    double *kv[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    double *bv[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};  // BiCGStab: vectors no operator gathers from
    double *d_sc = nullptr, *h_sc = nullptr;
    std::vector<GraphEntry> graphs;
    // arena shared through CUDA IPC: [flags | vectors]
    char *arena = nullptr;
    size_t arena_bytes = 0;
    bool peer = false;
    int nops = 0;
    std::vector<char *> peer_base;                    // [rank] mapped base of its arena (own base for me)
    std::vector<std::pair<double *, size_t>> bufs;    // my halo-capable vectors: (pointer, byte offset in the arena)
    std::vector<std::vector<long long>> peer_buf_off; // [rank][buffer id] byte offset in that rank's arena
    u64 *seq = nullptr, *expect = nullptr;            // device counters per op (push / wait side)
    unsigned int *ticket = nullptr, *ticket2 = nullptr;  // last-block tickets: producers / consumers
    std::vector<int> buf_level;       // buffer id -> level whose A operator reads it (-1: none)
    std::vector<int> halo_ready;      // buffer id -> (op id + 1) whose halo slices the producing kernel already pushed, 0 = none
    double **d_pm_tab = nullptr;      // [buffer id][neighbour slot] peer address of my slice (fused Jacobi push)
    int *d_err = nullptr, *h_err = nullptr;
    // peer-memory collectives (CollArea at byte offset coll_off of every arena)
    size_t coll_off = 0, tailb_off = 0;
    u64 *red_seq = nullptr, *tail_seq = nullptr;
    unsigned int *tail_ticket = nullptr;
    long long timeout_ns = 10000000000ll;  // SPARSH_HALO_TIMEOUT_MS overrides (default 10 s)
    bool dead = false;                     // a handshake timed out: flags and counters are out of step for good
};

namespace {

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// halo segments start on a 128-byte boundary of their vector: a cache line never mixes owned entries (which the
// interior rows of a co-resident CTA may pull into L1) with halo entries (which peers overwrite over NVLink)
inline int align16(int n) { return (n + 15) & ~15; }

int make_op(const sparsh_dist_op_desc &d, int halo_start, int id, DistOp &op) {
    const int shift = halo_start - d.ncol_local;
    SP_REQUIRE(shift >= 0, "halo segment overlaps the owned entries");
    op.id = id;
    op.nrow = d.nrow;
    op.ncol_local = d.ncol_local;
    op.nhalo = d.nhalo;
    op.shift = shift;
    op.ib = d.interior_begin;
    op.ie = d.interior_end;
    // halo columns move behind the halo segment of the operator that shares this vector space (see DistLevel)
    std::vector<int> ci;
    const int *cols = d.colindex;
    if (shift > 0) {
        ci.assign(d.colindex, d.colindex + d.nnz);
        for (int &c : ci)
            if (c >= d.ncol_local) c += shift;
        cols = ci.data();
    }
    SP_TRY(sparsh_matrix_create(d.nrow, d.ncol_local + shift + d.nhalo, d.nnz, d.rowptr, cols, d.val, d.diag, &op.M));
    op.send_rank.assign(d.send_rank, d.send_rank + d.n_send);
    op.send_ptr.assign(d.send_ptr, d.send_ptr + d.n_send + 1);
    op.recv_rank.assign(d.recv_rank, d.recv_rank + d.n_recv);
    op.recv_ptr.assign(d.recv_ptr, d.recv_ptr + d.n_recv + 1);
    const int total = d.n_send ? d.send_ptr[d.n_send] : 0;
    if (total > 0) {
        SP_CUDA(cudaMalloc(&op.d_send_idx, sizeof(int) * (size_t)total));
        SP_CUDA(cudaMalloc(&op.d_sendbuf, sizeof(double) * (size_t)total));
        SP_CUDA(cudaMemcpy(op.d_send_idx, d.send_idx, sizeof(int) * (size_t)total, cudaMemcpyHostToDevice));
    }
    return SPARSH_OK;
}
// rows of a square operator that some neighbour needs, as a CSR over the local rows (for the fused Jacobi push)
int make_push_map(const sparsh_dist_op_desc &d, DistOp &op) {
    std::vector<int> ptr((size_t)d.nrow + 1, 0);
    const int total = d.n_send ? d.send_ptr[d.n_send] : 0;
    for (int k = 0; k < total; k++) ptr[d.send_idx[k] + 1]++;
    for (int i = 0; i < d.nrow; i++) ptr[i + 1] += ptr[i];
    std::vector<int> nbr((size_t)std::max(total, 1)), off((size_t)std::max(total, 1)), cur(ptr.begin(), ptr.end() - 1);
    for (int s = 0; s < d.n_send; s++)
        for (int k = d.send_ptr[s]; k < d.send_ptr[s + 1]; k++) {
            const int pos = cur[d.send_idx[k]]++;
            nbr[pos] = s;
            off[pos] = k - d.send_ptr[s];
        }
    SP_CUDA(cudaMalloc(&op.d_pm_ptr, sizeof(int) * ptr.size()));
    SP_CUDA(cudaMalloc(&op.d_pm_nbr, sizeof(int) * nbr.size()));
    SP_CUDA(cudaMalloc(&op.d_pm_off, sizeof(int) * off.size()));
    SP_CUDA(cudaMemcpy(op.d_pm_ptr, ptr.data(), sizeof(int) * ptr.size(), cudaMemcpyHostToDevice));
    SP_CUDA(cudaMemcpy(op.d_pm_nbr, nbr.data(), sizeof(int) * nbr.size(), cudaMemcpyHostToDevice));
    SP_CUDA(cudaMemcpy(op.d_pm_off, off.data(), sizeof(int) * off.size(), cudaMemcpyHostToDevice));
    return SPARSH_OK;
}
void free_op(DistOp &op) {
    sparsh_matrix_destroy(op.M);
    cudaFree(op.d_send_idx);
    cudaFree(op.d_sendbuf);
    cudaFree(op.d_pm_ptr);
    cudaFree(op.d_pm_nbr);
    cudaFree(op.d_pm_off);
}

u64 *flag_slot(char *base, int nranks, int op, int kind, int r) {
    return reinterpret_cast<u64 *>(base) + ((size_t)(op * 2 + kind) * nranks + r);
}

int buffer_id(const sparsh_dist_s *h, const double *x) {
    for (size_t i = 0; i < h->bufs.size(); i++)
        if (h->bufs[i].first == x) return (int)i;
    return -1;
}

// ---- halo_mode 1: NVLink peer pushes --------------------------------------------------------------------------------
int peer_push(sparsh_dist_s *h, const DistOp &op, double *x) {
    if (op.send_rank.empty()) return SPARSH_OK;
    Context &c = ctx();
    Comm &m = comm();
    const int bid = buffer_id(h, x);
    SP_REQUIRE(bid >= 0, "halo exchange on a vector that is not in the shared arena");
    PushArgs a;
    std::memset(&a, 0, sizeof a);
    a.nnbr = (int)op.send_rank.size();
    for (int s = 0; s < a.nnbr; s++) {
        const int q = op.send_rank[s];
        a.ptr[s] = op.send_ptr[s];
        a.dst[s] = reinterpret_cast<double *>(h->peer_base[q] + h->peer_buf_off[q][bid]) + op.peer_dst_off[s];
        a.flag_dst[s] = flag_slot(h->peer_base[q], m.nranks, op.id, 0, m.rank);
        a.ack_local[s] = flag_slot(h->arena, m.nranks, op.id, 1, q);
    }
    a.ptr[a.nnbr] = op.send_ptr[a.nnbr];
    const int total = op.send_ptr.back();
    push_kernel<<<(total + 255) / 256, 256, 0, c.stream>>>(x, op.d_send_idx, total, a, h->seq + op.id, h->ticket + op.id, h->d_err,
                                                            h->timeout_ns);
    count_launch();
    return SPARSH_OK;
}
void wait_args(sparsh_dist_s *h, const DistOp &op, WaitArgs &a) {
    Comm &m = comm();
    std::memset(&a, 0, sizeof a);
    a.nnbr = (int)op.recv_rank.size();
    for (int r = 0; r < a.nnbr; r++) {
        const int q = op.recv_rank[r];
        a.flag_local[r] = flag_slot(h->arena, m.nranks, op.id, 0, q);
        a.ack_dst[r] = flag_slot(h->peer_base[q], m.nranks, op.id, 1, m.rank);
    }
}
// consumer side, fused into the CSR kernel that reads the halo: wait for the flags at CTA start, ack from the last CTA
void halo_sync(sparsh_dist_s *h, const DistOp &op, HaloSync &hs) {
    WaitArgs a;
    wait_args(h, op, a);
    hs.nnbr = a.nnbr;
    for (int r = 0; r < a.nnbr; r++) {
        hs.flag_local[r] = a.flag_local[r];
        hs.ack_dst[r] = a.ack_dst[r];
    }
    hs.expect = h->expect + op.id;
    hs.ticket = h->ticket2 + op.id;
    hs.err = h->d_err;
    hs.halo_begin = op.ncol_local + op.shift;
    hs.timeout_ns = h->timeout_ns;
}

// ---- halo_mode 0: NCCL point-to-point on a communication stream -----------------------------------------------------
int nccl_start(const DistOp &op, double *x) {
    Context &c = ctx();
    Comm &m = comm();
    const int total = op.send_rank.empty() ? 0 : op.send_ptr.back();
    if (total > 0) {
        pack_kernel<<<(total + 255) / 256, 256, 0, c.stream>>>(x, op.d_send_idx, total, op.d_sendbuf);
        count_launch();
    }
    SP_CUDA(cudaEventRecord(m.ev_ready, c.stream));
    SP_CUDA(cudaStreamWaitEvent(m.comm_stream, m.ev_ready, 0));
    SP_NCCL(ncclGroupStart());
    for (size_t s = 0; s < op.send_rank.size(); s++)
        SP_NCCL(ncclSend(op.d_sendbuf + op.send_ptr[s], (size_t)(op.send_ptr[s + 1] - op.send_ptr[s]), ncclDouble,
                         op.send_rank[s], m.comm, m.comm_stream));
    for (size_t r = 0; r < op.recv_rank.size(); r++)
        SP_NCCL(ncclRecv(x + op.ncol_local + op.shift + op.recv_ptr[r], (size_t)(op.recv_ptr[r + 1] - op.recv_ptr[r]),
                         ncclDouble, op.recv_rank[r], m.comm, m.comm_stream));
    SP_NCCL(ncclGroupEnd());
    SP_CUDA(cudaEventRecord(m.ev_done, m.comm_stream));
    return SPARSH_OK;
}
int nccl_finish() {
    SP_CUDA(cudaStreamWaitEvent(ctx().stream, comm().ev_done, 0));
    return SPARSH_OK;
}

// the auxiliary stream carries the generic halo pushes and the boundary strips as a launch of their own beside the
// interior rows; joined by events
struct StreamSwap {
    cudaStream_t saved;
    explicit StreamSwap(cudaStream_t s) : saved(ctx().stream) { ctx().stream = s; }
    ~StreamSwap() { ctx().stream = saved; }
};
int fork_aux() {
    Comm &m = comm();
    SP_CUDA(cudaEventRecord(m.ev_ready, ctx().stream));
    SP_CUDA(cudaStreamWaitEvent(m.comm_stream, m.ev_ready, 0));
    return SPARSH_OK;
}
int join_aux() {
    Comm &m = comm();
    SP_CUDA(cudaEventRecord(m.ev_done, m.comm_stream));
    SP_CUDA(cudaStreamWaitEvent(ctx().stream, m.ev_done, 0));
    return SPARSH_OK;
}

// y = epi(op x).  The rows that touch the halo (and, for the fused Jacobi, the rows a neighbour needs) form the two
// boundary strips, everything else is interior.  Peer mode: a generic push first if the halo of x is not already on
// its way, then the strips — their CTAs wait for the flags, compute, optionally store the new values into the
// neighbours and signal as soon as the last of them is done — beside the interior rows, which never wait: as two
// launches on two streams, or, for the fused reductions (one grid over all rows), as one grid whose first CTAs are the
// strips.  `push_output`: y is the next input of this same operator.
int apply(sparsh_dist_s *h, const DistOp &op, int epi, double *x, double *y, EpiArgs args, bool push_output = false) {
    if (!op.needs_exchange()) return launch_csr(op.M, epi, x, y, args, 0, op.nrow);
    const bool reduces = epi == EPI_SPMV_DOT || epi == EPI_RESNORM;
    // tiny interiors are not worth a separate range (SPARSH_SPLIT_MIN_ROWS overrides the default)
    static const int split_min = [] {
        const char *e = getenv("SPARSH_SPLIT_MIN_ROWS");
        return e ? atoi(e) : 1024;
    }();
    const bool split = op.ie - op.ib >= split_min && (op.ib > 0 || op.ie < op.nrow);
    if (!h->peer) {
        // NCCL point-to-point: interior rows overlap the transfer as a separate launch (the fused reductions need one
        // grid over all rows and are not split)
        const bool split2 = split && !reduces;
        SP_TRY(nccl_start(op, x));
        if (split2) SP_TRY(launch_csr(op.M, epi, x, y, args, op.ib, op.ie));
        SP_TRY(nccl_finish());
        if (split2) return launch_csr2(op.M, epi, x, y, args, 0, op.ib, op.ie, op.nrow, nullptr);
        return launch_csr(op.M, epi, x, y, args, 0, op.nrow);
    }
    Comm &m = comm();
    const int bx = buffer_id(h, x);
    SP_REQUIRE(bx >= 0, "halo exchange on a vector that is not in the shared arena");
    const bool need_push = h->halo_ready[bx] != op.id + 1;
    h->halo_ready[bx] = 0;
    HaloSync hs;
    halo_sync(h, op, hs);
    if (push_output && epi == EPI_JACOBI && !op.send_rank.empty()) {  // the strips carry the fused push
        const int by = buffer_id(h, y);
        SP_REQUIRE(by >= 0 && h->buf_level[by] >= 0, "fused push into a vector outside the arena");
        args.pm_ptr = op.d_pm_ptr;
        args.pm_nbr = op.d_pm_nbr;
        args.pm_off = op.d_pm_off;
        args.pm_dst = h->d_pm_tab + (size_t)by * MAX_NBR;
        hs.nsend = (int)op.send_rank.size();
        for (int s = 0; s < hs.nsend; s++) {
            const int q = op.send_rank[s];
            hs.flag_dst[s] = flag_slot(h->peer_base[q], m.nranks, op.id, 0, m.rank);
            hs.ack_local[s] = flag_slot(h->arena, m.nranks, op.id, 1, q);
        }
        hs.seq = h->seq + op.id;
        h->halo_ready[by] = op.id + 1;
    }
    // Boundary strips (with the push in front of them) on the high-priority auxiliary stream, interior rows as a launch
    // of their own on the main stream.  Measured on B200, 256^3 (profiles/r02i_n2_*.json, r02j_*.json): 0.1009 s against
    // 0.1058 s for strips and interior rows as one grid at N=2, 0.0815 / 0.0827 at N=4, 0.0727 / 0.0723 at N=8 — the
    // fork/join costs nothing measurable inside a CUDA graph, the extra launch is hidden behind the interior rows, and
    // the neighbours hear from the strips earlier.
    if (split && !reduces) {
        EpiArgs iargs = args;  // interior rows: nothing to send
        iargs.pm_ptr = nullptr;
        SP_TRY(fork_aux());
        {
            StreamSwap sw(m.comm_stream);
            if (need_push) SP_TRY(peer_push(h, op, x));
            SP_TRY(launch_csr3(op.M, epi, x, y, args, 0, op.ib, op.ie, op.nrow, 0, 0, &hs));
        }
        SP_TRY(launch_csr(op.M, epi, x, y, iargs, op.ib, op.ie));
        return join_aux();
    }
    // one launch (fused reductions, unsplit operators): the generic push (if any) first — a consumer grid whose strip
    // CTAs fill the GPU while they wait must never be in front of the push that the neighbours' strips are waiting for
    // (that is a cross-GPU deadlock: measured at 512^3, where a strip has more CTAs than the GPU holds) — then strips +
    // interior rows as one grid
    if (need_push) SP_TRY(peer_push(h, op, x));
    if (!split) return launch_csr3(op.M, epi, x, y, args, 0, op.nrow, 0, 0, 0, 0, &hs);
    return launch_csr3(op.M, epi, x, y, args, 0, op.ib, op.ie, op.nrow, op.ib, op.ie, &hs);
}

PeerTab peer_tab(const sparsh_dist_s *h) {
    Comm &m = comm();
    PeerTab t;
    std::memset(&t, 0, sizeof t);
    t.nranks = m.nranks;
    t.rank = m.rank;
    for (int r = 0; r < m.nranks; r++) t.base[r] = h->peer_base[r];
    return t;
}

// in-place sum over the ranks of `count` (<= 3) device scalars
int allreduce_sum(sparsh_dist_s *h, double *d_vals, int count) {
    Comm &m = comm();
    if (m.nranks == 1) return SPARSH_OK;
    if (h->peer) {
        SP_REQUIRE(count >= 1 && count < RED_SLOTS, "peer all-reduce handles up to 3 scalars");
        peer_allreduce_kernel<<<1, 32, 0, ctx().stream>>>(d_vals, count, peer_tab(h), h->coll_off, h->red_seq, h->d_err, h->timeout_ns);
        count_launch();
        SP_CUDA(cudaGetLastError());
        return SPARSH_OK;
    }
    SP_NCCL(ncclAllReduce(d_vals, d_vals, (size_t)count, ncclDouble, ncclSum, m.comm, ctx().stream));
    return SPARSH_OK;
}

// `feeds_A`: the vector this smoothing step leaves behind is next read by A_l itself (residual after pre-smoothing)
int dist_smooth(sparsh_dist_s *h, DistLevel &L, const double *b, double *&cur, double *&other, int sweeps, bool zero,
                bool feeds_A) {
    if (sweeps == 0) {
        if (zero) SP_TRY(k_fill(cur, (size_t)L.n, 0.0));
        return SPARSH_OK;
    }
    for (int s = 0; s < sweeps; s++) {
        if (s == 0 && zero) {
            SP_TRY(k_jacobi_zero((size_t)L.n, b, L.A.M->diag, h->prm.omega, other));
        } else {
            EpiArgs a;
            a.b = b;
            a.xi = cur;
            a.d = L.A.M->diag;
            a.omega = h->prm.omega;
            SP_TRY(apply(h, L.A, EPI_JACOBI, cur, other, a, s + 1 < sweeps || feeds_A));
        }
        std::swap(cur, other);
    }
    return SPARSH_OK;
}

// x must be a halo-capable arena vector of level 0.  One V-cycle, enqueue only.
int enqueue_dist_vcycle(sparsh_dist_s *h, const double *b, double *x, bool x_is_zero) {
    Context &c = ctx();
    Comm &m = comm();
    const int nd = (int)h->lev.size();
    std::vector<double *> X(nd + 1), T(nd);
    std::vector<const double *> B(nd + 1);
    for (int l = 0; l < nd; l++) {
        X[l] = l == 0 ? x : h->lev[l].xbuf;
        T[l] = h->lev[l].tbuf;
        B[l] = l == 0 ? b : h->lev[l].bbuf;
    }
    X[nd] = h->xtail_local;
    B[nd] = h->btail_local;
    for (int l = 0; l < nd; l++) {
        DistLevel &L = h->lev[l];
        SP_TRY(dist_smooth(h, L, B[l], X[l], T[l], h->prm.pre_sweeps, l > 0 || x_is_zero, true));
        EpiArgs a;
        a.b = B[l];
        SP_TRY(apply(h, L.A, EPI_RESID, X[l], L.rbuf, a));
        double *bnext = l + 1 < nd ? h->lev[l + 1].bbuf : h->btail_local;
        SP_TRY(apply(h, L.R, EPI_SPMV, L.rbuf, bnext, EpiArgs()));
    }
    // replicated tail: every rank contributes its part of the restricted right-hand side to all copies of the vector,
    // the levels below are solved redundantly, the owned rows of the correction are kept
    const int gblocks = std::max(1, std::min((h->n_own_tail0 + 255) / 256, 4 * c.sm_count));
    if (m.nranks > 1 && h->peer) {
        tail_exchange_kernel<<<gblocks, 256, 0, c.stream>>>(h->btail_local, h->d_tail_rows, h->n_own_tail0, peer_tab(h), h->tailb_off,
                                                            h->coll_off, h->tail_seq, h->tail_ticket, h->d_err, h->timeout_ns);
        count_launch();
    } else if (m.nranks > 1) {
        SP_CUDA(cudaMemcpyAsync(h->tail_send, h->btail_local, sizeof(double) * (size_t)h->n_own_tail0, cudaMemcpyDeviceToDevice, c.stream));
        SP_NCCL(ncclAllGather(h->tail_send, h->tail_recv, (size_t)h->tail_maxc, ncclDouble, m.comm, c.stream));
        const int tot = h->tail_maxc * m.nranks;
        scatter_map_kernel<<<(tot + 255) / 256, 256, 0, c.stream>>>(h->tail_recv, h->d_tail_map, tot, h->tail_b);
        count_launch();
    } else {
        const int tot = h->n_own_tail0;
        scatter_map_kernel<<<(tot + 255) / 256, 256, 0, c.stream>>>(h->btail_local, h->d_tail_map, tot, h->tail_b);
        count_launch();
    }
    SP_TRY(enqueue_vcycle(h->tail, h->tail_b, h->tail_x, true));
    if (m.nranks > 1 && h->peer) {
        tail_gather_ack_kernel<<<gblocks, 256, 0, c.stream>>>(h->tail_x, h->d_tail_rows, h->n_own_tail0, h->xtail_local, peer_tab(h),
                                                              h->coll_off, h->tail_seq);
        count_launch();
    } else if (h->n_own_tail0 > 0) {
        gather_rows_kernel<<<(h->n_own_tail0 + 255) / 256, 256, 0, c.stream>>>(h->tail_x, h->d_tail_rows, h->n_own_tail0, h->xtail_local);
        count_launch();
    }
    for (int l = nd; l > 0; l--) {
        DistLevel &F = h->lev[l - 1];
        SP_TRY(apply(h, F.P, EPI_PROLONG, X[l], X[l - 1], EpiArgs()));
        SP_TRY(dist_smooth(h, F, B[l - 1], X[l - 1], T[l - 1], h->prm.post_sweeps, false, false));
    }
    if (X[0] != x) SP_CUDA(cudaMemcpyAsync(x, X[0], sizeof(double) * (size_t)h->lev[0].n, cudaMemcpyDeviceToDevice, c.stream));
    SP_CUDA(cudaGetLastError());
    return SPARSH_OK;
}

template <class F>
int dist_run_graphed(sparsh_dist_s *h, const void *k0, const void *k1, int tag, F body) {
    // peer-push exchanges are plain kernels; NCCL collectives (and point-to-point calls in halo_mode 0) are capturable
    Context &c = ctx();
    if (!h->prm.use_graph) return body();
    GraphEntry *ent = nullptr;
    for (auto &g : h->graphs)
        if (g.k0 == k0 && g.k1 == k1 && g.tag == tag) ent = &g;
    if (!ent) {
        GraphEntry g;
        g.k0 = k0;
        g.k1 = k1;
        g.tag = tag;
        h->graphs.push_back(g);
        return body();
    }
    if (!ent->exec) {
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

int check_handshake(sparsh_dist_s *h) {
    if (!h->peer) return SPARSH_OK;
    SP_CUDA(cudaMemcpyAsync(h->h_err, h->d_err, sizeof(int), cudaMemcpyDeviceToHost, ctx().stream));
    SP_CUDA(cudaStreamSynchronize(ctx().stream));
    if (*h->h_err) {
        h->dead = true;
        set_error("multi-GPU halo handshake timed out (a neighbour never signalled); the distributed handle is unusable");
        return SPARSH_ERR_CUDA;
    }
    return SPARSH_OK;
}
// after a timed-out handshake the sequence counters of the ranks are out of step for good: refuse further work
int check_alive(const sparsh_dist_s *h) {
    SP_REQUIRE(h != nullptr, "hierarchy is NULL");
    SP_REQUIRE(!h->dead, "distributed handle is unusable after a halo-handshake timeout: destroy it and create a new one");
    return SPARSH_OK;
}

// all ranks exchange equally sized byte blocks (setup only)
int allgather_bytes_dev(const void *mine, size_t bytes, std::vector<char> &all, char *d_in, char *d_out) {
    Comm &m = comm();
    SP_CUDA(cudaMemcpy(d_in, mine, bytes, cudaMemcpyHostToDevice));
    SP_NCCL(ncclAllGather(d_in, d_out, bytes, ncclChar, m.comm, ctx().stream));
    SP_CUDA(cudaStreamSynchronize(ctx().stream));
    SP_CUDA(cudaMemcpy(all.data(), d_out, all.size(), cudaMemcpyDeviceToHost));
    return SPARSH_OK;
}
int allgather_bytes(const void *mine, size_t bytes, std::vector<char> &all) {
    Comm &m = comm();
    all.assign(bytes * (size_t)m.nranks, 0);
    if (m.nranks == 1) {
        std::memcpy(all.data(), mine, bytes);
        return SPARSH_OK;
    }
    char *d_in = nullptr, *d_out = nullptr;
    int rc = SPARSH_OK;
    if (cudaMalloc(&d_in, bytes) != cudaSuccess || cudaMalloc(&d_out, bytes * (size_t)m.nranks) != cudaSuccess) {
        set_error("out of device memory in the setup all-gather");
        cudaGetLastError();
        rc = SPARSH_ERR_CUDA;
    } else {
        rc = allgather_bytes_dev(mine, bytes, all, d_in, d_out);
    }
    cudaFree(d_in);
    cudaFree(d_out);
    return rc;
}

// the auxiliary stream runs the boundary strips (which feed the neighbours): highest priority, so their CTAs are
// scheduled ahead of the interior rows that share the GPU with them
int ensure_aux_stream(Comm &m) {
    if (m.comm_stream) return SPARSH_OK;
    int lo = 0, hi = 0;
    SP_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    SP_CUDA(cudaStreamCreateWithPriority(&m.comm_stream, cudaStreamNonBlocking, hi));
    SP_CUDA(cudaEventCreateWithFlags(&m.ev_ready, cudaEventDisableTiming));
    SP_CUDA(cudaEventCreateWithFlags(&m.ev_done, cudaEventDisableTiming));
    return SPARSH_OK;
}

}  // namespace

extern "C" {

int sparsh_dist_get_unique_id(char *id128) {
    static_assert(sizeof(ncclUniqueId) <= SPARSH_NCCL_ID_BYTES, "ncclUniqueId larger than the ABI slot");
    ncclUniqueId id;
    SP_NCCL(ncclGetUniqueId(&id));
    std::memset(id128, 0, SPARSH_NCCL_ID_BYTES);
    std::memcpy(id128, &id, sizeof id);
    return SPARSH_OK;
}

int sparsh_dist_init(const char *id128, int nranks, int rank) {
    SP_TRY(ensure_init());
    Comm &m = comm();
    if (m.comm) return SPARSH_OK;
    SP_REQUIRE(nranks >= 1 && rank >= 0 && rank < nranks, "bad rank / world size");
    ncclUniqueId id;
    std::memcpy(&id, id128, sizeof id);
    SP_NCCL(ncclCommInitRank(&m.comm, nranks, id, rank));
    m.nranks = nranks;
    m.rank = rank;
    return ensure_aux_stream(m);
}

int sparsh_dist_finalize(void) {
    Comm &m = comm();
    if (!m.comm) return SPARSH_OK;
    cudaStreamSynchronize(ctx().stream);
    cudaStreamSynchronize(m.comm_stream);
    ncclCommDestroy(m.comm);
    cudaStreamDestroy(m.comm_stream);
    cudaEventDestroy(m.ev_ready);
    cudaEventDestroy(m.ev_done);
    m = Comm();
    return SPARSH_OK;
}

int sparsh_dist_info(int *nranks, int *rank) {
    if (nranks) *nranks = comm().nranks;
    if (rank) *rank = comm().rank;
    return SPARSH_OK;
}

static int build_dist_hierarchy(sparsh_dist_s *h, int nd, const sparsh_dist_level_desc *lev, int ntail,
                                const sparsh_level_desc *tail, const int *tail_counts, const int *tail_rows,
                                const sparsh_params *params);

int sparsh_dist_hierarchy_create(int nd, const sparsh_dist_level_desc *lev, int ntail, const sparsh_level_desc *tail,
                                 const int *tail_counts, const int *tail_rows, const sparsh_params *params,
                                 sparsh_dist_t *out) {
    SP_TRY(ensure_init());
    SP_REQUIRE(nd >= 1 && ntail >= 1 && lev && tail && tail_counts && tail_rows && out, "bad distributed hierarchy description");
    sparsh_dist_s *h = new sparsh_dist_s();
    const int rc = build_dist_hierarchy(h, nd, lev, ntail, tail, tail_counts, tail_rows, params);
    if (rc != SPARSH_OK) {
        const std::string msg = sparsh_last_error();  // keep the first error: the teardown may overwrite it
        sparsh_dist_hierarchy_destroy(h);
        set_error(msg);
        return rc;
    }
    *out = h;
    return SPARSH_OK;
}

static int build_dist_hierarchy(sparsh_dist_s *h, int nd, const sparsh_dist_level_desc *lev, int ntail,
                                const sparsh_level_desc *tail, const int *tail_counts, const int *tail_rows,
                                const sparsh_params *params) {
    Comm &m = comm();
    SP_REQUIRE(m.comm != nullptr || m.nranks == 1, "sparsh_dist_init has not been called");
    NvtxRange nvtx("sparsh:dist-upload");
    SP_TRY(ensure_aux_stream(m));  // single-rank use without NCCL (tests) still needs the stream/event plumbing
    if (params)
        h->prm = *params;
    else
        sparsh_params_default(&h->prm);
    SP_REQUIRE(h->prm.smoother == 0, "the distributed path implements the Jacobi smoother only");
    h->peer = h->prm.halo_mode == 1 && m.nranks > 1 && m.nranks <= MAX_NBR;
    h->nops = 3 * nd;
    h->lev.resize(nd);
    if (const char *e = getenv("SPARSH_HALO_TIMEOUT_MS")) h->timeout_ns = std::max(1ll, atoll(e)) * 1000000ll;

    // ---- operators.  Vector space of level l is read by A_l (halo segment right after the owned entries) and by
    //      P_{l-1} (its halo segment sits behind A_l's, so the two exchanges never share memory)
    //      Every halo segment starts on a 128-byte boundary (align16 doubles).
    for (int l = 0; l < nd; l++) {
        DistLevel &L = h->lev[l];
        SP_TRY(make_op(lev[l].A, align16(lev[l].A.ncol_local), 3 * l + 0, L.A));
        SP_TRY(make_push_map(lev[l].A, L.A));
        // P_l gathers from the level l+1 vector: behind A_{l+1}'s halo segment there (the replicated tail has none)
        const int pstart = l + 1 < nd ? align16(align16(lev[l + 1].A.ncol_local) + lev[l + 1].A.nhalo) : align16(lev[l].P.ncol_local);
        SP_TRY(make_op(lev[l].P, pstart, 3 * l + 1, L.P));
        SP_TRY(make_op(lev[l].R, align16(lev[l].R.ncol_local), 3 * l + 2, L.R));
        L.n = lev[l].A.nrow;
        L.n_next = lev[l].R.nrow;
        const int astart = align16(L.n);
        L.xcap = (size_t)(l > 0 ? align16(astart + lev[l].A.nhalo) + lev[l - 1].P.nhalo : astart + lev[l].A.nhalo) + 2;
    }
    h->n_own_tail0 = tail_counts[m.rank];
    SP_REQUIRE(h->n_own_tail0 == h->lev[nd - 1].n_next, "owned rows of the first replicated level disagree with R");

    // ---- arena: flags first, then every vector that can be the target of a halo exchange (same ORDER on all ranks)
    //      [op flags | collective area | replicated right-hand side] sit at the SAME offsets on every rank; the vectors
    //      behind them have rank-dependent sizes, their offsets are exchanged below
    const size_t flag_bytes = align_up(sizeof(u64) * 2 * (size_t)h->nops * m.nranks, 256);
    h->coll_off = flag_bytes;
    h->tailb_off = h->coll_off + align_up(sizeof(CollArea), 256);
    h->n_tail0 = tail[0].nrow;
    const size_t fixed_bytes = h->tailb_off + align_up(sizeof(double) * ((size_t)h->n_tail0 + 2), 256);
    std::vector<size_t> want;  // bytes per buffer, in buffer-id order
    for (int l = 0; l < nd; l++) {
        want.push_back(sizeof(double) * h->lev[l].xcap);                                         // tbuf
        want.push_back(sizeof(double) * ((size_t)align16(h->lev[l].n) + lev[l].R.nhalo + 2));    // rbuf
        if (l > 0) want.push_back(sizeof(double) * h->lev[l].xcap);                              // xbuf
    }
    want.push_back(sizeof(double) * ((size_t)align16(h->n_own_tail0) + lev[nd - 1].P.nhalo + 2));  // xtail_local
    for (int i = 0; i < 5; i++) want.push_back(sizeof(double) * h->lev[0].xcap);                   // Krylov vectors
    size_t total = fixed_bytes;
    std::vector<size_t> off(want.size());
    for (size_t i = 0; i < want.size(); i++) {
        off[i] = total;
        total += align_up(want[i], 256);
    }
    h->arena_bytes = total;
    SP_CUDA(cudaMalloc(&h->arena, total));
    SP_CUDA(cudaMemset(h->arena, 0, total));
    size_t k = 0;
    auto take = [&](int level) {
        double *p = reinterpret_cast<double *>(h->arena + off[k]);
        h->bufs.emplace_back(p, off[k]);
        h->buf_level.push_back(level);
        k++;
        return p;
    };
    for (int l = 0; l < nd; l++) {
        h->lev[l].tbuf = take(l);
        h->lev[l].rbuf = take(-1);
        if (l > 0) h->lev[l].xbuf = take(l);
    }
    h->xtail_local = take(-1);
    for (int i = 0; i < 5; i++) h->kv[i] = take(0);
    h->tail_b = reinterpret_cast<double *>(h->arena + h->tailb_off);
    h->halo_ready.assign(h->bufs.size(), 0);
    for (int l = 1; l < nd; l++) SP_CUDA(cudaMalloc(&h->lev[l].bbuf, sizeof(double) * ((size_t)h->lev[l].n + 2)));

    SP_CUDA(cudaMalloc(&h->seq, sizeof(u64) * (size_t)h->nops));
    SP_CUDA(cudaMalloc(&h->expect, sizeof(u64) * (size_t)h->nops));
    SP_CUDA(cudaMalloc(&h->ticket, sizeof(unsigned int) * (size_t)h->nops));
    SP_CUDA(cudaMalloc(&h->ticket2, sizeof(unsigned int) * (size_t)h->nops));
    SP_CUDA(cudaMemset(h->ticket2, 0, sizeof(unsigned int) * (size_t)h->nops));
    SP_CUDA(cudaMalloc(&h->red_seq, sizeof(u64)));
    SP_CUDA(cudaMalloc(&h->tail_seq, sizeof(u64)));
    SP_CUDA(cudaMalloc(&h->tail_ticket, sizeof(unsigned int)));
    SP_CUDA(cudaMemset(h->red_seq, 0, sizeof(u64)));
    SP_CUDA(cudaMemset(h->tail_seq, 0, sizeof(u64)));
    SP_CUDA(cudaMemset(h->tail_ticket, 0, sizeof(unsigned int)));
    SP_CUDA(cudaMalloc(&h->d_err, sizeof(int)));
    SP_CUDA(cudaMallocHost(&h->h_err, sizeof(int)));
    SP_CUDA(cudaMemset(h->seq, 0, sizeof(u64) * (size_t)h->nops));
    SP_CUDA(cudaMemset(h->expect, 0, sizeof(u64) * (size_t)h->nops));
    SP_CUDA(cudaMemset(h->ticket, 0, sizeof(unsigned int) * (size_t)h->nops));
    SP_CUDA(cudaMemset(h->d_err, 0, sizeof(int)));
    *h->h_err = 0;

    // ---- peer mapping + the two small tables every producer needs about its consumers
    h->peer_base.assign(m.nranks, nullptr);
    h->peer_base[m.rank] = h->arena;
    if (h->peer) {
        cudaIpcMemHandle_t mine;
        SP_CUDA(cudaIpcGetMemHandle(&mine, h->arena));
        std::vector<char> all;
        SP_TRY(allgather_bytes(&mine, sizeof mine, all));
        bool ok = true;
        for (int r = 0; r < m.nranks && ok; r++) {
            if (r == m.rank) continue;
            cudaIpcMemHandle_t hd;
            std::memcpy(&hd, all.data() + (size_t)r * sizeof hd, sizeof hd);
            void *p = nullptr;
            if (cudaIpcOpenMemHandle(&p, hd, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
                cudaGetLastError();
                ok = false;
            }
            h->peer_base[r] = (char *)p;
        }
        // every rank must take the same decision
        int okv = ok ? 1 : 0;
        std::vector<char> oks;
        SP_TRY(allgather_bytes(&okv, sizeof okv, oks));
        for (int r = 0; r < m.nranks; r++) {
            int v;
            std::memcpy(&v, oks.data() + (size_t)r * sizeof v, sizeof v);
            if (!v) h->peer = false;
        }
    }
    {
        // buffer offsets of every rank
        std::vector<long long> mine(h->bufs.size());
        for (size_t i = 0; i < h->bufs.size(); i++) mine[i] = (long long)h->bufs[i].second;
        std::vector<char> all;
        SP_TRY(allgather_bytes(mine.data(), sizeof(long long) * mine.size(), all));
        h->peer_buf_off.assign(m.nranks, std::vector<long long>(mine.size()));
        for (int r = 0; r < m.nranks; r++)
            std::memcpy(h->peer_buf_off[r].data(), all.data() + (size_t)r * sizeof(long long) * mine.size(),
                        sizeof(long long) * mine.size());
        // where each sender's slice lands inside MY input vectors: table[op][sender] = element offset, -1 = none
        std::vector<long long> land((size_t)h->nops * m.nranks, -1);
        auto fill = [&](const DistOp &op) {
            for (size_t r = 0; r < op.recv_rank.size(); r++)
                land[(size_t)op.id * m.nranks + op.recv_rank[r]] = (long long)op.ncol_local + op.shift + op.recv_ptr[r];
        };
        for (auto &L : h->lev) {
            fill(L.A);
            fill(L.P);
            fill(L.R);
        }
        SP_TRY(allgather_bytes(land.data(), sizeof(long long) * land.size(), all));
        auto resolve = [&](DistOp &op) -> int {
            op.peer_dst_off.resize(op.send_rank.size());
            for (size_t s = 0; s < op.send_rank.size(); s++) {
                const int q = op.send_rank[s];
                long long v;
                std::memcpy(&v, all.data() + ((size_t)q * land.size() + (size_t)op.id * m.nranks + m.rank) * sizeof(long long),
                            sizeof v);
                SP_REQUIRE(v >= 0, "exchange plans of two ranks disagree");
                op.peer_dst_off[s] = v;
            }
            SP_REQUIRE((int)op.send_rank.size() <= MAX_NBR && (int)op.recv_rank.size() <= MAX_NBR, "too many neighbours");
            return SPARSH_OK;
        };
        for (auto &L : h->lev) {
            SP_TRY(resolve(L.A));
            SP_TRY(resolve(L.P));
            SP_TRY(resolve(L.R));
        }
        // fused Jacobi push: where my slice of A_l's exchange lands when the OUTPUT vector is buffer `bid`
        std::vector<double *> tab(h->bufs.size() * MAX_NBR, nullptr);
        for (size_t bid = 0; bid < h->bufs.size(); bid++) {
            if (h->buf_level[bid] < 0 || !h->peer) continue;
            const DistOp &A = h->lev[h->buf_level[bid]].A;
            for (size_t sidx = 0; sidx < A.send_rank.size(); sidx++) {
                const int q = A.send_rank[sidx];
                tab[bid * MAX_NBR + sidx] =
                    reinterpret_cast<double *>(h->peer_base[q] + h->peer_buf_off[q][bid]) + A.peer_dst_off[sidx];
            }
        }
        SP_CUDA(cudaMalloc(&h->d_pm_tab, sizeof(double *) * tab.size()));
        SP_CUDA(cudaMemcpy(h->d_pm_tab, tab.data(), sizeof(double *) * tab.size(), cudaMemcpyHostToDevice));
    }

    // ---- replicated tail
    sparsh_params tp = h->prm;
    tp.use_graph = 0;  // its launches are captured as part of the enclosing distributed graph
    SP_TRY(sparsh_hierarchy_create(ntail, tail, &tp, &h->tail));
    int maxc = 0, displ = 0, my_displ = 0;
    for (int r = 0; r < m.nranks; r++) {
        maxc = std::max(maxc, tail_counts[r]);
        if (r == m.rank) my_displ = displ;
        displ += tail_counts[r];
    }
    SP_REQUIRE(displ == h->n_tail0, "tail_counts do not add up to the rows of the first replicated level");
    h->tail_maxc = std::max(maxc, 1);
    std::vector<int> map((size_t)h->tail_maxc * m.nranks, -1);
    displ = 0;
    for (int r = 0; r < m.nranks; r++) {
        for (int q = 0; q < tail_counts[r]; q++) map[(size_t)r * h->tail_maxc + q] = tail_rows[displ + q];
        displ += tail_counts[r];
    }
    if (m.nranks == 1) map.assign(tail_rows, tail_rows + h->n_tail0);
    SP_CUDA(cudaMalloc(&h->d_tail_map, sizeof(int) * map.size()));
    SP_CUDA(cudaMemcpy(h->d_tail_map, map.data(), sizeof(int) * map.size(), cudaMemcpyHostToDevice));
    SP_CUDA(cudaMalloc(&h->d_tail_rows, sizeof(int) * (size_t)std::max(h->n_own_tail0, 1)));
    SP_CUDA(cudaMemcpy(h->d_tail_rows, tail_rows + my_displ, sizeof(int) * (size_t)h->n_own_tail0, cudaMemcpyHostToDevice));
    SP_CUDA(cudaMalloc(&h->tail_send, sizeof(double) * (size_t)h->tail_maxc));
    SP_CUDA(cudaMemset(h->tail_send, 0, sizeof(double) * (size_t)h->tail_maxc));
    SP_CUDA(cudaMalloc(&h->tail_recv, sizeof(double) * (size_t)h->tail_maxc * m.nranks));
    SP_CUDA(cudaMalloc(&h->tail_x, sizeof(double) * ((size_t)h->n_tail0 + 2)));
    SP_CUDA(cudaMalloc(&h->btail_local, sizeof(double) * ((size_t)h->n_own_tail0 + 2)));
    SP_CUDA(cudaMalloc(&h->d_sc, sizeof(double) * 16));
    SP_CUDA(cudaMallocHost(&h->h_sc, sizeof(double) * 16));
    SP_CUDA(cudaDeviceSynchronize());
    if (m.nranks > 1) {  // nobody may push before every arena is mapped and zeroed
        SP_NCCL(ncclAllReduce(h->d_sc, h->d_sc, 1, ncclDouble, ncclSum, m.comm, ctx().stream));
        SP_CUDA(cudaStreamSynchronize(ctx().stream));
    }
    return SPARSH_OK;
}

int sparsh_dist_hierarchy_destroy(sparsh_dist_t h) {
    if (!h) return SPARSH_OK;
    Comm &m = comm();
    if (ctx().ready) cudaStreamSynchronize(ctx().stream);
    for (auto &g : h->graphs)
        if (g.exec) cudaGraphExecDestroy(g.exec);
    for (auto &L : h->lev) {
        free_op(L.A);
        free_op(L.P);
        free_op(L.R);
        cudaFree(L.bbuf);
    }
    sparsh_hierarchy_destroy(h->tail);
    for (int r = 0; r < (int)h->peer_base.size(); r++)
        if (r != m.rank && h->peer_base[r]) cudaIpcCloseMemHandle(h->peer_base[r]);
    cudaFree(h->arena);
    cudaFree(h->tail_send);
    cudaFree(h->tail_recv);
    cudaFree(h->tail_x);
    cudaFree(h->d_tail_map);
    cudaFree(h->d_tail_rows);
    cudaFree(h->btail_local);
    cudaFree(h->seq);
    cudaFree(h->expect);
    cudaFree(h->ticket);
    cudaFree(h->ticket2);
    cudaFree(h->d_pm_tab);
    for (int i = 0; i < 7; i++) cudaFree(h->bv[i]);
    cudaFree(h->red_seq);
    cudaFree(h->tail_seq);
    cudaFree(h->tail_ticket);
    cudaFree(h->d_err);
    cudaFreeHost(h->h_err);
    cudaFree(h->d_sc);
    cudaFreeHost(h->h_sc);
    delete h;
    return SPARSH_OK;
}

int sparsh_dist_local_rows(sparsh_dist_t h, int level, int *nrow) {
    SP_REQUIRE(h != nullptr && level >= 0 && level <= (int)h->lev.size(), "bad level");
    *nrow = level < (int)h->lev.size() ? h->lev[level].n : h->n_own_tail0;
    return SPARSH_OK;
}

int sparsh_dist_level_matrix(sparsh_dist_t h, int level, sparsh_matrix_t *A) {
    SP_REQUIRE(h != nullptr && level >= 0 && level < (int)h->lev.size() && A, "bad level");
    *A = h->lev[level].A.M;
    return SPARSH_OK;
}

int sparsh_dist_spmv(sparsh_dist_t h, int level, const double *d_x_local, double *d_y_local) {
    SP_TRY(check_alive(h));
    SP_REQUIRE(level >= 0 && level < (int)h->lev.size(), "bad level");
    DistLevel &L = h->lev[level];
    SP_CUDA(cudaMemcpyAsync(L.tbuf, d_x_local, sizeof(double) * (size_t)L.n, cudaMemcpyDeviceToDevice, ctx().stream));
    SP_TRY(apply(h, L.A, EPI_SPMV, L.tbuf, d_y_local, EpiArgs()));
    return check_handshake(h);
}

int sparsh_dist_vcycle(sparsh_dist_t h, const double *d_b_local, double *d_x_local, int cycles, int x_is_zero) {
    SP_TRY(check_alive(h));
    SP_REQUIRE(cycles >= 0, "bad arguments");
    DistLevel &L0 = h->lev[0];
    double *z = h->kv[1];  // halo-capable staging for the caller's x
    SP_CUDA(cudaMemcpyAsync(z, d_x_local, sizeof(double) * (size_t)L0.n, cudaMemcpyDeviceToDevice, ctx().stream));
    for (int k = 0; k < cycles; k++) SP_TRY(enqueue_dist_vcycle(h, d_b_local, z, x_is_zero && k == 0));
    SP_CUDA(cudaMemcpyAsync(d_x_local, z, sizeof(double) * (size_t)L0.n, cudaMemcpyDeviceToDevice, ctx().stream));
    return check_handshake(h);
}

// Same arithmetic as cg_impl(precond = true) in krylov.cu (reference src/AMG_main_solvers.cpp:107-167); the three
// reductions of an iteration are completed by in-place all-reduces of device scalars.
int sparsh_dist_pcg(sparsh_dist_t h, const double *b, double *x, double tol, int max_iter, double *hist, int *iters_out) {
    SP_TRY(check_alive(h));
    NvtxRange nvtx("sparsh:dist-pcg");
    Context &c = ctx();
    DistLevel &L0 = h->lev[0];
    const size_t n = (size_t)L0.n;
    double *r = h->kv[0], *z = h->kv[1], *p = h->kv[2], *Ap = h->kv[3], *xs = h->kv[4];
    double *sc = h->d_sc;
    enum { S_PAP = 0, S_RZ = 1, S_RZNEW = 2, S_RR = 3 };
    auto read_rr = [&]() -> int {
        SP_CUDA(cudaMemcpyAsync(h->h_sc + S_RR, sc + S_RR, sizeof(double), cudaMemcpyDeviceToHost, c.stream));
        if (h->peer) SP_CUDA(cudaMemcpyAsync(h->h_err, h->d_err, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
        return SPARSH_OK;
    };
    SP_CUDA(cudaMemcpyAsync(xs, x, sizeof(double) * n, cudaMemcpyDeviceToDevice, c.stream));
    EpiArgs a;
    a.b = b;
    SP_TRY(apply(h, L0.A, EPI_RESID, xs, r, a));
    SP_TRY(k_dot(n, r, r, sc + S_RR));
    SP_TRY(allreduce_sum(h, sc + S_RR, 1));
    SP_TRY(dist_run_graphed(h, r, z, 1, [&]() { return enqueue_dist_vcycle(h, r, z, true); }));
    SP_CUDA(cudaMemcpyAsync(p, z, sizeof(double) * n, cudaMemcpyDeviceToDevice, c.stream));
    SP_TRY(k_dot(n, r, z, sc + S_RZ));
    SP_TRY(allreduce_sum(h, sc + S_RZ, 1));
    SP_TRY(read_rr());
    SP_CUDA(cudaStreamSynchronize(c.stream));
    double r1 = std::sqrt(h->h_sc[S_RR]);
    if (hist) hist[0] = r1;

    auto body = [&]() -> int {
        // Ap = A p and the local part of p.Ap (the fused reduction runs over the full row range: no interior split)
        EpiArgs e;
        e.xi = p;
        e.red_out = sc + S_PAP;
        SP_TRY(apply(h, L0.A, EPI_SPMV_DOT, p, Ap, e));
        SP_TRY(allreduce_sum(h, sc + S_PAP, 1));
        SP_TRY(k_pcg_update_xr(n, p, Ap, xs, r, sc + S_RZ, sc + S_PAP, sc + S_RR));
        SP_TRY(enqueue_dist_vcycle(h, r, z, true));
        SP_TRY(k_dot(n, z, r, sc + S_RZNEW));
        // z.r and the ||r||^2 partial left behind by the x/r update travel together (slots S_RZNEW, S_RR are adjacent)
        SP_TRY(allreduce_sum(h, sc + S_RZNEW, 2));
        SP_TRY(k_pcg_update_p(n, z, p, sc + S_RZNEW, sc + S_RZ));
        SP_TRY(k_scalar_copy(sc + S_RZ, sc + S_RZNEW));
        SP_TRY(read_rr());
        return SPARSH_OK;
    };
    int count = 0, rc = SPARSH_OK;
    while (count < max_iter && r1 > tol) {
        count++;
        SP_TRY(dist_run_graphed(h, x, b, 10, body));
        SP_CUDA(cudaStreamSynchronize(c.stream));
        if (h->peer && *h->h_err) {  // the flag rides on the all-reduces: every rank sees it in the same iteration
            h->dead = true;
            set_error("multi-GPU halo handshake timed out (a neighbour never signalled); the distributed handle is unusable");
            rc = SPARSH_ERR_CUDA;
            break;
        }
        r1 = std::sqrt(h->h_sc[S_RR]);
        if (hist) hist[count] = r1;
        if (!std::isfinite(r1)) break;
    }
    SP_CUDA(cudaMemcpyAsync(x, xs, sizeof(double) * n, cudaMemcpyDeviceToDevice, c.stream));
    SP_CUDA(cudaStreamSynchronize(c.stream));
    if (iters_out) *iters_out = count;
    if (rc != SPARSH_OK) return rc;
    return r1 <= tol ? SPARSH_OK : SPARSH_ERR_NOT_CONVERGED;
}

// Assemble a row-distributed host vector on every rank: full[rows[i]] = local[i] for the rows of all ranks (setup /
// result collection for the reference-style entry points whose callers hold global b and x; not on the solve path).
int sparsh_dist_allgather_rows(const double *h_local, const int *h_rows, int n_local, double *h_full, int n_full) {
    SP_TRY(ensure_init());
    Comm &m = comm();
    SP_REQUIRE(n_local >= 0 && n_full >= 0 && (n_local == 0 || (h_local && h_rows)) && h_full, "bad arguments");
    if (m.nranks == 1) {
        for (int i = 0; i < n_local; i++) h_full[h_rows[i]] = h_local[i];
        return SPARSH_OK;
    }
    SP_REQUIRE(m.comm != nullptr, "sparsh_dist_init has not been called");
    std::vector<char> all;
    SP_TRY(allgather_bytes(&n_local, sizeof n_local, all));
    int maxc = 1;
    std::vector<int> counts((size_t)m.nranks);
    for (int r = 0; r < m.nranks; r++) {
        std::memcpy(&counts[r], all.data() + (size_t)r * sizeof(int), sizeof(int));
        maxc = std::max(maxc, counts[r]);
    }
    std::vector<double> vpad((size_t)maxc, 0.0);
    std::vector<int> rpad((size_t)maxc, -1);
    std::copy(h_local, h_local + n_local, vpad.begin());
    std::copy(h_rows, h_rows + n_local, rpad.begin());
    std::vector<char> vall, rall;
    SP_TRY(allgather_bytes(vpad.data(), sizeof(double) * (size_t)maxc, vall));
    SP_TRY(allgather_bytes(rpad.data(), sizeof(int) * (size_t)maxc, rall));
    for (int r = 0; r < m.nranks; r++) {
        const double *v = reinterpret_cast<const double *>(vall.data() + (size_t)r * sizeof(double) * (size_t)maxc);
        const int *ri = reinterpret_cast<const int *>(rall.data() + (size_t)r * sizeof(int) * (size_t)maxc);
        for (int i = 0; i < counts[r]; i++) {
            SP_REQUIRE(ri[i] >= 0 && ri[i] < n_full, "row id out of range in the gathered vector");
            h_full[ri[i]] = v[i];
        }
    }
    return SPARSH_OK;
}

// AMG as a solver on the row-partitioned hierarchy: V-cycles until ||A x - b||_2 <= tol (absolute, as the reference:
// AMG_solver::AMG_solve_jacobi(b,x,-1), src/AMG_phases.cpp:194-226; single-GPU twin: sparsh_hierarchy_amg_solve).  One
// graph launch per cycle: the cycle, the fused residual-norm kernel over the local rows, the all-reduce.
int sparsh_dist_amg_solve(sparsh_dist_t h, const double *b, double *x, double tol, int max_cycles, double *hist, int *cycles_out) {
    SP_TRY(check_alive(h));
    Context &c = ctx();
    DistLevel &L0 = h->lev[0];
    const size_t n = (size_t)L0.n;
    double *xs = h->kv[4];
    double *sc = h->d_sc;
    enum { S_RES = 3 };
    auto resnorm = [&]() -> int {  // ||A x - b||^2 over all ranks -> h_sc[S_RES]  (reference :159, :219)
        EpiArgs a;
        a.b = b;
        a.red_out = sc + S_RES;
        SP_TRY(apply(h, L0.A, EPI_RESNORM, xs, nullptr, a));
        SP_TRY(allreduce_sum(h, sc + S_RES, 1));
        SP_CUDA(cudaMemcpyAsync(h->h_sc + S_RES, sc + S_RES, sizeof(double), cudaMemcpyDeviceToHost, c.stream));
        if (h->peer) SP_CUDA(cudaMemcpyAsync(h->h_err, h->d_err, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
        return SPARSH_OK;
    };
    SP_CUDA(cudaMemcpyAsync(xs, x, sizeof(double) * n, cudaMemcpyDeviceToDevice, c.stream));
    SP_TRY(resnorm());
    SP_CUDA(cudaStreamSynchronize(c.stream));
    double r1 = std::sqrt(h->h_sc[S_RES]);
    if (hist) hist[0] = r1;
    auto body = [&]() -> int {
        SP_TRY(enqueue_dist_vcycle(h, b, xs, false));
        return resnorm();
    };
    int cycles = 0, rc = SPARSH_OK;
    while (r1 > tol && cycles < max_cycles) {  // :196 (the reference has no cap: SURVEY F6)
        SP_TRY(dist_run_graphed(h, b, xs, 30, body));
        SP_CUDA(cudaStreamSynchronize(c.stream));
        cycles++;
        if (h->peer && *h->h_err) {
            h->dead = true;
            set_error("multi-GPU halo handshake timed out (a neighbour never signalled); the distributed handle is unusable");
            rc = SPARSH_ERR_CUDA;
            break;
        }
        r1 = std::sqrt(h->h_sc[S_RES]);
        if (hist) hist[cycles] = r1;
        if (!std::isfinite(r1)) break;
    }
    SP_CUDA(cudaMemcpyAsync(x, xs, sizeof(double) * n, cudaMemcpyDeviceToDevice, c.stream));
    SP_CUDA(cudaStreamSynchronize(c.stream));
    if (cycles_out) *cycles_out = cycles;
    if (rc != SPARSH_OK) return rc;
    return r1 <= tol ? SPARSH_OK : SPARSH_ERR_NOT_CONVERGED;
}

// Distributed AMG-preconditioned BiCGStab: the arithmetic of bicg_impl(precond = true) in krylov.cu, i.e. of the
// reference's Solver_PBiCG_1 (src/AMG_main_solvers.cpp:358-458); each group of dot products is completed by one
// in-place all-reduce of adjacent device scalars.
int sparsh_dist_pbicgstab(sparsh_dist_t h, const double *b, double *x, double tol, int max_iter, double *hist, int *iters_out) {
    SP_TRY(check_alive(h));
    Context &c = ctx();
    DistLevel &L0 = h->lev[0];
    const size_t n = (size_t)L0.n;
    for (int i = 0; i < 7; i++)
        if (!h->bv[i]) SP_CUDA(cudaMalloc(&h->bv[i], sizeof(double) * (n + 2)));
    // ph, sh are gathered from by A (arena vectors with halo segments); the others are purely local
    double *ph = h->kv[0], *sh = h->kv[1], *xs = h->kv[4];
    double *r0 = h->bv[0], *r = h->bv[1], *p = h->bv[2], *Ap = h->bv[3], *s = h->bv[4], *As = h->bv[5], *xl = h->bv[6];
    double *sc = h->d_sc;
    enum { S_A1 = 4, S_APR0 = 5, S_ASS = 6, S_ASAS = 7, S_RR0 = 8, S_RRN = 9 };  // as in krylov.cu
    auto read_res = [&]() -> int {
        SP_CUDA(cudaMemcpyAsync(h->h_sc + S_RRN, sc + S_RRN, sizeof(double), cudaMemcpyDeviceToHost, c.stream));
        if (h->peer) SP_CUDA(cudaMemcpyAsync(h->h_err, h->d_err, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
        return SPARSH_OK;
    };
    SP_CUDA(cudaMemcpyAsync(xs, x, sizeof(double) * n, cudaMemcpyDeviceToDevice, c.stream));
    SP_CUDA(cudaMemcpyAsync(xl, x, sizeof(double) * n, cudaMemcpyDeviceToDevice, c.stream));
    EpiArgs a;
    a.b = b;
    SP_TRY(apply(h, L0.A, EPI_RESID, xs, r0, a));                                                 // :383-384
    SP_CUDA(cudaMemcpyAsync(r, r0, sizeof(double) * n, cudaMemcpyDeviceToDevice, c.stream));      // :387
    SP_CUDA(cudaMemcpyAsync(p, r0, sizeof(double) * n, cudaMemcpyDeviceToDevice, c.stream));      // :388
    SP_TRY(k_dot(n, r0, r0, sc + S_RRN));                                                         // :390
    SP_TRY(allreduce_sum(h, sc + S_RRN, 1));
    SP_TRY(read_res());
    SP_CUDA(cudaStreamSynchronize(c.stream));
    double res = std::sqrt(h->h_sc[S_RRN]);
    if (hist) hist[0] = res;

    auto body = [&]() -> int {
        SP_TRY(enqueue_dist_vcycle(h, p, ph, true));                             // :399-400
        SP_TRY(k_dot(n, r, r0, sc + S_A1));                                      // :402
        SP_TRY(apply(h, L0.A, EPI_SPMV, ph, Ap, EpiArgs()));                     // :403
        SP_TRY(k_dot(n, Ap, r0, sc + S_APR0));                                   // :404
        SP_TRY(allreduce_sum(h, sc + S_A1, 2));                                  // (S_A1, S_APR0 adjacent)
        SP_TRY(k_bicg_s(n, r, Ap, s, sc + S_A1, sc + S_APR0));                   // :406-411
        SP_TRY(enqueue_dist_vcycle(h, s, sh, true));                             // :414-415
        SP_TRY(apply(h, L0.A, EPI_SPMV, sh, As, EpiArgs()));                     // :416
        SP_TRY(k_dot2(n, As, s, As, sc + S_ASS));                                // :418-419
        SP_TRY(allreduce_sum(h, sc + S_ASS, 2));
        SP_TRY(k_bicg_xr(n, xl, ph, sh, s, As, r, sc + S_A1, sc + S_APR0, sc + S_ASS, sc + S_ASAS, r0, sc + S_RR0));  // :424-425
        SP_TRY(allreduce_sum(h, sc + S_RR0, 2));                                 // r.r0 (:428) and r.r (:437)
        SP_TRY(k_bicg_p(n, r, p, Ap, sc + S_A1));                                // :428-434
        return read_res();
    };
    int count = 0, rc = SPARSH_OK;
    while (res > tol && count < max_iter) {  // :397 (no cap in the reference)
        SP_TRY(dist_run_graphed(h, x, b, 20, body));
        SP_CUDA(cudaStreamSynchronize(c.stream));
        count++;
        if (h->peer && *h->h_err) {
            h->dead = true;
            set_error("multi-GPU halo handshake timed out (a neighbour never signalled); the distributed handle is unusable");
            rc = SPARSH_ERR_CUDA;
            break;
        }
        res = std::sqrt(h->h_sc[S_RRN]);     // :437
        if (hist) hist[count] = res;
        if (!std::isfinite(res)) break;
    }
    SP_CUDA(cudaMemcpyAsync(x, xl, sizeof(double) * n, cudaMemcpyDeviceToDevice, c.stream));
    SP_CUDA(cudaStreamSynchronize(c.stream));
    if (iters_out) *iters_out = count;
    if (rc != SPARSH_OK) return rc;
    return res <= tol ? SPARSH_OK : SPARSH_ERR_NOT_CONVERGED;
}

}  // extern "C"

// spmv_common.cuh — device helpers shared by the row-sum kernel families (spmv.cu, spmv_pattern.cu): mbarrier / TMA
// bulk-copy PTX, the multi-GPU flag handshake fused into the consuming kernel, the epilogues, and the block reduction.
#pragma once
#include "internal.cuh"

namespace sparsh {

// ---------------------------------------------------------------------------------------------------------
// PTX helpers: mbarrier + 1-D TMA bulk copy global -> shared
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "SPARSH_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra SPARSH_DONE;\n"
        "bra SPARSH_WAIT;\n"
        "SPARSH_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// dst/src 16-byte aligned, bytes a multiple of 16
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// ---------------------------------------------------------------------------------------------------------
// Multi-GPU flag handshake fused into the consumer (see HaloSync in internal.cuh, producer side in dist.cu)
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ sparsh_u64 ld_acquire_sys_u64(const sparsh_u64 *p) {
    sparsh_u64 v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys_u64(sparsh_u64 *p, sparsh_u64 v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// a flag store that follows a __threadfence_system() of the same thread: the fence orders everything before it, so
// several flags can go out back to back without paying one system-scope membar each (st.release = membar + store)
__device__ __forceinline__ void st_relaxed_sys_u64(sparsh_u64 *p, sparsh_u64 v) {
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
struct HaloTurn {
    sparsh_u64 want, prev;
};
__device__ __forceinline__ long long global_ns() {
    long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void spin_ge(const sparsh_u64 *p, sparsh_u64 v, int *err, long long timeout_ns) {
    if (ld_acquire_sys_u64(p) >= v) return;
    const long long t0 = global_ns();
    while (ld_acquire_sys_u64(p) < v) {
        // a broken handshake must never hang the GPU: give up after timeout_ns of wall clock (ranks may legitimately be
        // seconds apart: graph instantiation, lazy module loads), and at once if somebody already did
        if (*reinterpret_cast<volatile int *>(err) != 0) break;
        if (global_ns() - t0 > timeout_ns) {
            atomicExch(err, 1);
            break;
        }
        __nanosleep(32);
    }
}
// called by every thread of the CTA, before the first gather of x; contains a CTA barrier
__device__ __forceinline__ HaloTurn halo_wait(const HaloSync &hs) {
    HaloTurn t;
    t.want = 0;
    t.prev = 0;
    if ((hs.nnbr == 0 && hs.nsend == 0) || (int)blockIdx.x >= hs.nstrip) return t;  // interior CTAs: nothing to wait for
    if (hs.nnbr > 0) t.want = *reinterpret_cast<const volatile sparsh_u64 *>(hs.expect) + 1;
    if (hs.nsend > 0) t.prev = *reinterpret_cast<const volatile sparsh_u64 *>(hs.seq);
    const int tid = threadIdx.x;
    if (tid < hs.nnbr) spin_ge(hs.flag_local[tid], t.want, hs.err, hs.timeout_ns);                         // slices have landed
    // The fused push writes into the ping-pong partner of the vector being read, whose halo segment last held slice
    // prev-1 (slice prev is the one this very kernel consumes): everything up to prev-1 must have been consumed.
    // Waiting for slice prev itself would deadlock — both neighbours only ack it when this sweep ends.
    if (tid >= 8 && tid - 8 < hs.nsend) spin_ge(hs.ack_local[tid - 8], t.prev > 0 ? t.prev - 1 : 0, hs.err, hs.timeout_ns);
    __syncthreads();
    return t;
}
// called by every thread of the CTA after its last read of x and its last remote store
__device__ __forceinline__ void halo_done(const HaloSync &hs, const HaloTurn &t) {
    if ((hs.nnbr == 0 && hs.nsend == 0) || (int)blockIdx.x >= hs.nstrip) return;
    if (hs.nsend > 0) __threadfence_system();  // my remote stores are performed before anyone sees the flag
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int k = atomicAdd(hs.ticket, 1u);
        if (k == (unsigned int)hs.nstrip - 1u) {  // the last STRIP CTA: neighbours hear from us while the interior still runs
            // every strip CTA fenced (system scope) before it took its ticket; ONE more fence here orders all of that
            // before the acks and flags, which then leave back to back as relaxed stores
            __threadfence_system();
            if (hs.nnbr > 0) {
                *reinterpret_cast<volatile sparsh_u64 *>(hs.expect) = t.want;
                for (int q = 0; q < hs.nnbr; q++) st_relaxed_sys_u64(hs.ack_dst[q], t.want);
            }
            if (hs.nsend > 0) {
                for (int q = 0; q < hs.nsend; q++) st_relaxed_sys_u64(hs.flag_dst[q], t.prev + 1);
                *reinterpret_cast<volatile sparsh_u64 *>(hs.seq) = t.prev + 1;
            }
            *hs.ticket = 0u;
            __threadfence();
        }
    }
}
__device__ __forceinline__ void block_rows(const RowRange &rr, int rows_per_cta, int &first, int &end) {
    int blk = blockIdx.x;
    first = rr.b1;
    end = rr.e1;
    if (blk >= rr.nblk1) {
        blk -= rr.nblk1;
        first = rr.b2;
        end = rr.e2;
        if (blk >= rr.nblk2) {
            blk -= rr.nblk2;
            first = rr.b3;
            end = rr.e3;
        }
    }
    first += blk * rows_per_cta;
}

// ---------------------------------------------------------------------------------------------------------
// Epilogues.  Arithmetic and evaluation order follow the reference's CPU path (SURVEY Appendix A):
//   store_residual   r = b - (A x)                              src/AMG_cycle_utilities.cpp:120-121
//   jacobi           x += (omega*(b - A x))/d                   src/AMG_smoothers.cpp:62-71
//   transfer_solution xf = (P xc) + xf                          src/AMG_cycle_utilities.cpp:111
//   sor (one colour) x -= (omega*((A x) - b))/d                 src/AMG_smoothers.cpp:90-98
//   residual         ||(A x) - b||                              src/AMG_cycle_utilities.cpp:88-92
// ---------------------------------------------------------------------------------------------------------
struct EpiRegs {
    double b, xi, d;
};

template <int EPI, bool LOAD_D = true>
__device__ __forceinline__ EpiRegs epi_load(const EpiArgs &a, const double *y, int row) {
    EpiRegs e;
    e.b = 0.0;
    e.xi = 0.0;
    e.d = 1.0;
    if (EPI == EPI_RESID || EPI == EPI_JACOBI || EPI == EPI_SOR || EPI == EPI_RESNORM) e.b = a.b[row];
    if (EPI == EPI_JACOBI || EPI == EPI_SPMV_DOT) e.xi = a.xi[row];
    if (EPI == EPI_PROLONG || EPI == EPI_SOR) e.xi = y[row];
    if (LOAD_D && (EPI == EPI_JACOBI || EPI == EPI_SOR)) e.d = a.d[row];
    return e;
}

// returns this row's contribution to the fused reduction (0 when the epilogue has none)
template <int EPI, bool PUSH>
__device__ __forceinline__ double epi_store(const EpiArgs &a, const EpiRegs &e, double s, double *y, int row,
                                            bool strip = true) {
    if (EPI == EPI_SPMV) {
        y[row] = s;
    } else if (EPI == EPI_RESID) {
        y[row] = __dsub_rn(e.b, s);
    } else if (EPI == EPI_JACOBI) {
        double h = __dsub_rn(e.b, s);
        const double v = __dadd_rn(e.xi, __ddiv_rn(__dmul_rn(a.omega, h), e.d));
        y[row] = v;  // (multi-GPU: the boundary strips push it to the neighbours afterwards, see fused_push)
    } else if (EPI == EPI_PROLONG) {
        y[row] = __dadd_rn(s, e.xi);
    } else if (EPI == EPI_SOR) {
        double h = __dsub_rn(s, e.b);
        y[row] = __dsub_rn(e.xi, __ddiv_rn(__dmul_rn(a.omega, h), e.d));
    } else if (EPI == EPI_SPMV_DOT) {
        y[row] = s;
        return __dmul_rn(e.xi, s);
    } else if (EPI == EPI_RESNORM) {
        double h = __dsub_rn(s, e.b);
        return __dmul_rn(h, h);
    }
    return 0.0;
}

// Multi-GPU, fused Jacobi + halo exchange: a row whose new value a neighbour needs stores it ALSO into that neighbour's
// halo segment of the next sweep's input vector (peer store over NVLink).  Called by the strip CTAs for each of their
// rows AFTER the row sums, as a phase of its own: kept out of the row loop it costs the hot path no register (inside
// epi_store it took the plain-CSR kernel from 32 to 64 registers, i.e. from 8 to 4 resident CTAs per SM).
template <int EPI, bool DIST>
__device__ __forceinline__ void fused_push(const EpiArgs &a, const double *y, int row) {
    if (DIST && EPI == EPI_JACOBI) {
        const int lo = a.pm_ptr[row], hi = a.pm_ptr[row + 1];
        if (lo < hi) {
            const double v = y[row];  // written by this very thread
            for (int k = lo; k < hi; k++) a.pm_dst[a.pm_nbr[k]][a.pm_off[k]] = v;
        }
    }
}
template <int EPI, bool DIST>
__device__ __forceinline__ bool pushes(const EpiArgs &a, bool strip_cta) {
    return DIST && EPI == EPI_JACOBI && strip_cta && a.pm_ptr != nullptr;
}

template <int EPI>
struct EpiTraits {
    static constexpr bool reduces = (EPI == EPI_SPMV_DOT || EPI == EPI_RESNORM);
    // multicolour SOR updates x in place: its gathers must not use the non-coherent path
    static constexpr bool coherent_x = (EPI == EPI_SOR);
};

// multi-GPU kernels: halo entries are written by peers over NVLink while the grid may already be resident, so the
// non-coherent path (ld.global.nc: data must be read-only for the kernel's lifetime) is off limits for the gathered
// vector.  Plain loads are ordered behind the flag acquire + CTA barrier of halo_wait, and a stale L1 line cannot exist:
// halo segments start on 128-byte boundaries (dist.cu), no CTA reads a halo entry before its flags are up, and interior
// CTAs never reference one.  (halo_begin is kept for kernels that want to tell the two apart.)
template <bool COHERENT, bool DIST>
__device__ __forceinline__ double load_xd(const double *x, int c, int /*halo_begin*/) {
    // (measured: plain loads cost the single-GPU kernels nothing — profiles/r02g_pattern_lean_v3_sweep.log, PLAIN rows)
    if (COHERENT || DIST) return x[c];
    return __ldg(x + c);
}

// ---------------------------------------------------------------------------------------------------------
// Deterministic two-stage reduction: fixed shuffle tree per block, block partials to global memory, then one CTA
// adds the partials in index order.  The result does not depend on block scheduling: bit-reproducible run to run.
// ---------------------------------------------------------------------------------------------------------
template <int THREADS>
__device__ __forceinline__ double block_sum(double v, double *sred) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncthreads();  // sred may still be read from a previous call
    if (lane == 0) sred[warp] = v;
    __syncthreads();
    v = (threadIdx.x < THREADS / 32) ? sred[threadIdx.x] : 0.0;
    if (warp == 0) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    }
    return v;  // valid in thread 0
}

// stage 1: one partial per block (fixed shuffle tree)
template <int THREADS>
__device__ __forceinline__ void block_partial(double contrib, double *partials) {
    __shared__ double sred[32];
    double v = block_sum<THREADS>(contrib, sred);
    if (threadIdx.x == 0) partials[blockIdx.x] = v;
}

// ---- launch plumbing shared by the kernel families --------------------------------------------------------------
struct LaunchDesc {
    RowRange rr;
    int rows1, rows2, rows3;
    HaloSync hs;
    bool dist = false;  // multi-GPU variant of the kernel (handshake + fused push compiled in)
};

inline int grid_for(LaunchDesc &d, int rows_per_cta) {
    const int n1 = (d.rows1 + rows_per_cta - 1) / rows_per_cta, n2 = (d.rows2 + rows_per_cta - 1) / rows_per_cta;
    const int n3 = (d.rows3 + rows_per_cta - 1) / rows_per_cta;
    d.rr.nblk1 = n1;
    d.rr.nblk2 = n2;
    d.hs.nstrip = n1 + n2;  // the CTAs of ranges 1 and 2 run the handshake; range 3 (interior rows) never waits
    return n1 + n2 + n3;
}

// csr-pattern8, lean variant (spmv_pattern.cu): applies when pattern 0 is short enough to travel in the kernel
// parameters and covers most rows; launch_pattern_lean runs `epi` over the rows of `d`
bool pattern_lean_applies(const sparsh_matrix_s *A);
int launch_pattern_lean(const sparsh_matrix_s *A, int epi, const double *x, double *y, const EpiArgs &args, LaunchDesc d);

// stage 2 of the fused reductions (spmv.cu): one CTA adds the `count` block partials in index order into *out
int launch_finalize_partials(int count, double *out);

}  // namespace sparsh

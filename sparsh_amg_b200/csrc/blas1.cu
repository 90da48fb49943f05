// blas1.cu — K8 of SURVEY §8a: vector kernels of the Krylov loops and their fused variants.
//
// Replaces cublasDdot/Dnrm2/Daxpy and the hand-written daxpby/daxpbyc of src/AMG_main_solvers.cu:17-33, plus the
// OpenMP loops of src/AMG_main_solvers.cpp:408-435.  All are pure HBM streams: 128-bit accesses where alignment
// allows, grid = a fixed multiple of the SM count (grid-stride), Krylov scalars stay in device memory so nothing
// syncs the host inside an iteration.  Reductions use the fixed two-stage tree of spmv.cu's scheme (bit-reproducible).
// Element-wise arithmetic uses separate mul/add in the reference's expression order, so vectors are bit-identical to
// the CPU path given identical scalars.
#include "internal.cuh"

namespace sparsh {

constexpr int BT = 256;

static inline int stream_grid(size_t n, int per_thread = 4) {
    Context &c = ctx();
    size_t want = (n + (size_t)BT * per_thread - 1) / ((size_t)BT * per_thread);
    size_t cap = (size_t)c.sm_count * 8;  // 8 resident CTAs of 256 threads per SM
    if (want < 1) want = 1;
    return (int)(want < cap ? want : cap);
}

// ---- deterministic reductions of up to 3 values -----------------------------------------------------------
template <int NV>
__device__ __forceinline__ void reduce_finalize(double (&v)[NV], double *partials, unsigned int *ticket, double *out) {
    __shared__ double sred[NV][32];
    __shared__ int s_last;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int q = 0; q < NV; q++) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v[q] += __shfl_xor_sync(0xffffffffu, v[q], off);
        if (lane == 0) sred[q][warp] = v[q];
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int q = 0; q < NV; q++) {
            double t = lane < BT / 32 ? sred[q][lane] : 0.0;
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) t += __shfl_xor_sync(0xffffffffu, t, off);
            if (lane == 0) partials[(size_t)q * RED_MAX_BLOCKS + blockIdx.x] = t;
        }
        if (lane == 0) {
            __threadfence();
            unsigned int tk = atomicAdd(ticket, 1u);
            s_last = (tk == gridDim.x - 1);
        }
    }
    __syncthreads();
    if (s_last) {
        __threadfence();
        double acc[NV];
#pragma unroll
        for (int q = 0; q < NV; q++) {
            acc[q] = 0.0;
            for (unsigned int i = threadIdx.x; i < gridDim.x; i += BT)
                acc[q] += __ldcg(partials + (size_t)q * RED_MAX_BLOCKS + i);
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], off);
        }
        __syncthreads();
        if (lane == 0)
#pragma unroll
            for (int q = 0; q < NV; q++) sred[q][warp] = acc[q];
        __syncthreads();
        if (warp == 0) {
#pragma unroll
            for (int q = 0; q < NV; q++) {
                double t = lane < BT / 32 ? sred[q][lane] : 0.0;
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) t += __shfl_xor_sync(0xffffffffu, t, off);
                if (lane == 0) out[q] = t;
            }
            if (lane == 0) *ticket = 0u;
        }
    }
}

// ---- element-wise ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(BT) fill_kernel(double *x, size_t n, double v) {
    for (size_t i = (size_t)blockIdx.x * BT + threadIdx.x; i < n; i += (size_t)gridDim.x * BT) x[i] = v;
}
__global__ void __launch_bounds__(BT) axpy_kernel(size_t n, double a, const double *__restrict__ x, double *y) {
    for (size_t i = (size_t)blockIdx.x * BT + threadIdx.x; i < n; i += (size_t)gridDim.x * BT)
        y[i] = __dadd_rn(y[i], __dmul_rn(a, x[i]));
}
__global__ void __launch_bounds__(BT) axpby_kernel(size_t n, double a, const double *__restrict__ x, double b, double *y) {
    for (size_t i = (size_t)blockIdx.x * BT + threadIdx.x; i < n; i += (size_t)gridDim.x * BT)
        y[i] = __dadd_rn(__dmul_rn(a, x[i]), __dmul_rn(b, y[i]));
}
// daxpbyc of src/AMG_main_solvers.cu:26-33: c = alpha*x + beta*y + gamma*c
__global__ void __launch_bounds__(BT)
    axpbypcz_kernel(size_t n, double a, const double *__restrict__ x, double b, const double *__restrict__ y, double c, double *z) {
    for (size_t i = (size_t)blockIdx.x * BT + threadIdx.x; i < n; i += (size_t)gridDim.x * BT)
        z[i] = __dadd_rn(__dadd_rn(__dmul_rn(a, x[i]), __dmul_rn(b, y[i])), __dmul_rn(c, z[i]));
}
// first Jacobi sweep from a zero guess: A*0 = 0, h = b - 0, x = 0 + (omega*h)/d   (src/AMG_smoothers.cpp:62-71)
__global__ void __launch_bounds__(BT)
    jacobi_zero_kernel(size_t n, const double *__restrict__ b, const double *__restrict__ d, double omega, double *x) {
    for (size_t i = (size_t)blockIdx.x * BT + threadIdx.x; i < n; i += (size_t)gridDim.x * BT)
        x[i] = __ddiv_rn(__dmul_rn(omega, b[i]), d[i]);
}

__global__ void __launch_bounds__(BT)
    dot_kernel(size_t n, const double *__restrict__ x, const double *__restrict__ y, double *partials, unsigned int *ticket, double *out) {
    double v[1] = {0.0};
    for (size_t i = (size_t)blockIdx.x * BT + threadIdx.x; i < n; i += (size_t)gridDim.x * BT)
        v[0] = __dadd_rn(v[0], __dmul_rn(x[i], y[i]));
    reduce_finalize<1>(v, partials, ticket, out);
}
__global__ void __launch_bounds__(BT)
    dot2_kernel(size_t n, const double *__restrict__ a, const double *__restrict__ b, const double *__restrict__ c, double *partials,
                unsigned int *ticket, double *out) {
    double v[2] = {0.0, 0.0};
    for (size_t i = (size_t)blockIdx.x * BT + threadIdx.x; i < n; i += (size_t)gridDim.x * BT) {
        const double ai = a[i];
        v[0] = __dadd_rn(v[0], __dmul_rn(ai, b[i]));
        v[1] = __dadd_rn(v[1], __dmul_rn(ai, c[i]));
    }
    reduce_finalize<2>(v, partials, ticket, out);
}

// ---- GMRES(m) building blocks (not in the reference, SURVEY §8f.2; arithmetic order = oracle so_gmres) ------------
// up to 4 dots of w against consecutive basis vectors in ONE pass over w: out[q] = V_q . w
__global__ void __launch_bounds__(BT)
    mdot4_kernel(size_t n, const double *__restrict__ V, size_t ld, int cnt, const double *__restrict__ w, double *partials,
                 unsigned int *ticket, double *out) {
    double v[4] = {0.0, 0.0, 0.0, 0.0};
    for (size_t i = (size_t)blockIdx.x * BT + threadIdx.x; i < n; i += (size_t)gridDim.x * BT) {
        const double wi = w[i];
#pragma unroll
        for (int q = 0; q < 4; q++)
            if (q < cnt) v[q] = __dadd_rn(v[q], __dmul_rn(V[(size_t)q * ld + i], wi));
    }
    reduce_finalize<4>(v, partials, ticket, out);
}
// w -= sum_q h[q] V_q  (q ascending; h in device memory)
__global__ void __launch_bounds__(BT)
    maxpy_sub_kernel(size_t n, const double *__restrict__ V, size_t ld, int k, const double *__restrict__ h, double *w) {
    extern __shared__ double sh[];
    for (int q = threadIdx.x; q < k; q += BT) sh[q] = h[q];
    __syncthreads();
    for (size_t i = (size_t)blockIdx.x * BT + threadIdx.x; i < n; i += (size_t)gridDim.x * BT) {
        double t = w[i];
        for (int q = 0; q < k; q++) t = __dsub_rn(t, __dmul_rn(sh[q], V[(size_t)q * ld + i]));
        w[i] = t;
    }
}
// out = sum_q y[q] V_q  (q ascending, from 0.0)
__global__ void __launch_bounds__(BT)
    lincomb_kernel(size_t n, const double *__restrict__ V, size_t ld, int k, const double *__restrict__ y, double *out) {
    extern __shared__ double sh[];
    for (int q = threadIdx.x; q < k; q += BT) sh[q] = y[q];
    __syncthreads();
    for (size_t i = (size_t)blockIdx.x * BT + threadIdx.x; i < n; i += (size_t)gridDim.x * BT) {
        double t = 0.0;
        for (int q = 0; q < k; q++) t = __dadd_rn(t, __dmul_rn(sh[q], V[(size_t)q * ld + i]));
        out[i] = t;
    }
}
// out = in / sqrt(*nrm2)
__global__ void __launch_bounds__(BT)
    scale_inv_sqrt_kernel(size_t n, const double *__restrict__ in, const double *nrm2, double *out) {
    const double d = sqrt(*nrm2);
    for (size_t i = (size_t)blockIdx.x * BT + threadIdx.x; i < n; i += (size_t)gridDim.x * BT) out[i] = __ddiv_rn(in[i], d);
}

// ---- PCG (src/AMG_main_solvers.cpp:140-150) -----------------------------------------------------------------
// alpha = rz/pAp (:142); x += alpha p (:144); r += (-alpha) Ap (:145); rr = r.r (for :152)
__global__ void __launch_bounds__(BT)
    pcg_update_xr_kernel(size_t n, const double *__restrict__ p, const double *__restrict__ Ap, double *x, double *r,
                         const double *rz, const double *pAp, double *partials, unsigned int *ticket, double *rr_out) {
    const double alpha = *rz / *pAp;
    const double nalpha = -alpha;
    double v[1] = {0.0};
    for (size_t i = (size_t)blockIdx.x * BT + threadIdx.x; i < n; i += (size_t)gridDim.x * BT) {
        x[i] = __dadd_rn(x[i], __dmul_rn(alpha, p[i]));
        const double ri = __dadd_rn(r[i], __dmul_rn(nalpha, Ap[i]));
        r[i] = ri;
        v[0] = __dadd_rn(v[0], __dmul_rn(ri, ri));
    }
    reduce_finalize<1>(v, partials, ticket, rr_out);
}
// beta = rz_new/rz_old (:149); p = 1.0*z + beta*p (:150)
__global__ void __launch_bounds__(BT)
    pcg_update_p_kernel(size_t n, const double *__restrict__ z, double *p, const double *rz_new, const double *rz_old) {
    const double beta = *rz_new / *rz_old;
    for (size_t i = (size_t)blockIdx.x * BT + threadIdx.x; i < n; i += (size_t)gridDim.x * BT)
        p[i] = __dadd_rn(z[i], __dmul_rn(beta, p[i]));
}
__global__ void scalar_copy_kernel(double *dst, const double *src) {
    *dst = *src;
}

// ---- BiCGStab (src/AMG_main_solvers.cpp:402-435) -------------------------------------------------------------
// s = r - alpha*Ap, alpha = alpha1/apr0 (:406-411)
__global__ void __launch_bounds__(BT)
    bicg_s_kernel(size_t n, const double *__restrict__ r, const double *__restrict__ Ap, double *s, const double *alpha1, const double *apr0) {
    const double alpha = *alpha1 / *apr0;
    for (size_t i = (size_t)blockIdx.x * BT + threadIdx.x; i < n; i += (size_t)gridDim.x * BT)
        s[i] = __dsub_rn(r[i], __dmul_rn(alpha, Ap[i]));
}
// omega1 = ass/asas (:418-419); x = x + alpha*ph + omega1*sh (:424); r = s - omega1*As (:425);
// out2[0] = r.r0 (for :428), out2[1] = r.r (for :437)
__global__ void __launch_bounds__(BT)
    bicg_xr_kernel(size_t n, double *x, const double *__restrict__ ph, const double *__restrict__ sh, const double *__restrict__ s,
                   const double *__restrict__ As, double *r, const double *alpha1, const double *apr0, const double *ass,
                   const double *asas, const double *__restrict__ r0, double *partials, unsigned int *ticket, double *out2) {
    const double alpha = *alpha1 / *apr0;
    const double omega1 = *ass / *asas;
    double v[2] = {0.0, 0.0};
    for (size_t i = (size_t)blockIdx.x * BT + threadIdx.x; i < n; i += (size_t)gridDim.x * BT) {
        x[i] = __dadd_rn(__dadd_rn(x[i], __dmul_rn(alpha, ph[i])), __dmul_rn(omega1, sh[i]));
        const double ri = __dsub_rn(s[i], __dmul_rn(omega1, As[i]));
        r[i] = ri;
        v[0] = __dadd_rn(v[0], __dmul_rn(ri, r0[i]));
        v[1] = __dadd_rn(v[1], __dmul_rn(ri, ri));
    }
    reduce_finalize<2>(v, partials, ticket, out2);
}
// sc[0]=alpha1 sc[1]=apr0 sc[2]=ass sc[3]=asas sc[4]=r.r0(new):  beta = (sc4/sc0)*(alpha/omega1) (:428-429);
// p = r + beta*(p - omega1*Ap) (:434)
__global__ void __launch_bounds__(BT) bicg_p_kernel(size_t n, const double *__restrict__ r, double *p, const double *__restrict__ Ap, const double *sc) {
    const double alpha = sc[0] / sc[1];
    const double omega1 = sc[2] / sc[3];
    double beta = sc[4] / sc[0];
    beta = beta * (alpha / omega1);
    for (size_t i = (size_t)blockIdx.x * BT + threadIdx.x; i < n; i += (size_t)gridDim.x * BT)
        p[i] = __dadd_rn(r[i], __dmul_rn(beta, __dsub_rn(p[i], __dmul_rn(omega1, Ap[i]))));
}
// CG (src/AMG_main_solvers.cpp:82-83): beta = rr_new/rr_old; p = 1.0*r + beta*p
__global__ void __launch_bounds__(BT)
    cg_update_p_kernel(size_t n, const double *__restrict__ r, double *p, const double *rr_new, const double *rr_old) {
    const double beta = *rr_new / *rr_old;
    for (size_t i = (size_t)blockIdx.x * BT + threadIdx.x; i < n; i += (size_t)gridDim.x * BT)
        p[i] = __dadd_rn(r[i], __dmul_rn(beta, p[i]));
}

// ---- host launchers ----------------------------------------------------------------------------------------------
#define LAUNCH_CHECK()            \
    do {                          \
        count_launch();           \
        SP_CUDA(cudaGetLastError()); \
        return SPARSH_OK;         \
    } while (0)

int k_fill(double *x, size_t n, double v) {
    if (n == 0) return SPARSH_OK;
    fill_kernel<<<stream_grid(n), BT, 0, ctx().stream>>>(x, n, v);
    LAUNCH_CHECK();
}
int k_axpy(size_t n, double a, const double *x, double *y) {
    if (n == 0) return SPARSH_OK;
    axpy_kernel<<<stream_grid(n), BT, 0, ctx().stream>>>(n, a, x, y);
    LAUNCH_CHECK();
}
int k_axpby(size_t n, double a, const double *x, double b, double *y) {
    if (n == 0) return SPARSH_OK;
    axpby_kernel<<<stream_grid(n), BT, 0, ctx().stream>>>(n, a, x, b, y);
    LAUNCH_CHECK();
}
int k_axpbypcz(size_t n, double a, const double *x, double b, const double *y, double c, double *z) {
    if (n == 0) return SPARSH_OK;
    axpbypcz_kernel<<<stream_grid(n), BT, 0, ctx().stream>>>(n, a, x, b, y, c, z);
    LAUNCH_CHECK();
}
int k_jacobi_zero(size_t n, const double *b, const double *d, double omega, double *x) {
    if (n == 0) return SPARSH_OK;
    jacobi_zero_kernel<<<stream_grid(n), BT, 0, ctx().stream>>>(n, b, d, omega, x);
    LAUNCH_CHECK();
}
int k_dot(size_t n, const double *x, const double *y, double *d_out) {
    Context &c = ctx();
    dot_kernel<<<stream_grid(n), BT, 0, c.stream>>>(n, x, y, c.partials, c.ticket, d_out);
    LAUNCH_CHECK();
}
int k_dot2(size_t n, const double *a, const double *b, const double *cc, double *d_out2) {
    Context &c = ctx();
    dot2_kernel<<<stream_grid(n), BT, 0, c.stream>>>(n, a, b, cc, c.partials, c.ticket, d_out2);
    LAUNCH_CHECK();
}
int k_mdot(size_t n, const double *V, size_t ld, int k, const double *w, double *d_out) {
    Context &c = ctx();
    for (int j0 = 0; j0 < k; j0 += 4) {  // d_out must have room for k rounded up to a multiple of 4
        mdot4_kernel<<<stream_grid(n), BT, 0, c.stream>>>(n, V + (size_t)j0 * ld, ld, k - j0 < 4 ? k - j0 : 4, w, c.partials, c.ticket, d_out + j0);
        count_launch();
        SP_CUDA(cudaGetLastError());
    }
    return SPARSH_OK;
}
int k_maxpy_sub(size_t n, const double *V, size_t ld, int k, const double *d_h, double *w) {
    maxpy_sub_kernel<<<stream_grid(n), BT, sizeof(double) * (size_t)k, ctx().stream>>>(n, V, ld, k, d_h, w);
    LAUNCH_CHECK();
}
int k_lincomb(size_t n, const double *V, size_t ld, int k, const double *d_y, double *out) {
    lincomb_kernel<<<stream_grid(n), BT, sizeof(double) * (size_t)k, ctx().stream>>>(n, V, ld, k, d_y, out);
    LAUNCH_CHECK();
}
int k_scale_inv_sqrt(size_t n, const double *in, const double *d_nrm2, double *out) {
    scale_inv_sqrt_kernel<<<stream_grid(n), BT, 0, ctx().stream>>>(n, in, d_nrm2, out);
    LAUNCH_CHECK();
}
int k_pcg_update_xr(size_t n, const double *p, const double *Ap, double *x, double *r, const double *rz,
                    const double *pAp, double *rr_out) {
    Context &c = ctx();
    pcg_update_xr_kernel<<<stream_grid(n), BT, 0, c.stream>>>(n, p, Ap, x, r, rz, pAp, c.partials, c.ticket, rr_out);
    LAUNCH_CHECK();
}
int k_pcg_update_p(size_t n, const double *z, double *p, const double *rz_new, const double *rz_old) {
    pcg_update_p_kernel<<<stream_grid(n), BT, 0, ctx().stream>>>(n, z, p, rz_new, rz_old);
    LAUNCH_CHECK();
}
int k_scalar_copy(double *dst, const double *src) {
    scalar_copy_kernel<<<1, 1, 0, ctx().stream>>>(dst, src);
    LAUNCH_CHECK();
}
int k_cg_update_p(size_t n, const double *r, double *p, const double *rr_new, const double *rr_old) {
    cg_update_p_kernel<<<stream_grid(n), BT, 0, ctx().stream>>>(n, r, p, rr_new, rr_old);
    LAUNCH_CHECK();
}
int k_bicg_s(size_t n, const double *r, const double *Ap, double *s, const double *alpha1, const double *apr0) {
    bicg_s_kernel<<<stream_grid(n), BT, 0, ctx().stream>>>(n, r, Ap, s, alpha1, apr0);
    LAUNCH_CHECK();
}
int k_bicg_xr(size_t n, double *x, const double *ph, const double *sh, const double *s, const double *As, double *r,
              const double *alpha1, const double *apr0, const double *ass, const double *asas, const double *r0,
              double *out2) {
    Context &c = ctx();
    bicg_xr_kernel<<<stream_grid(n), BT, 0, c.stream>>>(n, x, ph, sh, s, As, r, alpha1, apr0, ass, asas, r0, c.partials, c.ticket, out2);
    LAUNCH_CHECK();
}
int k_bicg_p(size_t n, const double *r, double *p, const double *Ap, const double *sc) {
    bicg_p_kernel<<<stream_grid(n), BT, 0, ctx().stream>>>(n, r, p, Ap, sc);
    LAUNCH_CHECK();
}

}  // namespace sparsh

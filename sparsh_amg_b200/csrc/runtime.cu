// runtime.cu — context, streams, memory and BLAS-1 entry points of the C-ABI (include/sparsh_b200.h).
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <vector>

#include "internal.cuh"

namespace sparsh {

static thread_local std::string g_err;
void set_error(const std::string &msg) { g_err = msg; }
int cuda_fail(cudaError_t e, const char *what, const char *file, int line) {
    char buf[512];
    snprintf(buf, sizeof buf, "CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e), file, line, what);
    g_err = buf;
    return e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ? SPARSH_ERR_NO_DEVICE : SPARSH_ERR_CUDA;
}

Context &ctx() {
    static Context c;
    return c;
}

int ensure_init() {
    if (ctx().ready) return SPARSH_OK;
    return sparsh_init(0);
}

}  // namespace sparsh

using namespace sparsh;

// ---- slab / scratch allocation (internal.cuh) -----------------------------------------------------------------------------
namespace sparsh {
struct DevSlab {
    char *base = nullptr;
    size_t size = 0;
    std::atomic<size_t> used{0};
};
namespace {
std::mutex g_slab_mutex;
std::vector<DevSlab *> g_slabs;  // live slabs: dev_free looks a pointer up here
thread_local DevSlab *t_slab = nullptr;
thread_local void *t_scratch = nullptr;
thread_local size_t t_scratch_bytes = 0;
}  // namespace

DevSlab *slab_create(size_t bytes) {
    if (bytes == 0) return nullptr;
    DevSlab *s = new DevSlab();
    if (cudaMalloc(&s->base, bytes) != cudaSuccess) {
        cudaGetLastError();
        delete s;
        return nullptr;
    }
    s->size = bytes;
    std::lock_guard<std::mutex> g(g_slab_mutex);
    g_slabs.push_back(s);
    return s;
}
void slab_bind(DevSlab *s) { t_slab = s; }
bool slab_bound() { return t_slab != nullptr; }
void slab_destroy(DevSlab *s) {
    if (!s) return;
    {
        std::lock_guard<std::mutex> g(g_slab_mutex);
        g_slabs.erase(std::remove(g_slabs.begin(), g_slabs.end(), s), g_slabs.end());
    }
    cudaFree(s->base);
    delete s;
}
cudaError_t dev_alloc_bytes(void **p, size_t bytes) {
    if (DevSlab *s = t_slab) {
        // the bump pointer only ever moves forward (compare-and-swap, never an add that is taken back: a rejected
        // request must not disturb the offsets concurrent threads are handed)
        const size_t need = (std::max<size_t>(bytes, 1) + 255) & ~(size_t)255;
        size_t at = s->used.load();
        while (at + need <= s->size) {
            if (s->used.compare_exchange_weak(at, at + need)) {
                *p = s->base + at;
                return cudaSuccess;
            }
        }
        // exhausted (the estimate was short): an allocation of its own
    }
    return cudaMalloc(p, bytes);
}
void dev_free(void *p) {
    if (!p) return;
    {
        std::lock_guard<std::mutex> g(g_slab_mutex);
        for (const DevSlab *s : g_slabs)
            if (static_cast<char *>(p) >= s->base && static_cast<char *>(p) < s->base + s->size) return;
    }
    cudaFree(p);
}
void *thread_scratch(size_t bytes) {
    if (bytes <= t_scratch_bytes) return t_scratch;
    if (t_scratch) cudaFree(t_scratch);
    t_scratch = nullptr;
    t_scratch_bytes = 0;
    if (cudaMalloc(&t_scratch, bytes) != cudaSuccess) {
        cudaGetLastError();
        t_scratch = nullptr;
        return nullptr;
    }
    t_scratch_bytes = bytes;
    return t_scratch;
}
void release_thread_scratch() {
    if (t_scratch) cudaFree(t_scratch);
    t_scratch = nullptr;
    t_scratch_bytes = 0;
}
}  // namespace sparsh

extern "C" {

const char *sparsh_last_error(void) { return g_err.c_str(); }

int sparsh_init(int device) {
    Context &c = ctx();
    if (c.ready && c.device == device) return SPARSH_OK;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        // no CPU fallback by design: the product path fails loudly without a GPU
        set_error("sparsh_b200: no CUDA device available (this library has no CPU fallback)");
        cudaGetLastError();
        return SPARSH_ERR_NO_DEVICE;
    }
    SP_REQUIRE(device >= 0 && device < ndev, "invalid device ordinal");
    SP_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    SP_CUDA(cudaGetDeviceProperties(&prop, device));
    c.device = device;
    c.sm_count = prop.multiProcessorCount;
    if (!c.own_stream) SP_CUDA(cudaStreamCreateWithFlags(&c.own_stream, cudaStreamNonBlocking));
    c.stream = c.own_stream;
    if (!c.partials) SP_CUDA(cudaMalloc(&c.partials, sizeof(double) * (size_t)RED_MAX_BLOCKS * RED_MAX_VALUES));
    if (!c.ticket) {
        SP_CUDA(cudaMalloc(&c.ticket, sizeof(unsigned int) * 4));
        SP_CUDA(cudaMemset(c.ticket, 0, sizeof(unsigned int) * 4));
    }
    if (!c.d_scalar) SP_CUDA(cudaMalloc(&c.d_scalar, sizeof(double) * 16));
    if (!c.h_scalar) SP_CUDA(cudaMallocHost(&c.h_scalar, sizeof(double) * 16));
    c.ready = true;
    return SPARSH_OK;
}

int sparsh_shutdown(void) {
    Context &c = ctx();
    if (!c.ready) return SPARSH_OK;
    cudaStreamSynchronize(c.stream);
    cudaFree(c.partials);
    cudaFree(c.ticket);
    cudaFree(c.d_scalar);
    cudaFreeHost(c.h_scalar);
    cudaStreamDestroy(c.own_stream);
    c = Context();
    return SPARSH_OK;
}

int sparsh_set_stream(void *s) {
    SP_TRY(ensure_init());
    Context &c = ctx();
    c.stream = s ? (cudaStream_t)s : c.own_stream;
    return SPARSH_OK;
}
int sparsh_get_stream(void **s) {
    SP_TRY(ensure_init());
    *s = (void *)ctx().stream;
    return SPARSH_OK;
}
int sparsh_sync(void) {
    SP_TRY(ensure_init());
    SP_CUDA(cudaStreamSynchronize(ctx().stream));
    return SPARSH_OK;
}
int sparsh_device_name(char *buf, size_t len, int *sm_count) {
    SP_TRY(ensure_init());
    cudaDeviceProp prop;
    SP_CUDA(cudaGetDeviceProperties(&prop, ctx().device));
    if (buf && len) {
        strncpy(buf, prop.name, len - 1);
        buf[len - 1] = 0;
    }
    if (sm_count) *sm_count = prop.multiProcessorCount;
    return SPARSH_OK;
}
long long sparsh_launch_count(void) { return ctx().launches; }
void sparsh_launch_count_reset(void) { ctx().launches = 0; }
void sparsh_launch_count_add(long long kernels) { ctx().launches += kernels; }

int sparsh_malloc(size_t bytes, void **d_ptr) {
    SP_TRY(ensure_init());
    SP_CUDA(cudaMalloc(d_ptr, bytes ? bytes : 8));
    return SPARSH_OK;
}
int sparsh_free(void *d_ptr) {
    if (d_ptr) SP_CUDA(cudaFree(d_ptr));
    return SPARSH_OK;
}
int sparsh_host_alloc(size_t bytes, void **h_ptr) {
    SP_TRY(ensure_init());
    SP_CUDA(cudaMallocHost(h_ptr, bytes ? bytes : 8));
    return SPARSH_OK;
}
int sparsh_host_free(void *h_ptr) {
    if (h_ptr) SP_CUDA(cudaFreeHost(h_ptr));
    return SPARSH_OK;
}
int sparsh_memcpy_h2d(void *d_dst, const void *h_src, size_t bytes) {
    SP_TRY(ensure_init());
    SP_CUDA(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, ctx().stream));
    SP_CUDA(cudaStreamSynchronize(ctx().stream));
    return SPARSH_OK;
}
int sparsh_memcpy_d2h(void *h_dst, const void *d_src, size_t bytes) {
    SP_TRY(ensure_init());
    SP_CUDA(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, ctx().stream));
    SP_CUDA(cudaStreamSynchronize(ctx().stream));
    return SPARSH_OK;
}
int sparsh_memcpy_d2d(void *d_dst, const void *d_src, size_t bytes) {
    SP_TRY(ensure_init());
    SP_CUDA(cudaMemcpyAsync(d_dst, d_src, bytes, cudaMemcpyDeviceToDevice, ctx().stream));
    return SPARSH_OK;
}
int sparsh_fill(double *d_x, size_t n, double value) {
    SP_TRY(ensure_init());
    return k_fill(d_x, n, value);
}

// ---- BLAS-1 -------------------------------------------------------------------------------------------------
static int fetch_scalar(int idx, double *h_out) {
    Context &c = ctx();
    SP_CUDA(cudaMemcpyAsync(c.h_scalar + idx, c.d_scalar + idx, sizeof(double), cudaMemcpyDeviceToHost, c.stream));
    SP_CUDA(cudaStreamSynchronize(c.stream));
    *h_out = c.h_scalar[idx];
    return SPARSH_OK;
}

int sparsh_dot(size_t n, const double *d_x, const double *d_y, double *h_out) {
    SP_TRY(ensure_init());
    SP_TRY(k_dot(n, d_x, d_y, ctx().d_scalar));
    return fetch_scalar(0, h_out);
}
int sparsh_dot_device(size_t n, const double *d_x, const double *d_y, double *d_out) {
    SP_TRY(ensure_init());
    SP_REQUIRE(d_out != nullptr, "d_out is NULL");
    return k_dot(n, d_x, d_y, d_out);
}
int sparsh_nrm2(size_t n, const double *d_x, double *h_out) {
    SP_TRY(ensure_init());
    SP_TRY(k_dot(n, d_x, d_x, ctx().d_scalar));
    double s = 0.0;
    SP_TRY(fetch_scalar(0, &s));
    *h_out = std::sqrt(s);
    return SPARSH_OK;
}
int sparsh_axpy(size_t n, double a, const double *d_x, double *d_y) {
    SP_TRY(ensure_init());
    return k_axpy(n, a, d_x, d_y);
}
int sparsh_axpby(size_t n, double a, const double *d_x, double b, double *d_y) {
    SP_TRY(ensure_init());
    return k_axpby(n, a, d_x, b, d_y);
}
int sparsh_axpbypcz(size_t n, double a, const double *d_x, double b, const double *d_y, double c, double *d_z) {
    SP_TRY(ensure_init());
    return k_axpbypcz(n, a, d_x, b, d_y, c, d_z);
}

}  // extern "C"

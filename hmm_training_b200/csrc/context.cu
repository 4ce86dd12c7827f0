// Context, error reporting, caching allocator and phase timers of libhmmb200.
#include <cstdlib>
#ifdef _OPENMP
#include <omp.h>
#endif

#include "common.cuh"

namespace hmmb {

static thread_local char g_err[1024] = "";
static Ctx g_ctx;

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char *what, const char *file, int line) {
    set_error("CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e), file, line, what);
    return e == cudaErrorMemoryAllocation ? HMMB_ERR_OOM : HMMB_ERR_CUDA;
}

Ctx &ctx() { return g_ctx; }

int require_init() {
    if (g_ctx.inited) return HMMB_OK;
    return hmmb_init(-1);
}

int dev_alloc(void **p, size_t bytes) {
    Ctx &c = g_ctx;
    if (bytes == 0) bytes = 256;
    bytes = (bytes + 255) & ~size_t(255);
    auto it = c.free_blocks.lower_bound(bytes);
    if (it != c.free_blocks.end() && it->first <= bytes + bytes / 4 + (1 << 20)) {
        *p = it->second;
        c.live_blocks[*p] = it->first;
        c.free_blocks.erase(it);
        return HMMB_OK;
    }
    cudaError_t e = cudaMalloc(p, bytes);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        dev_release_cache();
        e = cudaMalloc(p, bytes);
    }
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        set_error("device allocation of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
        *p = nullptr;
        return HMMB_ERR_OOM;
    }
    c.live_blocks[*p] = bytes;
    return HMMB_OK;
}

void dev_free(void *p) {
    if (!p) return;
    Ctx &c = g_ctx;
    auto it = c.live_blocks.find(p);
    if (it == c.live_blocks.end()) return;
    c.free_blocks.insert({it->second, p});
    c.live_blocks.erase(it);
}

void dev_release_cache() {
    Ctx &c = g_ctx;
    if (c.stream) cudaStreamSynchronize(c.stream);
    for (auto &kv : c.free_blocks) cudaFree(kv.second);
    c.free_blocks.clear();
}

int phase_id(const char *name) {
    Ctx &c = g_ctx;
    for (size_t i = 0; i < c.phase_names.size(); ++i)
        if (c.phase_names[i] == name) return (int)i;
    c.phase_names.push_back(name);
    c.phase_ms.push_back(0.0);
    c.phase_n.push_back(0);
    return (int)c.phase_names.size() - 1;
}

static cudaEvent_t get_event() {
    Ctx &c = g_ctx;
    if (!c.event_pool.empty()) {
        cudaEvent_t e = c.event_pool.back();
        c.event_pool.pop_back();
        return e;
    }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}

cudaEvent_t event_get() { return get_event(); }
void event_put(cudaEvent_t e) { g_ctx.event_pool.push_back(e); }

bool host_is_pinned(const void *p) {
    cudaPointerAttributes attr;
    const bool pinned = cudaPointerGetAttributes(&attr, p) == cudaSuccess &&
                        (attr.type == cudaMemoryTypeHost || attr.type == cudaMemoryTypeManaged);
    (void)cudaGetLastError();
    return pinned;
}

void par_memcpy(void *dst, const void *src, size_t bytes) {
#ifdef _OPENMP
    const int nt = bytes >= (size_t(1) << 20) ? omp_get_max_threads() : 1;
#else
    const int nt = 1;
#endif
    if (nt <= 1) {
        memcpy(dst, src, bytes);
        return;
    }
    const size_t slice = ((bytes + nt - 1) / nt + 4095) & ~size_t(4095);
#pragma omp parallel for schedule(static) num_threads(nt)
    for (int t = 0; t < nt; ++t) {
        const size_t lo = std::min(bytes, slice * t), hi = std::min(bytes, lo + slice);
        if (hi > lo) memcpy((char *)dst + lo, (const char *)src + lo, hi - lo);
    }
}

static constexpr size_t BOUNCE_BYTES = size_t(8) << 20;
static constexpr size_t BIG_COPY_MIN = size_t(4) << 20;

static int bounce_ready() {
    Ctx &c = g_ctx;
    for (int b = 0; b < 2; ++b) {
        if (!c.bounce[b]) {
            if (cudaHostAlloc(&c.bounce[b], BOUNCE_BYTES, cudaHostAllocDefault) != cudaSuccess) {
                (void)cudaGetLastError();
                c.bounce[b] = nullptr;
                return HMMB_ERR_OOM;
            }
        }
        if (!c.bounce_ev[b]) HMMB_CUDA(cudaEventCreateWithFlags(&c.bounce_ev[b], cudaEventDisableTiming));
    }
    return HMMB_OK;
}

int h2d_big(void *dst, const void *src, size_t bytes, cudaStream_t st) {
    Ctx &c = g_ctx;
    if (bytes == 0) return HMMB_OK;
    if (bytes < BIG_COPY_MIN || getenv("HMMB_NO_BOUNCE") || host_is_pinned(src) || bounce_ready() != HMMB_OK) {
        HMMB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
        return HMMB_OK;
    }
    int k = 0;
    for (size_t lo = 0; lo < bytes; lo += BOUNCE_BYTES, ++k) {
        const size_t n = std::min(BOUNCE_BYTES, bytes - lo);
        const int b = k & 1;
        HMMB_CUDA(cudaEventSynchronize(c.bounce_ev[b]));  // the DMA that last read this buffer (never recorded: returns at once)
        par_memcpy(c.bounce[b], (const char *)src + lo, n);
        HMMB_CUDA(cudaMemcpyAsync((char *)dst + lo, c.bounce[b], n, cudaMemcpyHostToDevice, st));
        HMMB_CUDA(cudaEventRecord(c.bounce_ev[b], st));
    }
    return HMMB_OK;
}

int d2h_big(void *dst, const void *src, size_t bytes, cudaStream_t st) {
    Ctx &c = g_ctx;
    if (bytes == 0) return HMMB_OK;
    if (bytes < BIG_COPY_MIN || getenv("HMMB_NO_BOUNCE") || host_is_pinned(dst) || bounce_ready() != HMMB_OK) {
        HMMB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st));
        HMMB_CUDA(cudaStreamSynchronize(st));
        return HMMB_OK;
    }
    // both buffers may still be the source of an earlier h2d_big on another stream
    for (int b = 0; b < 2; ++b) HMMB_CUDA(cudaEventSynchronize(c.bounce_ev[b]));
    const size_t nchunk = (bytes + BOUNCE_BYTES - 1) / BOUNCE_BYTES;
    auto issue = [&](size_t k) -> int {
        const size_t lo = k * BOUNCE_BYTES, n = std::min(BOUNCE_BYTES, bytes - lo);
        HMMB_CUDA(cudaMemcpyAsync(c.bounce[k & 1], (const char *)src + lo, n, cudaMemcpyDeviceToHost, st));
        HMMB_CUDA(cudaEventRecord(c.bounce_ev[k & 1], st));
        return HMMB_OK;
    };
    auto drain = [&](size_t k) -> int {
        const size_t lo = k * BOUNCE_BYTES, n = std::min(BOUNCE_BYTES, bytes - lo);
        HMMB_CUDA(cudaEventSynchronize(c.bounce_ev[k & 1]));
        par_memcpy((char *)dst + lo, c.bounce[k & 1], n);
        return HMMB_OK;
    };
    HMMB_TRY(issue(0));
    for (size_t k = 1; k < nchunk; ++k) {
        HMMB_TRY(issue(k));      // chunk k crosses PCIe while chunk k - 1 is copied out of its buffer
        HMMB_TRY(drain(k - 1));
    }
    HMMB_TRY(drain(nchunk - 1));
    return HMMB_OK;
}

void phase_begin(int id) {
    Ctx &c = g_ctx;
    PhaseRec r;
    r.phase = id;
    r.a = get_event();
    r.b = get_event();
    cudaEventRecord(r.a, c.stream);
    c.pending.push_back(r);
}

void phase_end(int id) {
    Ctx &c = g_ctx;
    (void)id;
    cudaEventRecord(c.pending.back().b, c.stream);
    if (c.pending.size() > 4096) phase_collect();
}

int phase_collect() {
    Ctx &c = g_ctx;
    if (c.pending.empty()) return HMMB_OK;
    HMMB_CUDA(cudaStreamSynchronize(c.stream));
    for (auto &r : c.pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) {
            c.phase_ms[r.phase] += ms;
            c.phase_n[r.phase] += 1;
        }
        c.event_pool.push_back(r.a);
        c.event_pool.push_back(r.b);
    }
    c.pending.clear();
    return HMMB_OK;
}

}  // namespace hmmb

using namespace hmmb;

// Arithmetic peak of this GPU for the roofline of the compute-bound kernels (VQ prefilter: fp32 FFMA; exact
// distances and the scorer: fp64 DFMA): eight independent FMA chains per thread, nothing else in the loop.
template <typename T>
__global__ void __launch_bounds__(256) k_fma_probe(T *__restrict__ out, int iters, T seed) {
    T a[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) a[u] = seed + (T)(threadIdx.x + u);
    const T b = (T)0.999999, c = (T)1e-7;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) a[u] = a[u] * b + c;  // contracted to one FMA
    }
    T s = 0;
#pragma unroll
    for (int u = 0; u < 8; ++u) s += a[u];
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

template <typename T>
static int fma_probe(double *tflops) {
    hmmb::Ctx &c = hmmb::ctx();
    const int grid = c.sm_count * 8, iters = sizeof(T) == 8 ? 4096 : 16384;
    T *buf = nullptr;
    HMMB_TRY(hmmb::dev_alloc_t(&buf, (size_t)grid * 256));
    cudaEvent_t e0 = hmmb::event_get(), e1 = hmmb::event_get();
    double best_ms = 1e30;
    for (int rep = 0; rep < 4; ++rep) {  // first launch = warm-up
        HMMB_CUDA(cudaEventRecord(e0, c.stream));
        HMMB_LAUNCH("peak_probe", k_fma_probe<T>, grid, 256, 0, buf, iters, (T)1);
        HMMB_CUDA(cudaEventRecord(e1, c.stream));
        HMMB_CUDA(cudaEventSynchronize(e1));
        float ms = 0.f;
        HMMB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        if (rep > 0 && ms < best_ms) best_ms = ms;
    }
    hmmb::event_put(e0);
    hmmb::event_put(e1);
    hmmb::dev_free(buf);
    *tflops = 2.0 * grid * 256.0 * 8.0 * iters / (best_ms * 1e-3) / 1e12;
    return HMMB_OK;
}

extern "C" {

int hmmb_init(int device) {
    Ctx &c = ctx();
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        (void)cudaGetLastError();
        set_error("no CUDA device available (%s); libhmmb200 has no CPU fallback",
                  e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        return HMMB_ERR_CUDA;
    }
    if (device < 0) {
        if (c.inited) return HMMB_OK;
        if (cudaGetDevice(&device) != cudaSuccess) device = 0;
    }
    if (device >= count) {
        set_error("device %d out of range (%d devices)", device, count);
        return HMMB_ERR_ARG;
    }
    if (c.inited && c.device == device) return HMMB_OK;
    if (c.inited) hmmb_shutdown();
    HMMB_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    HMMB_CUDA(cudaGetDeviceProperties(&prop, device));
    c.device = device;
    c.sm_count = prop.multiProcessorCount;
    c.cc_major = prop.major;
    c.cc_minor = prop.minor;
    c.smem_optin = prop.sharedMemPerBlockOptin;
    c.global_mem = (int64_t)prop.totalGlobalMem;
    HMMB_CUDA(cudaStreamCreateWithFlags(&c.own_stream, cudaStreamNonBlocking));
    c.stream = c.own_stream;
    HMMB_CUDA(cudaStreamCreateWithFlags(&c.copy_stream, cudaStreamNonBlocking));
    HMMB_CUDA(cudaStreamCreateWithFlags(&c.d2h_stream, cudaStreamNonBlocking));
    for (auto &st : c.stage_stream) HMMB_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
#ifdef _OPENMP
    // launchers such as torchrun export OMP_NUM_THREADS=1; the host-side blocking of a build is a handful of
    // memory-bound loops that still gain from a few threads per rank
    if (const char *t = getenv("HMMB_HOST_THREADS")) {
        const int n = atoi(t);
        if (n > 0) omp_set_num_threads(n);
    }
#endif
    c.inited = true;
    return HMMB_OK;
}

int hmmb_shutdown(void) {
    Ctx &c = ctx();
    if (!c.inited) return HMMB_OK;
    cudaSetDevice(c.device);
    phase_collect();
    dev_release_cache();
    for (auto &kv : c.live_blocks) cudaFree(kv.first);
    c.live_blocks.clear();
    if (c.stage) cudaFreeHost(c.stage);
    c.stage = nullptr;
    c.stage_bytes = 0;
    if (c.pstage) cudaFreeHost(c.pstage);
    c.pstage = nullptr;
    c.pstage_bytes = 0;
    for (int b = 0; b < 2; ++b) {
        if (c.bounce[b]) cudaFreeHost(c.bounce[b]);
        if (c.bounce_ev[b]) cudaEventDestroy(c.bounce_ev[b]);
        c.bounce[b] = nullptr;
        c.bounce_ev[b] = nullptr;
    }
    if (c.stage_busy) { cudaEventDestroy(c.stage_busy); c.stage_busy = nullptr; }
    if (c.pstage_busy) { cudaEventDestroy(c.pstage_busy); c.pstage_busy = nullptr; }
    for (auto ev : c.event_pool) cudaEventDestroy(ev);
    c.event_pool.clear();
    if (c.own_stream) cudaStreamDestroy(c.own_stream);
    if (c.copy_stream) cudaStreamDestroy(c.copy_stream);
    if (c.d2h_stream) cudaStreamDestroy(c.d2h_stream);
    for (auto &st : c.stage_stream) {
        if (st) cudaStreamDestroy(st);
        st = nullptr;
    }
    c.own_stream = c.stream = c.copy_stream = c.d2h_stream = nullptr;
    c.inited = false;
    return HMMB_OK;
}

const char *hmmb_last_error(void) { return g_err; }

const char *hmmb_version(void) { return "hmmb200 0.2 (sm_100a)"; }

int hmmb_device_info(int *sm_count, int *cc_major, int *cc_minor, int64_t *global_mem_bytes) {
    HMMB_TRY(require_init());
    Ctx &c = ctx();
    if (sm_count) *sm_count = c.sm_count;
    if (cc_major) *cc_major = c.cc_major;
    if (cc_minor) *cc_minor = c.cc_minor;
    if (global_mem_bytes) *global_mem_bytes = c.global_mem;
    return HMMB_OK;
}

int hmmb_set_stream(void *cuda_stream) {
    HMMB_TRY(require_init());
    Ctx &c = ctx();
    phase_collect();
    cudaStream_t next = cuda_stream ? (cudaStream_t)cuda_stream : c.own_stream;
    if (next != c.stream) {
        // A call may return with kernels still queued on the old stream (hmmb_vq_encode_dev) whose device blocks the
        // allocator already hands out again: the new stream starts behind everything queued on the old one.
        cudaEvent_t e = event_get();
        HMMB_CUDA(cudaEventRecord(e, c.stream));
        HMMB_CUDA(cudaStreamWaitEvent(next, e, 0));
        event_put(e);
    }
    c.stream = next;
    return HMMB_OK;
}

void *hmmb_get_stream(void) {
    if (require_init() != HMMB_OK) return nullptr;
    return (void *)ctx().stream;
}

int hmmb_synchronize(void) {
    HMMB_TRY(require_init());
    HMMB_CUDA(cudaStreamSynchronize(ctx().stream));
    return HMMB_OK;
}

void *hmmb_host_alloc(int64_t bytes) {
    if (require_init() != HMMB_OK) return nullptr;
    void *p = nullptr;
    if (cudaHostAlloc(&p, (size_t)(bytes > 0 ? bytes : 1), cudaHostAllocDefault) != cudaSuccess) {
        (void)cudaGetLastError();
        set_error("pinned host allocation of %lld bytes failed", (long long)bytes);
        return nullptr;
    }
    return p;
}

int hmmb_host_free(void *p) {
    if (!p) return HMMB_OK;
    HMMB_CUDA(cudaFreeHost(p));
    return HMMB_OK;
}

int64_t hmmb_launch_count(void) { return ctx().launches; }

double hmmb_phase_ms(const char *phase, int64_t *launches) {
    Ctx &c = ctx();
    if (!c.inited) return -1.0;
    phase_collect();
    for (size_t i = 0; i < c.phase_names.size(); ++i)
        if (c.phase_names[i] == phase) {
            if (launches) *launches = c.phase_n[i];
            return c.phase_n[i] ? c.phase_ms[i] : -1.0;
        }
    if (launches) *launches = 0;
    return -1.0;
}

int hmmb_phase_reset(void) {
    Ctx &c = ctx();
    if (!c.inited) return HMMB_OK;
    phase_collect();
    for (size_t i = 0; i < c.phase_ms.size(); ++i) {
        c.phase_ms[i] = 0.0;
        c.phase_n[i] = 0;
    }
    return HMMB_OK;
}

int hmmb_peak_probe(int what, double *tflops) {
    HMMB_TRY(require_init());
    if (!tflops || (what != 0 && what != 1)) { set_error("hmmb_peak_probe: what must be 0 (fp64) or 1 (fp32)"); return HMMB_ERR_ARG; }
    return what == 0 ? fma_probe<double>(tflops) : fma_probe<float>(tflops);
}

int hmmb_set_profiling(int enabled) {
    HMMB_TRY(require_init());
    phase_collect();
    ctx().profiling = enabled != 0;
    return HMMB_OK;
}

}  // extern "C"

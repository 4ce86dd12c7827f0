// Shared host/device plumbing for libhmmb200: context, error handling, caching device
// allocator, per-phase CUDA-event timing and the launch helper every kernel goes through.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <cmath>
#include <functional>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/hmmb200.h"

namespace hmmb {

// ---------------------------------------------------------------- errors
void set_error(const char *fmt, ...);
int cuda_fail(cudaError_t e, const char *what, const char *file, int line);

#define HMMB_CUDA(expr)                                                        \
    do {                                                                       \
        cudaError_t _e = (expr);                                               \
        if (_e != cudaSuccess) return ::hmmb::cuda_fail(_e, #expr, __FILE__, __LINE__); \
    } while (0)

#define HMMB_TRY(expr)                 \
    do {                               \
        int _rc = (expr);              \
        if (_rc != HMMB_OK) return _rc; \
    } while (0)

// ---------------------------------------------------------------- context
struct PhaseRec {
    int phase;
    cudaEvent_t a, b;
};

struct Ctx {
    bool inited = false;
    int device = -1;
    int sm_count = 0;
    int cc_major = 0, cc_minor = 0;
    size_t smem_optin = 0;
    int64_t global_mem = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;  // H2D of raw codewords, overlapped with host prep and repack
    std::vector<int32_t> len_scratch;    // per-sequence lengths of the build in progress (host)
    cudaStream_t d2h_stream = nullptr;   // results leaving while later stages still compute (pipelined scorer)
    cudaStream_t stage_stream[2] = {nullptr, nullptr};  // pipelined first E-step: stages alternate between these
    bool h2d_on_copy = false;            // small H2D copies of the running build go through copy_stream too
    std::function<int(int, int)> after_chunk;  // (chunk, nchunk): called after a codeword chunk has been queued on copy_stream
    int64_t launches = 0;
    bool profiling = false;
    std::vector<std::string> phase_names;
    std::vector<double> phase_ms;
    std::vector<int64_t> phase_n;
    std::vector<PhaseRec> pending;
    std::vector<cudaEvent_t> event_pool;
    // caching allocator
    std::multimap<size_t, void *> free_blocks;
    std::map<void *, size_t> live_blocks;
    // pinned host staging buffer (per-sequence metadata of the last build)
    void *stage = nullptr;
    size_t stage_bytes = 0;
    cudaEvent_t stage_busy = nullptr;   // recorded after the last copy out of `stage`
    // pinned staging of the initial parameters of a pipelined create
    void *pstage = nullptr;
    size_t pstage_bytes = 0;
    cudaEvent_t pstage_busy = nullptr;
    // two pinned bounce buffers for large copies from / to PAGEABLE host memory (h2d_big / d2h_big)
    void *bounce[2] = {nullptr, nullptr};
    cudaEvent_t bounce_ev[2] = {nullptr, nullptr};
    // device slot of hmmb_score, cleared by one memset per call: the precision guard's flag (int32 at [0]) and the
    // count of pairs k_score_exact recomputed (int64 at [2]), read only by hmmb_score_diagnostics
    int32_t *score_slot = nullptr;
};

Ctx &ctx();
int require_init();

int dev_alloc(void **p, size_t bytes);  // cached cudaMalloc (256 B granularity)
void dev_free(void *p);                 // returns the block to the cache
void dev_release_cache();

// Large copies between pageable host memory and the device: the driver's own staging moves ~10 GB/s; these go
// through two pinned bounce buffers with a multi-threaded memcpy of one chunk overlapping the DMA of the other.
// Pinned (or small) buffers take a plain cudaMemcpyAsync.  h2d_big returns when `src` may be reused (the last DMA
// may still be in flight on `st`); d2h_big returns with `dst` complete (it synchronises `st`).
bool host_is_pinned(const void *p);
void par_memcpy(void *dst, const void *src, size_t bytes);
int h2d_big(void *dst, const void *src, size_t bytes, cudaStream_t st);
int d2h_big(void *dst, const void *src, size_t bytes, cudaStream_t st);

int phase_id(const char *name);
void phase_begin(int id);
void phase_end(int id);
int phase_collect();  // synchronises and folds pending event pairs into phase_ms
cudaEvent_t event_get();          // pooled events (no timing semantics implied)
void event_put(cudaEvent_t e);

template <typename T>
inline int dev_alloc_t(T **p, size_t n) {
    return dev_alloc(reinterpret_cast<void **>(p), n * sizeof(T));
}

// Launch helper: counts the launch, optional event timing, checks the launch error.
#define HMMB_LAUNCH(phase_name, kernel, grid, block, smem, ...)                                  \
    do {                                                                                         \
        ::hmmb::Ctx &_c = ::hmmb::ctx();                                                         \
        static int _pid = -1;                                                                    \
        if (_pid < 0) _pid = ::hmmb::phase_id(phase_name);                                       \
        if (_c.profiling) ::hmmb::phase_begin(_pid);                                             \
        kernel<<<(grid), (block), (smem), _c.stream>>>(__VA_ARGS__);                             \
        if (_c.profiling) ::hmmb::phase_end(_pid);                                               \
        _c.launches++;                                                                           \
        cudaError_t _le = cudaGetLastError();                                                    \
        if (_le != cudaSuccess) return ::hmmb::cuda_fail(_le, #kernel, __FILE__, __LINE__);      \
    } while (0)

// ---------------------------------------------------------------- device helpers
#ifdef __CUDACC__
// Smallest positive double: the clamp that keeps "value > 0  <=>  structurally reachable"
// when a product of positive factors underflows (SURVEY.md §7.3 hard part 1).
__device__ __forceinline__ double tiny_pos() { return __longlong_as_double(1LL); }
__device__ __forceinline__ double neg_inf() { return __longlong_as_double(0xfff0000000000000LL); }
__device__ __forceinline__ double pos_inf() { return __longlong_as_double(0x7ff0000000000000LL); }

// Exact power-of-two rescale: returns 2^(1023 - ex) where ex is the biased exponent of s
// (s > 0), and adds the applied shift (ex - 1023) to esum.  Multiplying by it is exact.
__device__ __forceinline__ double pow2_rescale(double s, long long &esum) {
    int ex = (__double2hiint(s) >> 20) & 0x7ff;
    esum += (long long)(ex - 1023);
    return __hiloint2double((2046 - ex) << 20, 0);
}
__device__ __forceinline__ double pow2_rescale_noacc(double s) {
    int ex = (__double2hiint(s) >> 20) & 0x7ff;
    return __hiloint2double((2046 - ex) << 20, 0);
}
// true if the (non-negative) double is zero or a very small denormal: cheap integer test
// used to enter the exact slow paths.
__device__ __forceinline__ bool maybe_zero(double x) { return __double2hiint(x) == 0; }
#endif

}  // namespace hmmb

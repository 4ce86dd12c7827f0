// Host side of the Baum-Welch trainer, the forward scorer and the Viterbi decoder: sequence sorting/blocking,
// device layout, the EM loop, and the C ABI declared in include/hmmb200.h.
#include <algorithm>
#include <cstdlib>
#include <functional>
#include <memory>
#include <numeric>
#include <type_traits>

#include "bw_kernels.cuh"
#include "bwltr_kernels.cuh"
#include "viterbi_kernels.cuh"
#include "words_kernels.cuh"

namespace hmmb {

// ---------------------------------------------------------------- small kernels local to this TU
// B0 [W][N][M] (linear) -> Bt [W][M][N]; non-positive / NaN entries become structural zeros,
// which is what safe_log does to them (HMM/hmm_training.py:46-54, :323-325).
__global__ void k_load_B(const double *__restrict__ B, int N, int M, double *__restrict__ Bt,
                         int32_t *__restrict__ b_has_zero) {
    const size_t w = blockIdx.y;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < N * M; e += gridDim.x * blockDim.x) {
        const int k = e / N, j = e - k * N;
        const double v = B[(w * N + j) * M + k];
        Bt[w * (size_t)M * N + e] = v > 0.0 ? v : 0.0;
        if (!(v > 0.0) && b_has_zero) b_has_zero[w] = 1;  // benign race: every writer stores 1
    }
}
__global__ void k_load_clamped(const double *__restrict__ src, int64_t n, double *__restrict__ dst) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const double v = src[e];
        dst[e] = v > 0.0 ? v : 0.0;
    }
}
__global__ void k_fill(double *p, int64_t n, double v) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) p[e] = v;
}
// Per-sequence metadata that follows from the block table of the blocked layouts (uint4 row of the lane, word,
// identity order): filled on the device instead of crossing PCIe (16 of the 28 bytes per sequence).
__global__ void k_meta_blocked(const Blk *__restrict__ blks, int nblk, int64_t *__restrict__ foff, int32_t *__restrict__ word,
                               int32_t *__restrict__ order) {
    const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    for (int b = blockIdx.x * wpb + (threadIdx.x >> 5); b < nblk; b += gridDim.x * wpb) {
        const Blk k = blks[b];
        if (lane < k.nseq) {
            const int64_t i = (int64_t)k.first + lane;
            foff[i] = k.obs_base + lane;
            word[i] = k.word;
            if (order) order[i] = (int32_t)i;
        }
    }
}
__global__ void k_fill_i32(int32_t *p, int64_t n, int32_t v) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) p[e] = v;
}

// ---------------------------------------------------------------- scoring kernels
// VECB: per-state error bound of the forward recursion (needed for utterances of thousands of frames); the scalar
// bound is ~10 instructions per step cheaper and enough below SCORE4_SCALAR_BOUND_MAX_T frames (bw4_kernels.cuh)
constexpr int SCORE4_SCALAR_BOUND_MAX_T = 1000;
template <bool BIDIAG, bool VECB>
__global__ void __launch_bounds__(BW_THREADS)
k_score4(const Blk *__restrict__ blks, int nblk, int blocks_per_cta, const uint4 *__restrict__ obs_blk,
         const int32_t *__restrict__ len_sorted, const int32_t *__restrict__ order, const double *__restrict__ pi,
         const double *__restrict__ A, const double *__restrict__ Bt, int M, int W, double *__restrict__ ll_out,
         int32_t *__restrict__ any_nan) {
    extern __shared__ double sB[];
    double *sBmax = sB + (size_t)M * 4;
    unsigned char *sBmask = reinterpret_cast<unsigned char *>(sBmax + M);
    const int w = blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double a[BIDIAG ? 7 : 16], p[4], rmax;
    Masks4 mk;
    load_model4<BIDIAG>(pi, A, Bt, w, M, sB, sBmax, sBmask, a, p, rmax, mk);
    __syncthreads();
    const int b0 = blockIdx.x * blocks_per_cta;
    const int b1 = min(nblk, b0 + blocks_per_cta);
    for (int b = b0 + warp; b < b1; b += BW_WARPS) {
        const Blk bk = blks[b];
        const int T = lane < bk.nseq ? len_sorted[bk.first + lane] : 0;
        bool af;
        const double ll = fwd4_run<BIDIAG, false, VECB>(T, bk.tmax, obs_blk + bk.obs_base + lane, reinterpret_cast<const double2 *>(sB),
                                                  reinterpret_cast<const double2 *>(sB) + M, sBmax, sBmask, a, p, rmax, mk, nullptr, af);
        if (lane < bk.nseq) {
            ll_out[(size_t)order[bk.first + lane] * W + w] = ll;
            if (ll != ll) *any_nan = 1;  // precision guard marked this pair: k_score_exact has work to do
        }
    }
}

// Scorer with the eightfold-replicated B^T (conflict-free gather, see fwd4_run) and the lean forward pass
// (score4_lean_run) for models that allow it; 8 warps per CTA, one model per CTA, M <= SCORE4R_MAX_M.
// Shared memory: [M * 8] double2 (b0, b1), [M * 8] double2 (b2, b3), [M] per-codeword max, [M] support masks.
constexpr int SCORE4R_WARPS = 8;
constexpr int SCORE4R_MIN_CTAS = 2;
constexpr int SCORE4R_REP = 8;
constexpr int SCORE4R_MAX_M = 256;  // 64 KB of replicated B^T: three CTAs per SM
template <bool BIDIAG, bool VECB>
__global__ void __launch_bounds__(SCORE4R_WARPS * 32, SCORE4R_MIN_CTAS)
k_score4r(const Blk *__restrict__ blks, int nblk, int blocks_per_cta, const uint4 *__restrict__ obs_blk,
          const int32_t *__restrict__ len_sorted, const int32_t *__restrict__ order, const double *__restrict__ pi,
          const double *__restrict__ A, const double *__restrict__ Bt, int M, int W, double *__restrict__ ll_out,
          int32_t *__restrict__ any_nan) {
    extern __shared__ double sB[];
    constexpr int REP = SCORE4R_REP, NT = SCORE4R_WARPS * 32;
    // fixed SCORE4R_MAX_M-entry layout whatever M is: the second table sits at a literal offset from the first
    double2 *sB01 = reinterpret_cast<double2 *>(sB), *sB23 = sB01 + (size_t)SCORE4R_MAX_M * REP;
    double *sBmax = reinterpret_cast<double *>(sB23 + (size_t)SCORE4R_MAX_M * REP);
    unsigned char *sBmask = reinterpret_cast<unsigned char *>(sBmax + M);
    const int w = blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int has_zero = 0;
    {
        const double2 *src = reinterpret_cast<const double2 *>(Bt + (size_t)w * M * 4);
        for (int e = tid; e < M * REP; e += NT) {
            const int sym = e / REP;
            const double2 x = __ldg(src + 2 * sym), y = __ldg(src + 2 * sym + 1);
            sB01[e] = x;
            sB23[e] = y;
            if (e % REP == 0) {
                sBmax[sym] = fmax(fmax(x.x, x.y), fmax(y.x, y.y));
                const unsigned char mb = (unsigned char)((x.x > 0.0 ? 1 : 0) | (x.y > 0.0 ? 2 : 0) | (y.x > 0.0 ? 4 : 0) | (y.y > 0.0 ? 8 : 0));
                sBmask[sym] = mb;
                has_zero |= (mb != 0xF);
            }
        }
    }
    double a[BIDIAG ? 7 : 16], p[4], rmax;
    Masks4 mk;
    load_Api4<BIDIAG>(pi, A, w, a, p, rmax, mk);
    const bool b_has_zero = __syncthreads_or(has_zero) != 0;
    // alive sets without emission zeros: m_0 = support of pi, m_t = lutF(m_t-1); lean from the first t with m_t = all
    int tstar = -1;
    {
        unsigned m = mk.pmask;
        for (int t = 0; t < 4 && tstar < 0; ++t) {
            if (m == 0xFu && lut4(mk.lutF, 0xFu) == 0xFu) tstar = t;
            m = lut4(mk.lutF, m);
        }
    }
    const bool lean_model = !b_has_zero && tstar >= 0;
    const int slot = lane & (REP - 1);
    const int b0 = blockIdx.x * blocks_per_cta;
    const int b1 = min(nblk, b0 + blocks_per_cta);
    for (int b = b0 + warp; b < b1; b += SCORE4R_WARPS) {
        const Blk bk = blks[b];
        const int T = lane < bk.nseq ? len_sorted[bk.first + lane] : 0;
        const uint4 *op = obs_blk + bk.obs_base + lane;
        double ll;
        bool redo = !lean_model;
        if (lean_model) {
            bool bad;
            ll = score4_lean_run<BIDIAG, REP>(T, bk.tmax, op, sB01 + slot, sB01 + slot + (size_t)SCORE4R_MAX_M * REP, a, p, mk, tstar, bad);
            redo = __any_sync(0xffffffffu, bad && T > 0);
            if (redo) {  // (rare) the marked lanes again, with the full structural / precision logic
                bool af;
                const double ll2 = fwd4_run<BIDIAG, false, VECB, REP>(bad ? T : 0, bk.tmax, op, sB01, sB23, sBmax, sBmask, a, p, rmax,
                                                                      mk, nullptr, af, slot);
                if (bad) ll = ll2;
            }
        } else {
            bool af;
            ll = fwd4_run<BIDIAG, false, VECB, REP>(T, bk.tmax, op, sB01, sB23, sBmax, sBmask, a, p, rmax, mk, nullptr, af, slot);
        }
        if (lane < bk.nseq) {
            ll_out[(size_t)order[bk.first + lane] * W + w] = ll;
            if (ll != ll) *any_nan = 1;  // precision guard marked this pair: k_score_exact has work to do
        }
    }
}

template <int NP, typename SymT>
__global__ void __launch_bounds__(BW_THREADS)
k_scoreG(const SymT *__restrict__ obs, const int64_t *__restrict__ off_sorted, const int32_t *__restrict__ len_sorted,
         const int32_t *__restrict__ order, int64_t U, int64_t per_group, int N, int M, int W,
         const double *__restrict__ pi, const double *__restrict__ A, const double *__restrict__ Bt,
         double *__restrict__ ll_out, int32_t *__restrict__ any_nan) {
    __shared__ __align__(16) double sStage[BW_WARPS][128];
    const int w = blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int GPW = 32 / NP;
    const int j = lane % NP, gbase = lane - j;
    const int64_t group = ((int64_t)blockIdx.x * BW_WARPS + warp) * GPW + lane / NP;
    double acol[NP];
#pragma unroll
    for (int i = 0; i < NP; ++i) acol[i] = (i < N && j < N) ? __ldg(A + ((size_t)w * N + i) * N + j) : 0.0;
    const double pj = j < N ? __ldg(pi + (size_t)w * N + j) : 0.0;
    for (int64_t k = 0; k < per_group; ++k) {
        const int64_t r = group * per_group + k;
        const int T = r < U ? len_sorted[r] : 0;
        const int Tw = warp_max_int(T);
        if (Tw == 0) continue;
        const SymT *o = obs + (T > 0 ? off_sorted[r] : 0);
        const double ll = fwdG_run<NP, SymT, false>(T, Tw, N, j, gbase, lane, o, Bt + (size_t)w * M * N, acol, pj,
                                                    nullptr, sStage[warp]);
        if (T > 0 && j == 0) {
            ll_out[(size_t)order[r] * W + w] = ll;
            if (ll != ll) *any_nan = 1;
        }
    }
}

// test_hmm's argmax (HMM/hmm_testing.py:143-153): strict '>' from -inf, first model wins.
__global__ void k_argmax_first(const double *__restrict__ ll, int64_t U, int W, int32_t *__restrict__ out) {
    const int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= U) return;
    double best = neg_inf();
    int bi = -1;
    for (int w = 0; w < W; ++w) {
        const double v = ll[(size_t)u * W + w];
        if (v > best) { best = v; bi = w; }
    }
    out[u] = bi;
}

// Exact recomputation of the (utterance, model) pairs the precision guard marked with NaN; n_pairs counts them.
template <typename SymT, bool BLOCKED>
__global__ void __launch_bounds__(BW_THREADS)
k_score_exact(const void *__restrict__ obs, const int64_t *__restrict__ base_sorted, const int32_t *__restrict__ len_sorted,
              const int32_t *__restrict__ order, int64_t U, int N, int M, int W, const double *__restrict__ pi,
              const double *__restrict__ A, const double *__restrict__ Bt, double *__restrict__ ll_out,
              const int32_t *__restrict__ any_nan, int64_t *__restrict__ n_pairs) {
    if (*any_nan == 0) return;  // the scorers marked nothing: no scan of the [U, W] matrix
    const int lane = threadIdx.x & 31;
    const int64_t gw = (int64_t)blockIdx.x * BW_WARPS + (threadIdx.x >> 5);
    const int64_t nw = (int64_t)gridDim.x * BW_WARPS;
    for (int64_t i = gw; i < U; i += nw) {
        double *row = ll_out + (size_t)order[i] * W;
        const int T = len_sorted[i];
        for (int w0 = 0; w0 < W; w0 += 32) {
            const double v = (w0 + lane < W) ? row[w0 + lane] : 0.0;
            unsigned m = __ballot_sync(0xffffffffu, v != v);
            while (m) {
                const int w = w0 + __ffs(m) - 1;
                m &= m - 1;
                const double *piw = pi + (size_t)w * N, *Aw = A + (size_t)w * N * N, *Btw = Bt + (size_t)w * M * N;
                double logP;
                if (BLOCKED) {
                    BlkObs<SymT> o{reinterpret_cast<const uint4 *>(obs) + base_sorted[i]};
                    logP = exact_forward(T, N, lane, o, piw, Aw, Btw, (double *)nullptr);
                } else {
                    LinObs<SymT> o{reinterpret_cast<const SymT *>(obs) + base_sorted[i]};
                    logP = exact_forward(T, N, lane, o, piw, Aw, Btw, (double *)nullptr);
                }
                if (lane == 0) {
                    row[w] = logP;
                    atomicAdd(reinterpret_cast<unsigned long long *>(n_pairs), 1ULL);
                }
                __syncwarp();
            }
        }
    }
}

// Raw codewords of a pinned host buffer are uploaded on the copy stream in a few chunks, started
// before the host-side sorting / blocking so that PCIe time hides it; when the input is already in
// sorted order a chunk's blocks are repacked as soon as the chunk has landed.
struct EarlyUpload {
    static constexpr int MAX_CHUNKS = 8;
    void *d_raw = nullptr;
    const char *src = nullptr;
    int nchunk = 0;                 // planned chunks
    int issued = 0;                 // chunks already queued on the copy stream
    size_t hi[MAX_CHUNKS] = {};     // end byte of each chunk
    cudaEvent_t ev[MAX_CHUNKS] = {};
    bool active() const { return nchunk > 0; }
    // queue chunks [issued, upto) on the copy stream.  The first chunks go out before the host-side
    // sorting / blocking (PCIe works while the host does), the rest only after the (small)
    // per-sequence metadata has been queued: copies of different streams share one DMA queue, and the
    // metadata must not wait behind the whole codeword stream.
    int issue(int upto) {
        Ctx &c = ctx();
        for (int k = issued; k < upto && k < nchunk; ++k) {
            const size_t lo = k == 0 ? 0 : hi[k - 1];
            HMMB_CUDA(cudaMemcpyAsync((char *)d_raw + lo, src + lo, hi[k] - lo, cudaMemcpyHostToDevice, c.copy_stream));
            HMMB_CUDA(cudaEventRecord(ev[k], c.copy_stream));
            issued = k + 1;
            if (c.after_chunk) HMMB_TRY(c.after_chunk(k, nchunk));
        }
        return HMMB_OK;
    }
    ~EarlyUpload() {
        if (nchunk > 0) cudaStreamSynchronize(ctx().copy_stream);
        for (int k = 0; k < nchunk; ++k) event_put(ev[k]);
        dev_free(d_raw);
    }
};

// Deferred prepare: the trainer may leave the repack of the uploaded chunks to its first E-step,
// which then runs stage by stage (repack -> forward -> backward of the CTAs whose codewords have
// landed) while the later chunks are still crossing PCIe.
struct PendingPrepare {
    static constexpr int MAX_STAGES = EarlyUpload::MAX_CHUNKS;  // the trainer runs one stage per chunk on alternating streams
    std::unique_ptr<EarlyUpload> up;
    int idx_bytes = 1;
    int nstage = 0;
    int ev_index[MAX_STAGES] = {};   // upload chunk whose event completes the stage
    int blk_end[MAX_STAGES] = {};    // blocks [.., blk_end) have all their codewords on the device after the stage
    int cta_end[MAX_STAGES] = {};    // CTA work items [.., cta_end) only touch those blocks
};

// Stages of the pipelined first E-step (N = 4 and left-to-right).  The tail of a fit call behind the last upload chunk
// is the last stage's repack + forward + backward, and a stage launches whole work items: with the resident iterations'
// list (two items per SM, one fat backward CTA each) a stage of config 3 kept a quarter of the SMs busy for the 1.5 ms one
// item takes, and more stages only made that worse (4 stages 6.1 ms per fit call, 8 stages 8.0).  With the finer list the
// staged E-step launches from (SeqSet::cta_begin_fine, about eight items per SM) the picture turns: 4 stages 5.75 ms,
// 8 stages 5.50.  Left-to-right kernels (config 4, 200 MB of codewords + 131 MB of parameters up): 2 stages 16.1 ms per
// fit call, 4 stages 14.0 - 14.6, 8 stages 13.85.
constexpr int PIPE_STAGES = 8;
static_assert(PIPE_STAGES <= PendingPrepare::MAX_STAGES, "one upload chunk per stage");
static int score_stages(bool want_ll) {
    // 1 M utterances x 10 models, pinned buffers, 2 / 3 / 4 / 6 / 8 stages: 5.11 / 4.66 / 4.50 / 4.35 / 4.41 ms with the
    // log-likelihood matrix going back stage by stage, 4.17 / 3.95 / 3.82 / 4.01 / 3.95 ms argmax only (the probe script
    // that swept this is in the history at commit 03a55a2)
    return want_ll ? 6 : 4;
}

// ---------------------------------------------------------------- sequence set (shared by BW and scoring)
// Device layout of a sequence set: blocks of 32 same-word sequences for the N = 4 kernels or for the left-to-right
// kernels (N = 8 / 16), or one codeword stream for the lanes-per-state kernels (any N)
enum Layout { LAYOUT_LANES, LAYOUT_N4, LAYOUT_LTR };

struct SeqSet {
    int64_t R = 0, frames = 0;
    int N = 0, M = 0, NP = 0, sym_bytes = 1;
    Layout layout = LAYOUT_LANES;
    bool blocked() const { return layout != LAYOUT_LANES; }
    std::vector<int32_t> order;       // sorted -> original
    std::vector<int64_t> seq_begin;   // per word [W+1] (sorted order)
    std::vector<int32_t> cta_begin;   // per word [W+1]
    int nblk = 0, ncta = 0;
    // N = 4, pipelined create only: a finer work list for the staged first E-step.  A stage holds a fraction of the
    // blocks; cut into the resident iterations' items (about two per SM, sized for the fat backward CTA) it would keep
    // a quarter of the SMs busy, and the tail behind the last upload chunk would be one such item (~1.5 ms)
    std::vector<int32_t> cta_begin_fine;
    int ncta_fine = 0;
    CtaWork *d_work_fine = nullptr;
    // N = 4 with the exact item count (seqset_build): the forward kernel keeps a list of its own, items of whole rounds
    // (it has no per-item state to reduce, cuts every item into FWD4_SPLIT CTAs of 8 warps, and is bound by the HBM
    // write stream: 296 x 4 CTAs of 26.4 blocks take four block-times each just like 280 x 4 of 28, and 6 % longer in total)
    int ncta_fwd = 0;
    CtaWork *d_work_fwd = nullptr;
    int64_t spill_steps = 0;          // special: sum of tmax over blocks
    int tmax_all = 0;                 // longest sequence
    // device
    void *d_obs = nullptr;            // special: uint4 blocks; generic: canonical symbols
    void *d_meta = nullptr;           // one allocation behind d_off / d_foff / d_len / d_word / d_order
    int64_t *d_off = nullptr, *d_foff = nullptr;  // d_foff: frame prefix (generic) / uint4 row of the lane (N = 4 path)
    int32_t *d_len = nullptr, *d_word = nullptr, *d_order = nullptr;
    Blk *d_blks = nullptr;
    CtaWork *d_work = nullptr;
    int *d_bad = nullptr;                  // device flag: a codeword >= M was seen by the repack / convert kernels
    std::unique_ptr<PendingPrepare> pend;  // non-null while the repack is left to the first E-step
    void release() {
        pend.reset();  // waits for the copy stream before the raw buffer goes back to the allocator
        dev_free(d_bad);
        d_bad = nullptr;
        dev_free(d_obs); dev_free(d_meta); dev_free(d_blks); dev_free(d_work); dev_free(d_work_fine); dev_free(d_work_fwd);
        d_work_fwd = nullptr;
        d_obs = d_meta = nullptr; d_off = d_foff = nullptr; d_len = d_word = d_order = nullptr; d_blks = nullptr; d_work = nullptr;
        d_work_fine = nullptr;
    }
};

// Small host-to-device copies of a build.  While a codeword upload is in flight on the copy stream they go
// through that stream as well — one DMA queue, so they keep their place between the first chunks of the upload and the rest
// instead of being served after it (copies of different streams are not served in issue order) — and
// h2d_join() orders the compute stream behind them.
static int h2d_small(void *dst, const void *src, size_t bytes) {
    Ctx &c = ctx();
    HMMB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c.h2d_on_copy ? c.copy_stream : c.stream));
    return HMMB_OK;
}
static int h2d_join() {
    Ctx &c = ctx();
    if (!c.h2d_on_copy) return HMMB_OK;
    cudaEvent_t e = event_get();
    HMMB_CUDA(cudaEventRecord(e, c.copy_stream));
    HMMB_CUDA(cudaStreamWaitEvent(c.stream, e, 0));
    event_put(e);
    return HMMB_OK;
}

static int pick_np(int N) { return N <= 4 ? 4 : (N <= 8 ? 8 : (N <= 16 ? 16 : 32)); }

// Is every one of the W row-major N x N matrices A upper-bidiagonal (a_ij > 0 only for j = i or j = i + 1, the
// reference's left-to-right topology)?  Zeros of A stay zeros under re-estimation, so the answer holds for a whole fit.
static bool upper_bidiagonal(const double *A, int W, int N) {
    const size_t nA = (size_t)W * N * N;
    for (size_t e = 0; e < nA; ++e) {
        const int ij = (int)(e % (size_t)(N * N)), i = ij / N, j = ij % N;
        if (j != i && j != i + 1 && A[e] > 0.0) return false;
    }
    return true;
}

// Kernel family of W models with N states, M codewords and the transition matrices A (nullptr: not known yet).
struct Family {
    Layout blocked;  // the blocked layout whose kernels hold this (N, M), LAYOUT_LANES if none does
    bool bidiag;     // every A is upper-bidiagonal: the 7-term N = 4 kernels; LAYOUT_LTR requires it
    bool full_spill; // N = 4 E-step: spill every alpha-hat row instead of rebuilding the plain odd ones (reference arm)
    Layout layout() const { return blocked == LAYOUT_LTR && !bidiag ? LAYOUT_LANES : blocked; }
};

// The one place that reads the switches routing models to the other kernel family: HMMB_FORCE_GENERIC (every shape to
// the lanes-per-state kernels), HMMB_NO_LTR (N = 8 / 16 to them) and HMMB_FORCE_DENSE_A (A treated as dense); also
// HMMB_FULL_SPILL (the N = 4 E-step writes and reads every alpha-hat row).
static Family pick_family(int N, int M, const double *A, int W) {
    Family f{LAYOUT_LANES, A && !getenv("HMMB_FORCE_DENSE_A") && upper_bidiagonal(A, W, N), getenv("HMMB_FULL_SPILL") != nullptr};
    if (getenv("HMMB_FORCE_GENERIC")) return f;
    if (N == 4 && M <= BW4_MAX_M) {
        f.blocked = LAYOUT_N4;
    } else if ((N == 8 || N == 16) && M <= LTR_MAX_SYM && !getenv("HMMB_NO_LTR")) {
        // can the left-to-right kernels (bwltr_kernels.cuh) hold this model shape?
        const size_t stage = (size_t)LTR_WARPS * 32 * (N * 8 + 16);
        const size_t smem_b = (size_t)M * N * 8 + stage + (size_t)2 * N * 8 + (size_t)LTR_WARPS * 2 * N * 8 + 64;
        if (smem_b <= ctx().smem_optin) f.blocked = LAYOUT_LTR;
    }
    return f;
}

// Calls f(std::integral_constant<int, NP>{}, SymT{}) with the lanes per state and the codeword type of the
// lanes-per-state layout s, that is with the template arguments of its kernels.
template <typename F>
static int with_lanes(const SeqSet &s, F &&f) {
    auto sym = [&](auto np) { return s.sym_bytes == 1 ? f(np, uint8_t{}) : f(np, uint16_t{}); };
    switch (s.NP) {
        case 4: return sym(std::integral_constant<int, 4>{});
        case 8: return sym(std::integral_constant<int, 8>{});
        case 16: return sym(std::integral_constant<int, 16>{});
        case 32: return sym(std::integral_constant<int, 32>{});
    }
    return HMMB_ERR_UNSUPPORTED;
}

// Calls f(SymT{}, std::bool_constant<BLOCKED>{}) with how the codewords of s are stored: packed u16 entries in the
// blocked layouts, 1 or 2 bytes each in the lanes-per-state layout (the exact and rescue kernels read either).
template <typename F>
static int with_codewords(const SeqSet &s, F &&f) {
    if (s.blocked()) return f(uint16_t{}, std::true_type{});
    return s.sym_bytes == 1 ? f(uint8_t{}, std::false_type{}) : f(uint16_t{}, std::false_type{});
}

// Grid of the lanes-per-state kernels over R sequences: NP lanes per group of one sequence at a time, at most 16 CTAs
// per SM, each group taking per_group consecutive sequences.
struct LanesGrid {
    unsigned grid;
    int64_t per_group;
};
static LanesGrid lanes_grid(int64_t R, int NP) {
    const int64_t groups_per_cta = BW_WARPS * (32 / NP);
    const int64_t grid = std::min<int64_t>((std::max<int64_t>(R, 1) + groups_per_cta - 1) / groups_per_cta,
                                           (int64_t)ctx().sm_count * 16);
    const int64_t total_groups = grid * groups_per_cta;
    return {(unsigned)grid, (R + total_groups - 1) / total_groups};
}

// repack blocks [b0, b1) of the blocked layouts from the raw codewords (any input width)
template <typename InT>
static int launch_repack_typed(SeqSet &s, const InT *d_in, int b0, int b1, int *d_bad) {
    HMMB_LAUNCH("prepare", k_repack_blocks4<InT>, b1 - b0, REPACK_WARPS * 32, 0, d_in, s.d_off, s.d_len, s.d_blks, b0, s.nblk, (uint4 *)s.d_obs, s.M, d_bad);
    return HMMB_OK;
}
static int launch_repack_range(SeqSet &s, const void *d_in, int idx_bytes, int b0, int b1, int *d_bad) {
    if (b1 <= b0) return HMMB_OK;
    switch (idx_bytes) {
        case 1: return launch_repack_typed(s, (const uint8_t *)d_in, b0, b1, d_bad);
        case 2: return launch_repack_typed(s, (const uint16_t *)d_in, b0, b1, d_bad);
        case 4: return launch_repack_typed(s, (const uint32_t *)d_in, b0, b1, d_bad);
        default: return launch_repack_typed(s, (const unsigned long long *)d_in, b0, b1, d_bad);
    }
}

// first block whose codewords are not completely inside the first `hi_bytes` bytes of the raw stream
// (input already in sorted order: block order = raw order)
static int blocks_within(const std::vector<Blk> &blks, int from, const int64_t *off_s, const int32_t *len_s, int idx_bytes,
                         size_t hi_bytes) {
    int end = from;
    while (end < (int)blks.size()) {
        const Blk &b = blks[end];
        const int64_t last = (int64_t)b.first + b.nseq - 1;
        if ((size_t)(off_s[last] + len_s[last]) * (size_t)idx_bytes > hi_bytes) break;
        ++end;
    }
    return end;
}

template <typename InT>
static int launch_prepare(SeqSet &s, const InT *d_in, int64_t nsym, int *d_bad, const std::vector<Blk> &blks,
                          const EarlyUpload &up, bool in_sorted_order, const int64_t *off_s, const int32_t *len_s) {
    Ctx &c = ctx();
    if (s.blocked()) {
        int done = 0;
        if (up.active() && in_sorted_order) {
            for (int k = 0; k < up.nchunk; ++k) {
                const int end = k == up.nchunk - 1 ? s.nblk : blocks_within(blks, done, off_s, len_s, (int)sizeof(InT), up.hi[k]);
                HMMB_CUDA(cudaStreamWaitEvent(c.stream, up.ev[k], 0));
                if (end > done) HMMB_TRY(launch_repack_typed(s, d_in, done, end, d_bad));
                done = end;
            }
        } else {
            if (up.active()) HMMB_CUDA(cudaStreamWaitEvent(c.stream, up.ev[up.nchunk - 1], 0));
            if (s.nblk > 0) HMMB_TRY(launch_repack_typed(s, d_in, 0, s.nblk, d_bad));
        }
    } else {
        if (up.active()) HMMB_CUDA(cudaStreamWaitEvent(c.stream, up.ev[up.nchunk - 1], 0));
        int grid = (int)std::min<int64_t>((nsym + 255) / 256, (int64_t)c.sm_count * 8);
        if (grid < 1) grid = 1;
        if (s.sym_bytes == 1)
            HMMB_LAUNCH("prepare", (k_convert_obs<InT, uint8_t>), grid, 256, 0, d_in, nsym, (uint8_t *)s.d_obs, s.M, d_bad);
        else
            HMMB_LAUNCH("prepare", (k_convert_obs<InT, uint16_t>), grid, 256, 0, d_in, nsym, (uint16_t *)s.d_obs, s.M, d_bad);
    }
    return HMMB_OK;
}

// Sort sequences by (word, length desc), build blocks / CTA work items, move the codewords
// to the device in `layout`.  word_of_seq == nullptr: a single "word"
// (scoring: every utterance is scored against every model).
static int seqset_build(SeqSet &s, const void *obs, int idx_bytes, int obs_on_device, const int64_t *offsets,
                        const int32_t *word_of_seq, int64_t R, int W, int N, int M, Layout layout, bool defer = false,
                        const std::function<int()> *mid_hook = nullptr, int max_stages = 2) {
    Ctx &c = ctx();
    if (R < 0 || W <= 0 || !offsets || (R > 0 && !obs)) { set_error("bad sequence arguments"); return HMMB_ERR_ARG; }
    if (N < 1 || N > HMMB_MAX_STATES) { set_error("N=%d outside supported range 1..%d", N, HMMB_MAX_STATES); return HMMB_ERR_UNSUPPORTED; }
    if (M < 1 || M > 65536) { set_error("M=%d outside supported range 1..65536", M); return HMMB_ERR_UNSUPPORTED; }
    if (idx_bytes != 1 && idx_bytes != 2 && idx_bytes != 4 && idx_bytes != 8) { set_error("idx_bytes must be 1, 2, 4 or 8"); return HMMB_ERR_ARG; }
    s.R = R; s.N = N; s.M = M; s.NP = pick_np(N);
    s.sym_bytes = M <= 256 ? 1 : 2;
    s.layout = layout;

    std::unique_ptr<EarlyUpload> up_owner(new EarlyUpload());
    EarlyUpload &up = *up_owner;
    struct H2dGuard { ~H2dGuard() { ctx().h2d_on_copy = false; ctx().after_chunk = nullptr; } } h2d_guard;
    if (!obs_on_device && R > 0 && offsets[R] > offsets[0] && offsets[R] - offsets[0] < (int64_t(1) << 40)) {
        const char *src = (const char *)obs + (size_t)offsets[0] * idx_bytes;
        const size_t in_bytes = (size_t)(offsets[R] - offsets[0]) * idx_bytes;
        cudaPointerAttributes attr;
        const bool pinned = cudaPointerGetAttributes(&attr, src) == cudaSuccess && attr.type == cudaMemoryTypeHost;
        (void)cudaGetLastError();
        if (pinned && in_bytes >= (size_t(4) << 20)) {
            HMMB_TRY(dev_alloc(&up.d_raw, in_bytes));
            // the recycled block may still be in use by work queued on the compute stream
            cudaEvent_t fence = event_get();
            HMMB_CUDA(cudaEventRecord(fence, c.stream));
            HMMB_CUDA(cudaStreamWaitEvent(c.copy_stream, fence, 0));
            event_put(fence);
            const int nchunk = (int)std::min<size_t>(EarlyUpload::MAX_CHUNKS, std::max<size_t>(1, in_bytes >> 24));
            up.src = src;
            for (int k = 0; k < nchunk; ++k) {
                up.hi[k] = k == nchunk - 1 ? in_bytes : ((in_bytes / nchunk) * (k + 1)) & ~size_t(255);
                up.ev[k] = event_get();
                up.nchunk = k + 1;
            }
            // as many chunks as the host-side pass below takes (~0.55 ms per million sequences = one chunk of config 3's
            // eight); the metadata goes next in the DMA queue, the rest of the codewords behind it.  The first stage of the
            // pipelined E-step cannot start before the metadata has landed: with two chunks ahead of it (the default
            // until late in round 2) that was 1.8 ms into the call, with one 1.5 ms — 5.6 -> 5.4 ms per fit call
            HMMB_TRY(up.issue(std::max(1, nchunk / 8)));
            c.h2d_on_copy = true;
        }
    }

    // Per-sequence metadata is staged in ONE pinned host buffer (cached in the context) and goes to the device
    // with a single copy: [off int64 | len int32 | order int32 | foff int64 | word int32].  The blocked layouts
    // only send the first 12 (input in sorted order) or 16 bytes per sequence: the rest follows from the block
    // table (k_meta_blocked).
    const size_t nR = (size_t)std::max<int64_t>(R, 1);
    const size_t meta_bytes = nR * (2 * sizeof(int64_t) + 3 * sizeof(int32_t));
    if (c.stage_busy) {  // the previous build's metadata copy (possibly still queued behind a codeword upload)
        cudaEventSynchronize(c.stage_busy);
        event_put(c.stage_busy);
        c.stage_busy = nullptr;
    }
    if (c.stage_bytes < meta_bytes) {
        if (c.stage) cudaFreeHost(c.stage);
        c.stage = nullptr;
        c.stage_bytes = 0;
        if (cudaHostAlloc(&c.stage, meta_bytes + (meta_bytes >> 2), cudaHostAllocDefault) != cudaSuccess) {
            (void)cudaGetLastError();
            set_error("pinned staging allocation of %zu bytes failed", meta_bytes);
            return HMMB_ERR_OOM;
        }
        c.stage_bytes = meta_bytes + (meta_bytes >> 2);
    }
    int64_t *off_s = reinterpret_cast<int64_t *>(c.stage);
    int32_t *len_s = reinterpret_cast<int32_t *>(off_s + nR);
    int32_t *order_s = len_s + nR;
    int64_t *foff_s = reinterpret_cast<int64_t *>(order_s + nR);
    int32_t *word_s = reinterpret_cast<int32_t *>(foff_s + nR);

    // One pass: validate, lengths, "already in (word, length descending) order?", and the staging arrays filled
    // for that (usual) case; only an unsorted input pays for the sort and a second fill.
    // (len: a context-owned scratch vector — a fresh 4 MB vector per build costs more in page faults than the loop)
    std::vector<int32_t> &len = c.len_scratch;
    if ((int64_t)len.size() < R) len.resize((size_t)R);
    int bad_kind = 0;
    int64_t bad_at = -1;
    int unsorted = 0;
    int tmax_all = 0;
    auto clamp_len = [](int64_t T) { return (int32_t)(T > 0 && T <= (1 << 30) ? T : 0); };
#pragma omp parallel for schedule(static) reduction(| : unsorted) reduction(max : tmax_all) if (R > 65536)
    for (int64_t r = 0; r < R; ++r) {
        const int64_t T = offsets[r + 1] - offsets[r];
        const int32_t wb = word_of_seq ? word_of_seq[r] : 0;
        int kind = 0;
        if (T == 0) kind = 1;
        else if (T < 0) kind = 2;
        else if (T > (1 << 30)) kind = 3;
        else if (wb < 0 || wb >= W) kind = 4;
        if (kind) {
#pragma omp critical
            if (bad_at < 0 || r < bad_at) { bad_at = r; bad_kind = kind; }
        }
        const int32_t l = clamp_len(T);
        len[r] = l;
        if (r > 0) {
            const int32_t wa = word_of_seq ? word_of_seq[r - 1] : 0;
            if (wa > wb || (wa == wb && clamp_len(offsets[r] - offsets[r - 1]) < l)) unsorted |= 1;
        }
        order_s[r] = (int32_t)r;
        off_s[r] = offsets[r] - offsets[0];
        len_s[r] = l;
        word_s[r] = wb;
        tmax_all = std::max(tmax_all, (int)l);
    }
    if (bad_kind == 1) {
        // reference: IndexError at hmm_training.py:376 / hmm_testing.py:75 for an empty recording
        set_error("sequence %lld is empty (T == 0)", (long long)bad_at);
        return HMMB_ERR_EMPTY;
    } else if (bad_kind == 2) {
        set_error("offsets not monotone at sequence %lld", (long long)bad_at);
        return HMMB_ERR_ARG;
    } else if (bad_kind == 3) {
        set_error("sequence %lld too long", (long long)bad_at);
        return HMMB_ERR_UNSUPPORTED;
    } else if (bad_kind == 4) {
        set_error("word_of_seq[%lld]=%d outside [0,%d)", (long long)bad_at, word_of_seq[bad_at], W);
        return HMMB_ERR_ARG;
    }
    s.frames = R > 0 ? offsets[R] - offsets[0] : 0;
    if (unsorted) {
        std::stable_sort(order_s, order_s + R, [&](int32_t x, int32_t y) {
            const int wx = word_of_seq ? word_of_seq[x] : 0, wy = word_of_seq ? word_of_seq[y] : 0;
            if (wx != wy) return wx < wy;
            return len[x] > len[y];
        });
#pragma omp parallel for schedule(static) if (R > 65536)
        for (int64_t i = 0; i < R; ++i) {
            const int32_t r = order_s[i];
            off_s[i] = offsets[r] - offsets[0];
            len_s[i] = len[r];
            word_s[i] = word_of_seq ? word_of_seq[r] : 0;
        }
    }
    const int nwords = word_of_seq ? W : 1;
    s.seq_begin.assign(nwords + 1, 0);
    s.tmax_all = tmax_all;
    // sequences of a word are contiguous in the sorted order: word boundaries by binary search
    for (int w = 0; w < nwords; ++w)
        s.seq_begin[w + 1] = std::upper_bound(word_s, word_s + R, (int32_t)w) - word_s;
    if (unsorted) s.order.assign(order_s, order_s + R);  // empty = identity (input already in sorted order)
    else s.order.clear();
    if (!s.blocked()) {
        int64_t facc = 0;  // frame prefix (generic path only; the N = 4 path stores block rows here)
        for (int64_t i = 0; i < R; ++i) {
            foff_s[i] = facc;
            facc += len_s[i];
        }
    }

    std::vector<Blk> blks;
    std::vector<CtaWork> work, work_fine, work_fwd;
    blks.reserve((size_t)(R / 32 + nwords + 1));
    int64_t obs_rows = 0;
    if (s.blocked()) {
        const int SPC = SPC4;  // packed u16 entries (codeword | conflict rank) per uint4
        const int cta_warps = s.layout == LAYOUT_N4 ? BWD4_MAX_WARPS : LTR_WARPS;
        std::vector<int> word_blk_begin(nwords + 1, 0);
        for (int w = 0; w < nwords; ++w) {
            word_blk_begin[w] = (int)blks.size();
            for (int64_t i = s.seq_begin[w]; i < s.seq_begin[w + 1]; i += 32) {
                Blk b;
                b.word = w;
                b.first = (int32_t)i;
                b.nseq = (int32_t)std::min<int64_t>(32, s.seq_begin[w + 1] - i);
                b.tmax = len_s[i];  // sorted by length descending within the word
                b.obs_base = obs_rows;
                b.spill_base = s.spill_steps;
                obs_rows += (int64_t)((b.tmax + SPC - 1) / SPC) * 32;
                s.spill_steps += b.tmax;
                blks.push_back(b);
            }
        }
        word_blk_begin[nwords] = (int)blks.size();
        s.nblk = (int)blks.size();
        // CTA work items: ~2 per SM (N = 4) / ~4 per SM (left-to-right kernels, one 8-warp CTA per SM), at least one
        // warp-round each
        // (N = 4: one fat backward CTA per SM, about two waves; the forward kernel splits every item over FWD4_SPLIT CTAs)
        const int target = s.layout == LAYOUT_N4 ? c.sm_count * 2 : c.sm_count * 4;
        int bpc = std::max(1, (s.nblk + target - 1) / target);
        if (bpc > 1 || s.layout != LAYOUT_N4) bpc = (bpc + cta_warps - 1) / cta_warps * cta_warps;
        s.cta_begin.assign(nwords + 1, 0);
        // N = 4, large inputs: EXACTLY `target` items of (almost) equal size, apportioned to the words by their block counts
        // (largest remainder).  The fat backward CTA works in rounds of 16 blocks and one CTA occupies an SM, so the kernel
        // takes waves x rounds-per-item: items rounded up to whole rounds left config 3 with 280 items of 7 rounds on 2 x 148
        // CTA slots — 14 rounds per SM for 13.2 rounds of work, 16 SMs idle in the second wave.  296 items of 105.6 blocks
        // are 6 full rounds and one with 10 of the 16 warps busy, which is shorter than a full one.
        std::vector<int> items_of_word;
        if (s.layout == LAYOUT_N4 && (int64_t)s.nblk >= (int64_t)target * cta_warps * 2) {
            items_of_word.assign(nwords, 0);
            std::vector<std::pair<double, int>> rem;
            int64_t assigned = 0;
            for (int w = 0; w < nwords; ++w) {
                const int nb = word_blk_begin[w + 1] - word_blk_begin[w];
                if (nb == 0) continue;
                const double q = (double)nb * target / s.nblk;
                items_of_word[w] = std::max(1, (int)q);
                assigned += items_of_word[w];
                rem.emplace_back(q - (int)q, w);
            }
            std::sort(rem.begin(), rem.end(), [](const std::pair<double, int> &a, const std::pair<double, int> &b) {
                return a.first != b.first ? a.first > b.first : a.second < b.second;
            });
            for (size_t k = 0; k < rem.size() && assigned < target; ++k, ++assigned) ++items_of_word[rem[k].second];
        }
        for (int w = 0; w < nwords; ++w) {
            s.cta_begin[w] = (int)work.size();
            if (!items_of_word.empty()) {
                for (int b = word_blk_begin[w]; b < word_blk_begin[w + 1]; b += bpc) {  // the forward kernel's list
                    CtaWork cw;
                    cw.word = w;
                    cw.blk_begin = b;
                    cw.blk_end = std::min(word_blk_begin[w + 1], b + bpc);
                    cw.seq_begin = blks[b].first;
                    work_fwd.push_back(cw);
                }
                const int b0 = word_blk_begin[w], nb = word_blk_begin[w + 1] - b0, ni = items_of_word[w];
                for (int i = 0; i < ni; ++i) {
                    CtaWork cw;
                    cw.word = w;
                    cw.blk_begin = b0 + (int)((int64_t)nb * i / ni);
                    cw.blk_end = b0 + (int)((int64_t)nb * (i + 1) / ni);
                    if (cw.blk_end == cw.blk_begin) continue;
                    cw.seq_begin = blks[cw.blk_begin].first;
                    work.push_back(cw);
                }
                continue;
            }
            for (int b = word_blk_begin[w]; b < word_blk_begin[w + 1]; b += bpc) {
                CtaWork cw;
                cw.word = w;
                cw.blk_begin = b;
                cw.blk_end = std::min(word_blk_begin[w + 1], b + bpc);
                cw.seq_begin = blks[b].first;
                work.push_back(cw);
            }
        }
        s.cta_begin[nwords] = (int)work.size();
        s.ncta = (int)work.size();
        s.ncta_fwd = (int)work_fwd.size();
        if (s.layout == LAYOUT_N4 && defer) {
            const int fine_items = c.sm_count * 8;  // about eight per SM (SeqSet::cta_begin_fine)
            int bpf = std::max(1, (s.nblk + fine_items - 1) / fine_items);
            if (bpf > 1) bpf = (bpf + cta_warps - 1) / cta_warps * cta_warps;
            if (bpf < bpc) {
                s.cta_begin_fine.assign(nwords + 1, 0);
                for (int w = 0; w < nwords; ++w) {
                    s.cta_begin_fine[w] = (int)work_fine.size();
                    for (int b = word_blk_begin[w]; b < word_blk_begin[w + 1]; b += bpf) {
                        CtaWork cw;
                        cw.word = w;
                        cw.blk_begin = b;
                        cw.blk_end = std::min(word_blk_begin[w + 1], b + bpf);
                        cw.seq_begin = blks[b].first;
                        work_fine.push_back(cw);
                    }
                }
                s.cta_begin_fine[nwords] = (int)work_fine.size();
                s.ncta_fine = (int)work_fine.size();
            }
        }
    }

    // ---- device buffers
    HMMB_TRY(dev_alloc(&s.d_meta, meta_bytes));
    s.d_off = reinterpret_cast<int64_t *>(s.d_meta);
    s.d_len = reinterpret_cast<int32_t *>(s.d_off + nR);
    s.d_order = s.d_len + nR;
    s.d_foff = reinterpret_cast<int64_t *>(s.d_order + nR);
    s.d_word = reinterpret_cast<int32_t *>(s.d_foff + nR);
    if (R > 0) {
        const size_t sent = !s.blocked() ? meta_bytes : nR * (unsorted ? 16 : 12);
        HMMB_TRY(h2d_small(s.d_meta, c.stage, sent));
        c.stage_busy = event_get();
        HMMB_CUDA(cudaEventRecord(c.stage_busy, c.h2d_on_copy ? c.copy_stream : c.stream));
    }
    if (s.blocked()) {
        HMMB_TRY(dev_alloc_t(&s.d_blks, std::max<size_t>(blks.size(), 1)));
        HMMB_TRY(dev_alloc_t(&s.d_work, std::max<size_t>(work.size(), 1)));
        if (!blks.empty()) {
            HMMB_TRY(h2d_small(s.d_blks, blks.data(), blks.size() * sizeof(Blk)));
            HMMB_TRY(h2d_small(s.d_work, work.data(), work.size() * sizeof(CtaWork)));
            if (s.ncta_fine > 0) {
                HMMB_TRY(dev_alloc_t(&s.d_work_fine, work_fine.size()));
                HMMB_TRY(h2d_small(s.d_work_fine, work_fine.data(), work_fine.size() * sizeof(CtaWork)));
            }
            if (s.ncta_fwd > 0) {
                HMMB_TRY(dev_alloc_t(&s.d_work_fwd, work_fwd.size()));
                HMMB_TRY(h2d_small(s.d_work_fwd, work_fwd.data(), work_fwd.size() * sizeof(CtaWork)));
            }
        }
        HMMB_TRY(dev_alloc(&s.d_obs, (size_t)std::max<int64_t>(obs_rows, 1) * sizeof(uint4)));
    } else {
        HMMB_TRY(dev_alloc(&s.d_obs, (size_t)std::max<int64_t>(s.frames, 1) * s.sym_bytes));
    }
    // the caller's own small uploads (accumulator layout, initial parameters) also go ahead of the
    // rest of the codewords in the DMA queue
    if (mid_hook) HMMB_TRY((*mid_hook)());
    HMMB_TRY(h2d_join());
    c.h2d_on_copy = false;
    if (up.active()) HMMB_TRY(up.issue(up.nchunk));  // the rest of the codewords, behind the metadata
    if (up.active() && c.after_chunk) HMMB_TRY(c.after_chunk(up.nchunk - 1, up.nchunk));  // (all chunks were out before the hook existed)
    if (s.blocked() && s.nblk > 0)
        HMMB_LAUNCH("prepare", k_meta_blocked, std::min((s.nblk + 7) / 8, c.sm_count * 8), 256, 0, s.d_blks, s.nblk, s.d_foff,
                    s.d_word, unsorted ? (int32_t *)nullptr : s.d_order);
    // raw codewords -> device (if needed) -> canonical layout
    const void *d_in = obs;
    void *d_tmp = nullptr;
    const size_t in_bytes = (size_t)s.frames * idx_bytes;
    if (R > 0) {
        const char *src = (const char *)obs + (size_t)offsets[0] * idx_bytes;
        if (up.active()) {
            d_in = up.d_raw;  // already on its way (copy stream); launch_prepare waits on the chunk events
        } else if (!obs_on_device) {
            HMMB_TRY(dev_alloc(&d_tmp, in_bytes));
            HMMB_TRY(h2d_big(d_tmp, src, in_bytes, c.stream));  // pageable codewords: through the pinned bounce buffers
            d_in = d_tmp;
        } else {
            d_in = src;
        }
    }
    HMMB_TRY(dev_alloc_t(&s.d_bad, 1));
    int *d_bad = s.d_bad;
    HMMB_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int), c.stream));
    if (defer && s.blocked() && up.active() && !unsorted && s.nblk > 0) {
        // leave the repack to the first E-step (bw_estep): record which blocks / CTA work items each stage completes
        std::unique_ptr<PendingPrepare> p(new PendingPrepare());
        p->idx_bytes = idx_bytes;
        p->nstage = std::max(1, std::min<int>(std::min<int>(PendingPrepare::MAX_STAGES, max_stages), up.nchunk));
        int bdone = 0, cdone = 0;
        const std::vector<CtaWork> &wl = s.ncta_fine > 0 ? work_fine : work;  // the list the staged E-step launches from
        const int nwl = (int)wl.size();
        for (int j = 0; j < p->nstage; ++j) {
            const int k = (j + 1) * up.nchunk / p->nstage - 1;  // the stage is complete when chunk k has landed
            p->ev_index[j] = k;
            bdone = (j == p->nstage - 1) ? s.nblk : blocks_within(blks, bdone, off_s, len_s, idx_bytes, up.hi[k]);
            while (cdone < nwl && wl[cdone].blk_end <= bdone) ++cdone;
            p->blk_end[j] = bdone;
            p->cta_end[j] = (j == p->nstage - 1) ? nwl : cdone;
        }
        p->up = std::move(up_owner);
        s.pend = std::move(p);
        return HMMB_OK;
    }
    int rc = HMMB_OK;
    if (R > 0) {
        switch (idx_bytes) {
            case 1: rc = launch_prepare(s, (const uint8_t *)d_in, s.frames, d_bad, blks, up, !unsorted, off_s, len_s); break;
            case 2: rc = launch_prepare(s, (const uint16_t *)d_in, s.frames, d_bad, blks, up, !unsorted, off_s, len_s); break;
            case 4: rc = launch_prepare(s, (const uint32_t *)d_in, s.frames, d_bad, blks, up, !unsorted, off_s, len_s); break;
            default: rc = launch_prepare(s, (const unsigned long long *)d_in, s.frames, d_bad, blks, up, !unsorted, off_s, len_s); break;
        }
    }
    int bad = 0;
    if (rc == HMMB_OK) {
        cudaError_t e = cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, c.stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c.stream);
        if (e != cudaSuccess) rc = cuda_fail(e, "prepare sync", __FILE__, __LINE__);
    }
    dev_free(d_tmp);
    if (rc != HMMB_OK) return rc;
    if (bad) {
        set_error("codeword out of range: some observation is >= M=%d (reference: IndexError)", M);
        return HMMB_ERR_RANGE;
    }
    return HMMB_OK;
}

}  // namespace hmmb

using namespace hmmb;

// ---------------------------------------------------------------- the trainer handle
struct hmmb_bw {
    SeqSet s;                     // N = 4: blocked layout; otherwise the generic (lanes = states) layout
    SeqSet sl;                    // N = 8 / 16: additional blocked layout for the left-to-right kernels
    bool has_ltr = false;         // sl was built
    bool use_ltr = false;         // every word's A is upper-bidiagonal (checked in set_params): run the sl kernels
    uint8_t *d_allfull = nullptr; // per sequence: every spilled alpha-hat > 0 (written by the forward kernels)
    uint32_t *d_oddmask = nullptr; // N = 4: per (block, odd step) the lanes that wrote that alpha-hat row (k_bw_fwd4)
    bool full_spill = false;      // N = 4: every alpha-hat row written and read (HMMB_FULL_SPILL, see pick_family)
    bool check_bad = false;       // pipelined prepare: the codeword-range flag has not been read back yet
    std::unique_ptr<PendingPrepare> pend_release;  // consumed by the E-step; freed after the next stream sync
    void *d_raw = nullptr;        // raw codewords uploaded once when both layouts are built
    // Pipelined create with left-to-right initial parameters: only `sl` is built (its repack is left to the first
    // E-step, stage by stage behind the upload); `s` carries the sizes alone.  The raw codewords and the sequence
    // table are kept so that the generic layout can still be built should dense parameters arrive later.
    bool ltr_only = false;
    int raw_idx_bytes = 0;
    // ... and its initial B goes up in `bpieces` word ranges interleaved with the codeword chunks (B^T of piece p is
    // ready at bt_ready[p], recorded on the copy stream), so that the first stage does not wait for all of B
    // thin-state rescue (hmm_device.cuh): sticky per-word state masks, slots behind the accumulators
    uint32_t *d_thinmask = nullptr;   // [W]
    int32_t *d_thin_new = nullptr;    // states flagged since the host last looked
    int32_t *d_redo = nullptr;        // [W] words whose M-step was held back for a repeat of the iteration
    int32_t *d_redo_in = nullptr;     // [W] copy of d_redo that the repeat runs on (the M-step rewrites d_redo)
    int32_t *d_slot_of = nullptr;     // [W][N] slot of a flagged state, -1 = none
    int32_t *act_cur = nullptr;       // the word mask the E-step launches use (d_active, or d_redo in a repeat)
    int64_t slot_cap = 0, rstride = 0;
    int n_slots = 0;
    int64_t n_thin_total = 0;
    int bpieces = 0, bpieces_issued = 0;
    cudaEvent_t bt_ready[PendingPrepare::MAX_STAGES] = {};
    double *d_ptmp = nullptr;     // upload buffer of those parameters (released after the first E-step)
    std::vector<int64_t> keep_offsets;
    std::vector<int32_t> keep_words;
    SeqSet &cur() { return use_ltr ? sl : s; }
    int W = 0, N = 0, M = 0;
    double *d_pi = nullptr, *d_A = nullptr, *d_Bt = nullptr;
    double *d_spill = nullptr, *d_llseq = nullptr, *d_accum = nullptr, *d_partials = nullptr;
    double *d_prev = nullptr, *d_hist = nullptr;
    int32_t *d_active = nullptr, *d_iters = nullptr, *d_any = nullptr, *d_cta_begin = nullptr;
    int32_t *d_cta_begin_fine = nullptr;  // per-word ranges of the staged first E-step's finer work list (SeqSet::cta_begin_fine)
    bool estep_fine = false;              // the partials of the last E-step are laid out by the finer list
    int32_t *d_bzero = nullptr;   // per word: B has an exact zero (disables the lean backward path)
    bool bidiag = false;          // every word's A is upper-bidiagonal (checked in set_params)
    int64_t *d_seq_begin = nullptr;
    // precision guard: sticky per-sequence hand-over flags, counters, exact-kernel scratch
    uint8_t *d_flag = nullptr, *d_flag_base = nullptr;  // d_flag = d_flag_base + FLAG_HDR
    int32_t *d_newflags = nullptr;
    int64_t *d_nexact = nullptr;
    double *d_exact_scratch = nullptr;
    int exact_grid = 1;
    int64_t exact_stride = 0;
    int64_t n_backward_handover = 0;
    int64_t nacc = 0, astride = 0, accum_n = 0, pstride = 0;
    int hist_cap = 0;
    int rank = 0, world = 1;
    hmmb_allreduce_fn allreduce = nullptr;
    void *user = nullptr;
    int overlap_groups = 1;        // > 1: left-to-right E-step in word groups, each group's accumulators all-reduced
                                   // while the next group's backward pass runs (hmmb_bw_set_overlap)
    bool estep_reduced = false;    // the E-step just launched did the reduce + all-reduce itself
    bool params_set = false, any_active = true;
};

// alpha-hat spill of the N = 4 kernels (behind its front padding, see bw_finish_create)
static double2 *spill4(hmmb_bw *h) { return reinterpret_cast<double2 *>(h->d_spill) + (size_t)BWD4_SPILL_PAD * 64; }
// odd-row lane masks of the N = 4 kernels, one word per spill row (even rows unused), with the same front padding
static unsigned *oddmask4(hmmb_bw *h) { return h->d_oddmask + BWD4_SPILL_PAD; }

static void bw_drop_pieces(hmmb_bw *h) {
    for (auto &e : h->bt_ready) {
        if (e) event_put(e);
        e = nullptr;
    }
    h->bpieces = h->bpieces_issued = 0;
    dev_free(h->d_ptmp);
    h->d_ptmp = nullptr;
}

static void bw_release(hmmb_bw *h) {
    if (h->d_ptmp && ctx().inited) cudaStreamSynchronize(ctx().copy_stream);
    bw_drop_pieces(h);
    h->pend_release.reset();
    h->s.release();
    h->sl.release();
    dev_free(h->d_allfull);
    dev_free(h->d_oddmask);
    dev_free(h->d_raw);
    dev_free(h->d_pi); dev_free(h->d_A); dev_free(h->d_Bt); dev_free(h->d_spill); dev_free(h->d_llseq);
    dev_free(h->d_accum); dev_free(h->d_partials); dev_free(h->d_prev); dev_free(h->d_hist); dev_free(h->d_active);
    dev_free(h->d_iters); dev_free(h->d_any); dev_free(h->d_cta_begin); dev_free(h->d_cta_begin_fine); dev_free(h->d_seq_begin);
    dev_free(h->d_bzero); dev_free(h->d_flag_base); dev_free(h->d_newflags); dev_free(h->d_nexact); dev_free(h->d_exact_scratch);
    dev_free(h->d_thinmask); dev_free(h->d_thin_new); dev_free(h->d_redo); dev_free(h->d_redo_in); dev_free(h->d_slot_of);
}

static int bw_alloc_accum(hmmb_bw *h) {
    dev_free(h->d_accum);
    h->d_accum = nullptr;
    h->accum_n = (int64_t)h->W * h->astride + (int64_t)h->world * h->W * 2 + (int64_t)h->world * h->slot_cap * h->rstride;
    return dev_alloc_t(&h->d_accum, (size_t)h->accum_n);
}

static int bw_set_params_impl(hmmb_bw *h, const double *pi0, const double *A0, const double *B0, bool sync);
static int bw_after_sync(hmmb_bw *h);

// Buffers sized by the sequence set, accumulator layout, the small per-word uploads (second half of hmmb_bw_create).
static int bw_finish_create(hmmb_bw *h, int64_t R) {
    Ctx &c = ctx();
    SeqSet &s = h->s;
    const int W = h->W, N = h->N, M = h->M;
    h->nacc = (int64_t)N + (int64_t)N * N + (int64_t)M * N;
    // stride multiple of 16 doubles: every word's count rows start on a 128-byte line (TMA bulk reductions)
    h->astride = (h->nacc + 1 + 15) & ~int64_t(15);
    h->pstride = h->nacc + 2;  // + the CTA's (max, sum exp) pair of the convergence statistic
    h->hist_cap = 0;
#define TRYF(expr) HMMB_TRY(expr)
#define CUDAF(expr) HMMB_CUDA(expr)
    TRYF(dev_alloc_t(&h->d_pi, (size_t)W * N));
    TRYF(dev_alloc_t(&h->d_A, (size_t)W * N * N));
    TRYF(dev_alloc_t(&h->d_Bt, (size_t)W * M * N));
    TRYF(dev_alloc_t(&h->d_llseq, (size_t)std::max<int64_t>(R, 1)));
    TRYF(bw_alloc_accum(h));
    TRYF(dev_alloc_t(&h->d_prev, (size_t)W));
    TRYF(dev_alloc_t(&h->d_active, (size_t)W));
    h->act_cur = h->d_active;
    TRYF(dev_alloc_t(&h->d_iters, (size_t)W));
    TRYF(dev_alloc_t(&h->d_any, 1));
    TRYF(dev_alloc_t(&h->d_bzero, (size_t)W));
    h->rstride = ((int64_t)N + M + 15) & ~int64_t(15);
    TRYF(dev_alloc_t(&h->d_thinmask, (size_t)W));
    TRYF(dev_alloc_t(&h->d_thin_new, 1));
    TRYF(dev_alloc_t(&h->d_redo, (size_t)W));
    TRYF(dev_alloc_t(&h->d_redo_in, (size_t)W));
    TRYF(dev_alloc_t(&h->d_slot_of, (size_t)W * N));
    TRYF(dev_alloc_t(&h->d_flag_base, (size_t)std::max<int64_t>(R, 1) + FLAG_HDR));  // header: see raise_flag
    h->d_flag = h->d_flag_base + FLAG_HDR;
    TRYF(dev_alloc_t(&h->d_newflags, 1));
    TRYF(dev_alloc_t(&h->d_nexact, 1));
    {
        // exact log-space kernel: one warp per handed-over sequence, log alpha scratch per warp
        h->exact_stride = (int64_t)std::max(s.tmax_all, 1) * N;
        int64_t warps = std::min<int64_t>((int64_t)c.sm_count * 8, std::max<int64_t>(1, (256LL << 20) / (h->exact_stride * 8)));
        warps = std::min<int64_t>(warps, std::max<int64_t>(1, (R + 31) / 32));
        h->exact_grid = (int)std::max<int64_t>(1, (warps + BW_WARPS - 1) / BW_WARPS);
        TRYF(dev_alloc_t(&h->d_exact_scratch, (size_t)h->exact_grid * BW_WARPS * h->exact_stride));
    }
    TRYF(dev_alloc_t(&h->d_seq_begin, (size_t)W + 1));
    TRYF(h2d_small(h->d_seq_begin, s.seq_begin.data(), (W + 1) * sizeof(int64_t)));
    size_t spill_bytes;
    if (s.layout == LAYOUT_N4) {
        // + BWD4_SPILL_PAD rows in front: k_bw_bwd4 loads row t - 2 unconditionally (for t < 2 that is the tail of
        // the previous block, or this padding for the first block; the values are never used)
        spill_bytes = (size_t)(std::max<int64_t>(s.spill_steps, 1) + BWD4_SPILL_PAD) * 64 * sizeof(double2);
        TRYF(dev_alloc_t(&h->d_partials, (size_t)std::max(std::max(s.ncta, s.ncta_fine), 1) * h->pstride));
        TRYF(dev_alloc_t(&h->d_cta_begin, (size_t)W + 1));
        if (s.ncta_fine > 0) {
            TRYF(dev_alloc_t(&h->d_cta_begin_fine, (size_t)W + 1));
            TRYF(h2d_small(h->d_cta_begin_fine, s.cta_begin_fine.data(), (W + 1) * sizeof(int32_t)));
        }
        TRYF(dev_alloc_t(&h->d_allfull, (size_t)std::max<int64_t>(R, 1)));
        TRYF(dev_alloc_t(&h->d_oddmask, (size_t)(std::max<int64_t>(s.spill_steps, 1) + BWD4_SPILL_PAD)));
        TRYF(h2d_small(h->d_cta_begin, s.cta_begin.data(), (W + 1) * sizeof(int32_t)));
    } else {
        spill_bytes = (size_t)std::max<int64_t>(s.frames, 1) * N * sizeof(double);
        if (h->has_ltr) {
            spill_bytes = std::max(spill_bytes, (size_t)std::max<int64_t>(h->sl.spill_steps, 1) * 32 * N * sizeof(double));
            TRYF(dev_alloc_t(&h->d_allfull, (size_t)std::max<int64_t>(R, 1)));
        }
    }
    int rc = dev_alloc((void **)&h->d_spill, spill_bytes);
    if (rc != HMMB_OK) {
        set_error("alpha spill of %.2f GB does not fit in device memory; shard the sequences over more GPUs",
                  spill_bytes / 1e9);
        return HMMB_ERR_OOM;
    }
#undef TRYF
#undef CUDAF
    return HMMB_OK;
}


// (C linkage comes from the declarations in include/hmmb200.h)

int hmmb_bw_create(hmmb_bw_t **out, const void *obs, int idx_bytes, int obs_on_device, const int64_t *offsets,
                   const int32_t *word_of_seq, int64_t R, int W, int N, int M) {
    return hmmb_bw_create_ex(out, obs, idx_bytes, obs_on_device, offsets, word_of_seq, R, W, N, M, 0, nullptr, nullptr,
                             nullptr);
}

int hmmb_bw_create_ex(hmmb_bw_t **out, const void *obs, int idx_bytes, int obs_on_device, const int64_t *offsets,
                      const int32_t *word_of_seq, int64_t R, int W, int N, int M, int flags, const double *pi0,
                      const double *A0, const double *B0) {
    HMMB_TRY(require_init());
    if (!out || !word_of_seq) { set_error("hmmb_bw_create: null argument"); return HMMB_ERR_ARG; }
    *out = nullptr;
    Ctx &c = ctx();
    hmmb_bw *h = new hmmb_bw();
    h->W = W; h->N = N; h->M = M;
    auto fail = [&](int code) { bw_release(h); delete h; return code; };
    int rc;
    const bool have_params = pi0 && A0 && B0;
    // N = 8 / 16: the generic layout in `s` and, if the left-to-right kernels hold the shape, the blocked one in `sl`
    // (set_params picks between them)
    const Family fam = pick_family(N, M, have_params ? A0 : nullptr, W);
    const Layout s_layout = fam.blocked == LAYOUT_N4 ? LAYOUT_N4 : LAYOUT_LANES;
    h->has_ltr = fam.blocked == LAYOUT_LTR;
    // Pipelined create for the left-to-right kernels (N = 8 / 16): pinned host codewords, initial parameters given
    // and every A upper-bidiagonal.  Only the blocked layout is built, and its repack is left to the first E-step.
    const bool ltr_pipe = fam.layout() == LAYOUT_LTR && (flags & HMMB_BW_PIPELINE_UPLOAD) && !obs_on_device && R > 0 &&
                          offsets && obs && offsets[R] > offsets[0] &&
                          host_is_pinned((const char *)obs + (size_t)offsets[0] * idx_bytes);
    if (h->has_ltr && !ltr_pipe && !obs_on_device && R > 0 && offsets && obs && offsets[R] > offsets[0]) {
        // both layouts are built from the codewords: upload them once
        const size_t in_bytes = (size_t)(offsets[R] - offsets[0]) * idx_bytes;
        rc = dev_alloc(&h->d_raw, in_bytes);
        if (rc != HMMB_OK) return fail(rc);
        rc = h2d_big(h->d_raw, (const char *)obs + (size_t)offsets[0] * idx_bytes, in_bytes, c.stream);
        if (rc != HMMB_OK) return fail(rc);
        // seqset_build indexes a device stream from offsets[0]
        obs = (const char *)h->d_raw - (size_t)offsets[0] * idx_bytes;
        obs_on_device = 1;
    }
    // everything that follows the sequence set (buffers sized by it, the small uploads, optionally the
    // initial parameters).  In a pipelined create it runs INSIDE seqset_build, between the metadata and the
    // rest of the codeword upload, so that none of it waits behind that upload.
    bool finished = false;
    std::function<int()> finish = [&]() -> int {
        finished = true;
        if (ltr_pipe) {  // the generic set only carries the sizes (see hmmb_bw.ltr_only)
            h->s.R = h->sl.R; h->s.frames = h->sl.frames; h->s.N = N; h->s.M = M; h->s.NP = pick_np(N);
            h->s.sym_bytes = M <= 256 ? 1 : 2;
            h->s.seq_begin = h->sl.seq_begin;
            h->s.tmax_all = h->sl.tmax_all;
        }
        HMMB_TRY(bw_finish_create(h, R));
        if (have_params) HMMB_TRY(bw_set_params_impl(h, pi0, A0, B0, false));
        return HMMB_OK;
    };
    if (ltr_pipe) {
        h->ltr_only = true;
        h->raw_idx_bytes = idx_bytes;
        h->bpieces = PIPE_STAGES;
        rc = seqset_build(h->sl, obs, idx_bytes, 0, offsets, word_of_seq, R, W, N, M, LAYOUT_LTR, true, &finish, PIPE_STAGES);
        if (rc != HMMB_OK) return fail(rc);
        if (h->bpieces_issued > 0 && (!h->sl.pend || h->bpieces_issued < h->bpieces)) {
            // no staged E-step will wait for the pieces one by one: order the compute stream behind the last one
            c.after_chunk = nullptr;
            if (h->bpieces_issued < h->bpieces) { set_error("parameter upload incomplete"); return fail(HMMB_ERR_CUDA); }
            cudaStreamWaitEvent(c.stream, h->bt_ready[h->bpieces - 1], 0);
        }
        if (!h->sl.pend) {
            // input not in (word, length descending) order: the build did the repack itself and its raw buffer is
            // gone, so the generic layout is built now, from the host codewords, as in a plain create
            h->ltr_only = false;
            rc = seqset_build(h->s, obs, idx_bytes, 0, offsets, word_of_seq, R, W, N, M, s_layout);
            if (rc != HMMB_OK) return fail(rc);
        } else {
            h->keep_offsets.assign(offsets, offsets + R + 1);
            h->keep_words.assign(word_of_seq, word_of_seq + R);
        }
    } else {
        const bool pipeline = (flags & HMMB_BW_PIPELINE_UPLOAD) != 0 && !h->has_ltr;
        rc = seqset_build(h->s, obs, idx_bytes, obs_on_device, offsets, word_of_seq, R, W, N, M, s_layout, pipeline,
                          pipeline ? &finish : nullptr, PIPE_STAGES);
        if (rc != HMMB_OK) return fail(rc);
        if (h->has_ltr) {
            rc = seqset_build(h->sl, obs, idx_bytes, obs_on_device, offsets, word_of_seq, R, W, N, M, LAYOUT_LTR);
            if (rc != HMMB_OK) return fail(rc);
            dev_free(h->d_raw);
            h->d_raw = nullptr;
        }
    }
    if (!finished) {
        rc = finish();
        if (rc != HMMB_OK) return fail(rc);
    }
    if (!h->s.pend && !h->sl.pend) {
        // (a pipelined create returns with its uploads in flight; otherwise everything is on the device now)
        cudaError_t e = cudaStreamSynchronize(c.stream);
        if (e != cudaSuccess) return fail(cuda_fail(e, "create sync", __FILE__, __LINE__));
    }
    *out = h;
    return HMMB_OK;
}

int hmmb_bw_destroy(hmmb_bw_t *h) {
    if (!h) return HMMB_OK;
    if (ctx().inited) cudaStreamSynchronize(ctx().stream);
    bw_release(h);
    delete h;
    return HMMB_OK;
}

int64_t hmmb_bw_total_frames(hmmb_bw_t *h) { return h ? h->s.frames : 0; }

const char *hmmb_bw_kernel_family(hmmb_bw_t *h) {
    if (!h) return "";
    if (h->use_ltr) return "left_to_right";
    if (h->s.layout == LAYOUT_N4) return h->bidiag ? "n4_left_to_right" : "n4_dense";
    return "generic";
}

// hmmb_bw.ltr_only and parameters with a dense A: build the generic layout now, from the raw codewords the handle kept.
static int bw_build_generic_lazily(hmmb_bw *h) {
    Ctx &c = ctx();
    if (h->sl.pend) {
        // no E-step has run yet: finish the deferred repack here, then take the raw buffer over
        PendingPrepare &p = *h->sl.pend;
        HMMB_CUDA(cudaStreamSynchronize(c.copy_stream));
        HMMB_TRY(launch_repack_range(h->sl, p.up->d_raw, p.idx_bytes, 0, h->sl.nblk, h->sl.d_bad));
        HMMB_CUDA(cudaStreamSynchronize(c.stream));
        h->d_raw = p.up->d_raw;
        p.up->d_raw = nullptr;
        h->sl.pend.reset();
        h->check_bad = true;
    } else if (h->pend_release) {
        HMMB_CUDA(cudaStreamSynchronize(c.stream));
        HMMB_TRY(bw_after_sync(h));
    }
    if (!h->d_raw) { set_error("dense transition matrices: the trainer no longer holds the raw codewords"); return HMMB_ERR_UNSUPPORTED; }
    const int64_t R = h->sl.R;
    HMMB_TRY(seqset_build(h->s, (const char *)h->d_raw - (size_t)h->keep_offsets[0] * h->raw_idx_bytes, h->raw_idx_bytes, 1,
                          h->keep_offsets.data(), h->keep_words.data(), R, h->W, h->N, h->M, LAYOUT_LANES));
    // (bw_finish_create sized the alpha spill for both layouts already)
    h->ltr_only = false;
    dev_free(h->d_raw);
    h->d_raw = nullptr;
    h->keep_offsets.clear(); h->keep_offsets.shrink_to_fit();
    h->keep_words.clear(); h->keep_words.shrink_to_fit();
    return HMMB_OK;
}

// sync == false (pipelined create): the parameters go through a pinned staging buffer so that the call
// neither blocks nor waits behind the codeword upload; everything stays ordered on the compute stream.
static int bw_set_params_impl(hmmb_bw *h, const double *pi0, const double *A0, const double *B0, bool sync) {
    Ctx &c = ctx();
    const int W = h->W, N = h->N, M = h->M;
    double *tmp = nullptr;
    const size_t nB = (size_t)W * N * M, nA = (size_t)W * N * N, nP = (size_t)W * N;
    HMMB_TRY(dev_alloc_t(&tmp, nB + nA + nP));
    bool pieces = false;
    if (h->d_ptmp) {  // parameters of a pipelined create still on their way: let them land before they are replaced
        HMMB_CUDA(cudaStreamSynchronize(c.copy_stream));
        bw_drop_pieces(h);
    }
    if (sync) {
        HMMB_TRY(h2d_big(tmp, B0, nB * sizeof(double), c.stream));
        HMMB_CUDA(cudaMemcpyAsync(tmp + nB, A0, nA * sizeof(double), cudaMemcpyHostToDevice, c.stream));
        HMMB_CUDA(cudaMemcpyAsync(tmp + nB + nA, pi0, nP * sizeof(double), cudaMemcpyHostToDevice, c.stream));
    } else {
        // Parts the caller holds in pinned memory go up straight from there (they must stay valid until the first
        // hmmb_bw_iterate returns, like the codewords of a pipelined create); the rest is staged.
        const bool pinB = nB * sizeof(double) >= (size_t(1) << 20) && host_is_pinned(B0);
        const bool pinA = pinB && host_is_pinned(A0), pinP = pinB && host_is_pinned(pi0);
        const size_t bytes = ((pinB ? 0 : nB) + (pinA ? 0 : nA) + (pinP ? 0 : nP)) * sizeof(double);
        if (c.pstage_busy) {
            cudaEventSynchronize(c.pstage_busy);
            event_put(c.pstage_busy);
            c.pstage_busy = nullptr;
        }
        if (c.pstage_bytes < bytes) {
            if (c.pstage) cudaFreeHost(c.pstage);
            c.pstage = nullptr;
            c.pstage_bytes = 0;
            if (cudaHostAlloc(&c.pstage, bytes, cudaHostAllocDefault) != cudaSuccess) {
                (void)cudaGetLastError();
                set_error("pinned staging allocation of %zu bytes failed", bytes);
                dev_free(tmp);
                return HMMB_ERR_OOM;
            }
            c.pstage_bytes = bytes;
        }
        double *ps = static_cast<double *>(c.pstage);
        auto put = [&](double *dst, const double *src, size_t n, bool pinned) -> int {
            if (pinned) return h2d_small(dst, src, n * sizeof(double));
            if (n * sizeof(double) >= (size_t(1) << 20)) par_memcpy(ps, src, n * sizeof(double));
            else memcpy(ps, src, n * sizeof(double));
            const int rc = h2d_small(dst, ps, n * sizeof(double));
            ps += n;
            return rc;
        };
        // Pipelined left-to-right create: B goes up in word ranges interleaved with the codeword chunks — piece 0
        // now, piece j behind the first chunk of stage j (EarlyUpload::issue calls the hook) — each followed on the
        // copy stream by its transposition kernel and an event, so that stage j of the first E-step only waits for
        // the B^T of its own words instead of for all 131 MB of config 4.
        pieces = h->ltr_only && c.h2d_on_copy && h->bpieces > 1 && W >= h->bpieces;
        double *psB = ps;
        if (!pieces) {
            HMMB_TRY(put(tmp, B0, nB, pinB));
        } else if (!pinB) {
            ps += nB;  // staged piece by piece (below)
        }
        HMMB_TRY(put(tmp + nB, A0, nA, pinA));
        HMMB_TRY(put(tmp + nB + nA, pi0, nP, pinP));
        if (pieces) {
            const int P = h->bpieces;
            HMMB_CUDA(cudaMemsetAsync(h->d_bzero, 0, (size_t)W * sizeof(int32_t), c.copy_stream));
            auto issue_piece = [h, tmp, B0, psB, pinB, P, W, N, M](int p) -> int {
                Ctx &c = ctx();
                const size_t w0 = (size_t)W * p / P, w1 = (size_t)W * (p + 1) / P, n = (w1 - w0) * N * M, o = w0 * N * M;
                const double *src = B0 + o;
                if (!pinB) {
                    par_memcpy(psB + o, B0 + o, n * sizeof(double));
                    src = psB + o;
                }
                HMMB_CUDA(cudaMemcpyAsync(tmp + o, src, n * sizeof(double), cudaMemcpyHostToDevice, c.copy_stream));
                cudaStream_t keep = c.stream;
                c.stream = c.copy_stream;  // (the launch macro uses the context's stream)
                struct Restore { Ctx &c; cudaStream_t s; ~Restore() { c.stream = s; } } restore{c, keep};
                dim3 gp((unsigned)std::min((N * M + 255) / 256, 64), (unsigned)(w1 - w0));
                HMMB_LAUNCH("bw_load", k_load_B, gp, 256, 0, tmp + o, N, M, h->d_Bt + o, h->d_bzero + w0);
                h->bt_ready[p] = event_get();
                HMMB_CUDA(cudaEventRecord(h->bt_ready[p], c.copy_stream));
                if (p == P - 1 && !pinB) {
                    c.pstage_busy = event_get();
                    HMMB_CUDA(cudaEventRecord(c.pstage_busy, c.copy_stream));
                }
                return HMMB_OK;
            };
            HMMB_TRY(issue_piece(0));
            h->bpieces_issued = 1;
            c.after_chunk = [h, issue_piece, P](int k, int nchunk) -> int {
                while (h->bpieces_issued < P && (k == nchunk - 1 || (int64_t)h->bpieces_issued * nchunk / P <= k))
                    HMMB_TRY(issue_piece(h->bpieces_issued++));
                return HMMB_OK;
            };
            if (bytes && pinB) {
                c.pstage_busy = event_get();
                HMMB_CUDA(cudaEventRecord(c.pstage_busy, c.copy_stream));
            }
        } else if (bytes) {
            c.pstage_busy = event_get();
            HMMB_CUDA(cudaEventRecord(c.pstage_busy, c.h2d_on_copy ? c.copy_stream : c.stream));
        }
        HMMB_TRY(h2d_join());  // the kernels below read tmp
    }
    if (!pieces) {
        dim3 gb((unsigned)std::min((N * M + 255) / 256, 64), (unsigned)W);
        HMMB_CUDA(cudaMemsetAsync(h->d_bzero, 0, (size_t)W * sizeof(int32_t), c.stream));
        HMMB_LAUNCH("bw_load", k_load_B, gb, 256, 0, tmp, N, M, h->d_Bt, h->d_bzero);
    }
    // upper-bidiagonal A (the reference's left-to-right default) selects the 7-term N = 4 kernels and the
    // left-to-right kernels for N = 8 / 16
    const Family fam = pick_family(N, M, A0, W);
    h->bidiag = fam.bidiag;
    h->full_spill = fam.full_spill;
    h->use_ltr = h->has_ltr && h->bidiag;
    if (h->ltr_only && !h->use_ltr) HMMB_TRY(bw_build_generic_lazily(h));
    HMMB_LAUNCH("bw_load", k_load_clamped, (unsigned)std::min<size_t>((nA + 255) / 256, 1024), 256, 0, tmp + nB, (int64_t)nA, h->d_A);
    HMMB_LAUNCH("bw_load", k_load_clamped, (unsigned)std::min<size_t>((nP + 255) / 256, 1024), 256, 0, tmp + nB + nA, (int64_t)nP, h->d_pi);
    HMMB_LAUNCH("bw_load", k_fill, (unsigned)((W + 255) / 256), 256, 0, h->d_prev, (int64_t)W, -INFINITY);
    HMMB_LAUNCH("bw_load", k_fill_i32, (unsigned)((W + 255) / 256), 256, 0, h->d_active, (int64_t)W, 1);
    HMMB_LAUNCH("bw_load", k_fill_i32, (unsigned)((W + 255) / 256), 256, 0, h->d_iters, (int64_t)W, 0);
    if (h->d_hist) HMMB_LAUNCH("bw_load", k_fill, 64, 256, 0, h->d_hist, (int64_t)W * h->hist_cap, (double)NAN);
    HMMB_CUDA(cudaMemsetAsync(h->d_flag_base, 0, (size_t)std::max<int64_t>(h->s.R, 1) + FLAG_HDR, c.stream));
    HMMB_CUDA(cudaMemsetAsync(h->d_newflags, 0, sizeof(int32_t), c.stream));
    HMMB_CUDA(cudaMemsetAsync(h->d_nexact, 0, sizeof(int64_t), c.stream));
    h->n_backward_handover = 0;
    // (new parameters: the thin-state flags of the old model go; the slot region keeps its allocation)
    HMMB_CUDA(cudaMemsetAsync(h->d_thinmask, 0, (size_t)W * sizeof(uint32_t), c.stream));
    HMMB_CUDA(cudaMemsetAsync(h->d_thin_new, 0, sizeof(int32_t), c.stream));
    HMMB_CUDA(cudaMemsetAsync(h->d_redo, 0, (size_t)W * sizeof(int32_t), c.stream));
    HMMB_CUDA(cudaMemsetAsync(h->d_slot_of, 0xff, (size_t)W * N * sizeof(int32_t), c.stream));
    h->n_slots = 0;
    h->n_thin_total = 0;
    if (sync) HMMB_CUDA(cudaStreamSynchronize(c.stream));
    if (pieces) h->d_ptmp = tmp;  // still the target of copies to come: released after the first E-step
    else dev_free(tmp);           // stream-ordered reuse: later users of the block are queued behind the kernels above
    h->params_set = true;
    h->any_active = true;
    return HMMB_OK;
}

int hmmb_bw_set_params(hmmb_bw_t *h, const double *pi0, const double *A0, const double *B0) {
    HMMB_TRY(require_init());
    if (!h || !pi0 || !A0 || !B0) { set_error("hmmb_bw_set_params: null argument"); return HMMB_ERR_ARG; }
    return bw_set_params_impl(h, pi0, A0, B0, true);
}

int hmmb_bw_set_dist(hmmb_bw_t *h, int rank, int world, hmmb_allreduce_fn allreduce, void *user) {
    HMMB_TRY(require_init());
    if (world > 1 && !allreduce) {  // no hook given: the library's own communicator, if one was created
        int cw = 1;
        hmmb_comm_rank(nullptr, &cw);
        if (cw == world) allreduce = hmmb_comm_allreduce;
    }
    if (!h || world < 1 || rank < 0 || rank >= world || (world > 1 && !allreduce)) {
        set_error("hmmb_bw_set_dist: bad arguments (rank=%d world=%d)", rank, world);
        return HMMB_ERR_ARG;
    }
    h->rank = rank; h->world = world; h->allreduce = allreduce; h->user = user;
    return bw_alloc_accum(h);
}

int hmmb_bw_set_overlap(hmmb_bw_t *h, int groups) {
    HMMB_TRY(require_init());
    if (!h || groups < 1 || groups > 64) { set_error("hmmb_bw_set_overlap: groups must be 1..64"); return HMMB_ERR_ARG; }
    h->overlap_groups = groups;
    return HMMB_OK;
}

static int bw_ensure_hist(hmmb_bw *h, int cap) {
    if (cap <= h->hist_cap) return HMMB_OK;
    Ctx &c = ctx();
    double *nh = nullptr;
    HMMB_TRY(dev_alloc_t(&nh, (size_t)h->W * cap));
    HMMB_LAUNCH("bw_load", k_fill, 64, 256, 0, nh, (int64_t)h->W * cap, (double)NAN);
    if (h->d_hist && h->hist_cap > 0)
        HMMB_CUDA(cudaMemcpy2DAsync(nh, cap * sizeof(double), h->d_hist, h->hist_cap * sizeof(double),
                                    h->hist_cap * sizeof(double), h->W, cudaMemcpyDeviceToDevice, c.stream));
    HMMB_CUDA(cudaStreamSynchronize(c.stream));
    dev_free(h->d_hist);
    h->d_hist = nh;
    h->hist_cap = cap;
    return HMMB_OK;
}

template <typename SymT, bool BLOCKED>
static int launch_exact(hmmb_bw *h) {
    SeqSet &s = h->cur();
    HMMB_LAUNCH("bw_exact", (k_bw_exact<SymT, BLOCKED>), h->exact_grid, BW_THREADS, 0, s.d_obs, BLOCKED ? s.d_foff : s.d_off,
                s.d_len, s.d_word, s.R, h->N, h->M, h->d_pi, h->d_A, h->d_Bt, h->d_llseq, h->act_cur, h->d_flag,
                h->d_exact_scratch, h->exact_stride, h->d_accum, h->astride, h->d_nexact, SYM_MASK);
    return HMMB_OK;
}

template <int NP, typename SymT>
static int launch_generic_estep(hmmb_bw *h) {
    SeqSet &s = h->s;
    const LanesGrid g = lanes_grid(s.R, NP);
    HMMB_LAUNCH("bw_forward", (k_bw_fwdG<NP, SymT>), g.grid, BW_THREADS, 0, (const SymT *)s.d_obs, s.d_off, s.d_len,
                s.d_word, s.d_foff, s.R, g.per_group, h->N, h->M, h->d_pi, h->d_A, h->d_Bt, h->d_spill, h->d_llseq,
                h->act_cur, h->d_flag);
    HMMB_TRY((launch_exact<SymT, false>(h)));
    HMMB_LAUNCH("bw_backward", (k_bw_bwdG<NP, SymT>), g.grid, BW_THREADS, 0, (const SymT *)s.d_obs, s.d_off, s.d_len,
                s.d_word, s.d_foff, s.R, g.per_group, h->N, h->M, h->d_A, h->d_Bt, h->d_spill, h->d_llseq, h->act_cur,
                h->d_accum, h->astride, h->d_flag, h->d_newflags);
    return HMMB_OK;
}

// First E-step of a pipelined fit on the blocked layout s (N = 4 or left-to-right): stage j = the blocks whose codewords
// have landed (copy-stream event), repacked and pushed through forward + backward while the next chunks are still on
// PCIe.  A stage is a fraction of a wave of CTAs, so consecutive stages go to two alternating side streams: the next
// stage's repack and forward pass fill the SMs that the tail of this stage's backward pass leaves idle.  Everything a
// stage writes (blocked codewords, spill, per-sequence results, per-CTA partials or fp64 atomics into the accumulators)
// is private to its blocks; the compute stream joins both side streams afterwards.  stage(c0, c1) launches the work
// items [c0, c1) on the context's stream.  Sequences the forward passes handed over are redone by the exact kernel after
// the stages (their accumulator contributions are independent of the backward pass).
template <typename StageFn>
static int run_staged_estep(hmmb_bw *h, SeqSet &s, StageFn &&stage) {
    Ctx &c = ctx();
    PendingPrepare &p = *s.pend;
    int bdone = 0, cdone = 0;
    cudaStream_t main_stream = c.stream;
    const bool side = p.nstage > 2;
    struct Restore { Ctx &c; cudaStream_t s; ~Restore() { c.stream = s; } } restore{c, main_stream};
    if (side) {
        cudaEvent_t fork = event_get();
        HMMB_CUDA(cudaEventRecord(fork, main_stream));
        for (auto st : c.stage_stream) HMMB_CUDA(cudaStreamWaitEvent(st, fork, 0));
        event_put(fork);
    }
    for (int j = 0; j < p.nstage; ++j) {
        if (side) c.stream = c.stage_stream[j & 1];
        HMMB_CUDA(cudaStreamWaitEvent(c.stream, p.up->ev[p.ev_index[j]], 0));
        HMMB_TRY(launch_repack_range(s, p.up->d_raw, p.idx_bytes, bdone, p.blk_end[j], s.d_bad));
        if (p.cta_end[j] > cdone) HMMB_TRY(stage(cdone, p.cta_end[j]));
        bdone = p.blk_end[j];
        cdone = p.cta_end[j];
    }
    c.stream = main_stream;
    if (side) {
        for (auto st : c.stage_stream) {
            cudaEvent_t join = event_get();
            HMMB_CUDA(cudaEventRecord(join, st));
            HMMB_CUDA(cudaStreamWaitEvent(main_stream, join, 0));
            event_put(join);
        }
    }
    h->check_bad = true;
    h->pend_release = std::move(s.pend);  // raw buffer + events: released after the next stream sync
    HMMB_TRY((launch_exact<uint16_t, true>(h)));
    return HMMB_OK;
}

// warps of the fat backward CTA and its dynamic shared memory: B^T (replicated REP times), one count table per warp,
// the gamma_0 sums; as many warps as fit beside the kernel's static arrays (sRed, the codeword slots: ~19 KB)
static int bwd4_warps(int M, int rep, bool bidiag, size_t smem_optin, size_t *smem) {
    int nw = bidiag ? BWD4_MAX_WARPS : 12;
    auto bytes = [&](int w) { return (size_t)M * rep * 4 * sizeof(double) + (size_t)w * M * 4 * sizeof(double) + (size_t)w * 4 * sizeof(double); };
    const size_t avail = smem_optin > 20 * 1024 ? smem_optin - 20 * 1024 : 0;
    while (nw > 1 && bytes(nw) > avail) --nw;
    *smem = bytes(nw);
    return nw;
}

template <bool BIDIAG, int MT, int REP>
static int launch_special_estep(hmmb_bw *h) {
    Ctx &c = ctx();
    SeqSet &s = h->s;
    if (s.ncta == 0) { s.pend.reset(); return HMMB_OK; }
    const size_t smem_f = (size_t)h->M * 5 * sizeof(double) + (size_t)((h->M + 15) & ~15);
    size_t smem_b = 0;
    const int bwd_threads = 32 * bwd4_warps(h->M, REP, BIDIAG, c.smem_optin, &smem_b);
    HMMB_CUDA(cudaFuncSetAttribute((k_bw_bwd4<BIDIAG, MT, REP>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b));
    // forward / backward pass over the CTA work items [c0, c1) of `list`
    auto fwd = [&](const CtaWork *list, int c0, int c1) -> int {
        HMMB_LAUNCH("bw_forward", k_bw_fwd4<BIDIAG>, (c1 - c0) * FWD4_SPLIT, BW_THREADS, smem_f, list + c0, s.d_blks,
                    (const uint4 *)s.d_obs, s.d_len, h->d_pi, h->d_A, h->d_Bt, h->M, spill4(h), h->d_llseq, h->act_cur,
                    h->d_flag, h->d_allfull, FWD4_SPLIT, SYM_MASK, oddmask4(h), h->full_spill);
        return HMMB_OK;
    };
    auto bwd = [&](const CtaWork *list, int c0, int c1) -> int {
        HMMB_LAUNCH("bw_backward", (k_bw_bwd4<BIDIAG, MT, REP>), c1 - c0, bwd_threads, smem_b, list + c0, s.d_blks,
                    (const uint4 *)s.d_obs, s.d_len, h->d_A, h->d_Bt, h->M, spill4(h), h->d_llseq, h->act_cur, h->d_bzero,
                    h->d_allfull, h->d_partials + (size_t)c0 * h->pstride, h->pstride, h->d_flag, h->d_newflags,
                    oddmask4(h), h->full_spill);
        return HMMB_OK;
    };
    if (s.pend) {
        // the staged E-step launches from the finer work list where it exists
        const CtaWork *stage_work = s.ncta_fine > 0 ? s.d_work_fine : s.d_work;
        const int stage_ncta = s.ncta_fine > 0 ? s.ncta_fine : s.ncta;
        HMMB_TRY(run_staged_estep(h, s, [&](int c0, int c1) -> int {
            HMMB_TRY(fwd(stage_work, c0, c1));
            return bwd(stage_work, c0, c1);
        }));
        // the per-CTA statistic, taken inside k_bw_bwd4 while the sequences the exact kernel redid still carried their
        // NaN mark, is retaken
        HMMB_LAUNCH("bw_exact", k_bw_llstat_fix, stage_ncta, BW_THREADS, 0, stage_work, s.d_blks, h->d_llseq, h->act_cur,
                    h->d_flag, h->d_partials, h->pstride, h->M);
        h->estep_fine = s.ncta_fine > 0;  // k_bw_reduce sums this E-step's partials over the finer list's per-word ranges
        return HMMB_OK;
    }
    h->estep_fine = false;
    HMMB_TRY(s.ncta_fwd ? fwd(s.d_work_fwd, 0, s.ncta_fwd) : fwd(s.d_work, 0, s.ncta));
    HMMB_TRY((launch_exact<uint16_t, true>(h)));
    return bwd(s.d_work, 0, s.ncta);
}

template <int NS>
static int launch_ltr_estep(hmmb_bw *h) {
    SeqSet &s = h->sl;
    if (s.ncta == 0) return HMMB_OK;
    const int M = h->M;
    const size_t smem_f = (size_t)M * NS * 8 + (size_t)M * 8 + (size_t)M * 2;
    const size_t smem_b = (size_t)M * NS * 8 + (size_t)LTR_WARPS * 32 * Ltr<NS>::ROWB + (size_t)2 * NS * 8 +
                          (size_t)LTR_WARPS * 2 * NS * 8;
    HMMB_CUDA(cudaFuncSetAttribute(k_bw_fwdL<NS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_f));
    HMMB_CUDA(cudaFuncSetAttribute(k_bw_bwdL<NS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b));
    // forward / backward pass over the CTA work items [c0, c1)
    auto fwd = [&](int c0, int c1) -> int {
        HMMB_LAUNCH("bw_forward", k_bw_fwdL<NS>, c1 - c0, LTR_THREADS, smem_f, s.d_work + c0, s.d_blks, (const uint4 *)s.d_obs,
                    s.d_len, h->d_pi, h->d_A, h->d_Bt, M, (double2 *)h->d_spill, h->d_llseq, h->act_cur, h->d_flag,
                    h->d_allfull);
        return HMMB_OK;
    };
    auto bwd = [&](int c0, int c1) -> int {
        HMMB_LAUNCH("bw_backward", k_bw_bwdL<NS>, c1 - c0, LTR_THREADS, smem_b, s.d_work + c0, s.d_blks, (const uint4 *)s.d_obs,
                    s.d_len, h->d_A, h->d_Bt, M, (const double2 *)h->d_spill, h->d_llseq, h->act_cur, h->d_bzero,
                    h->d_allfull, h->d_accum, h->astride, h->d_flag, h->d_newflags);
        return HMMB_OK;
    };
    if (s.pend) {
        // the accumulators take fp64 atomics from every stage and the convergence statistic is taken from the
        // per-sequence values by k_bw_reduce afterwards, so nothing has to be retaken after the exact kernel
        return run_staged_estep(h, s, [&](int c0, int c1) -> int {
            if (h->bpieces_issued > 0) {
                // B^T of this stage's words (pieces are word ranges [W p / P, W (p + 1) / P), ready in order)
                const int w_last = (int)(std::upper_bound(s.cta_begin.begin(), s.cta_begin.end(), c1 - 1) - s.cta_begin.begin()) - 1;
                int need = 0;
                while (need < h->bpieces - 1 && (int64_t)h->W * (need + 1) / h->bpieces <= w_last) ++need;
                HMMB_CUDA(cudaStreamWaitEvent(ctx().stream, h->bt_ready[need], 0));
            }
            HMMB_TRY(fwd(c0, c1));
            return bwd(c0, c1);
        });
    }
    HMMB_TRY(fwd(0, s.ncta));
    HMMB_TRY((launch_exact<uint16_t, true>(h)));
    const int groups = (h->allreduce && h->world > 1) ? std::min(h->overlap_groups, h->W) : 1;
    if (groups <= 1) return bwd(0, s.ncta);
    // Communication / compute overlap (config 4: 133 MB of accumulators per iteration).  The convergence
    // statistic and the sequence counts only need the forward pass, so k_bw_reduce runs first; the backward
    // pass then goes word group by word group, and each group's slice of the accumulator buffer is handed to the
    // all-reduce hook as soon as its kernels are queued — the hook runs it on a side stream while the next
    // group's backward pass computes.  hook(NULL, 0) at the end joins the side stream.
    HMMB_LAUNCH("bw_reduce", k_bw_reduce, dim3((unsigned)h->W, 1u), RED_THREADS, 0, (const double *)nullptr, h->pstride,
                h->d_cta_begin, h->d_llseq, h->d_seq_begin, h->d_accum, h->astride, h->nacc,
                h->d_accum + (size_t)h->W * h->astride, h->rank, h->W, h->act_cur);
    for (int g = 0; g < groups; ++g) {
        const int w0 = (int)((int64_t)h->W * g / groups), w1 = (int)((int64_t)h->W * (g + 1) / groups);
        const int c0 = s.cta_begin[w0], c1 = s.cta_begin[w1];
        if (c1 > c0) HMMB_TRY(bwd(c0, c1));
        int rc = h->allreduce(h->d_accum + (size_t)w0 * h->astride, (int64_t)(w1 - w0) * h->astride, h->user);
        if (rc != 0) { set_error("allreduce hook failed (%d)", rc); return HMMB_ERR_CUDA; }
    }
    int rc = h->allreduce(h->d_accum + (size_t)h->W * h->astride, (int64_t)h->world * h->W * 2, h->user);  // LL statistics
    if (rc == 0) rc = h->allreduce(nullptr, 0, h->user);                                                     // join
    if (rc != 0) { set_error("allreduce hook failed (%d)", rc); return HMMB_ERR_CUDA; }
    h->estep_reduced = true;
    return HMMB_OK;
}

static int bw_estep(hmmb_bw *h) {
    if (h->use_ltr) return h->N == 16 ? launch_ltr_estep<16>(h) : launch_ltr_estep<8>(h);
    SeqSet &s = h->s;
    if (s.layout == LAYOUT_N4) {
        if (h->M == 256) return h->bidiag ? launch_special_estep<true, 256, BWD4_REP>(h) : launch_special_estep<false, 256, BWD4_REP>(h);
        if (h->M < 256) return h->bidiag ? launch_special_estep<true, 0, BWD4_REP>(h) : launch_special_estep<false, 0, BWD4_REP>(h);
        return h->bidiag ? launch_special_estep<true, 0, 1>(h) : launch_special_estep<false, 0, 1>(h);
    }
    return with_lanes(s, [&](auto np, auto sym) { return launch_generic_estep<decltype(np)::value, decltype(sym)>(h); });
}

// Called right after a cudaStreamSynchronize of the compute stream: the pipelined prepare's upload
// state can go, and its codeword-range flag is read back (the check hmmb_bw_create makes itself when
// it does the repack).
static int bw_after_sync(hmmb_bw *h) {
    if (h->pend_release && h->ltr_only && h->pend_release->up && !h->d_raw) {
        // the raw codewords stay with the handle (lazy generic layout, see hmmb_bw.ltr_only)
        cudaStreamSynchronize(ctx().copy_stream);
        h->d_raw = h->pend_release->up->d_raw;
        h->pend_release->up->d_raw = nullptr;
    }
    h->pend_release.reset();
    if (h->d_ptmp && !h->sl.pend) bw_drop_pieces(h);  // (the first E-step has consumed them)
    if (h->check_bad) {
        h->check_bad = false;
        int bad = 0;
        HMMB_CUDA(cudaMemcpy(&bad, (h->ltr_only ? h->sl : h->s).d_bad, sizeof(int), cudaMemcpyDeviceToHost));
        if (bad) {
            set_error("codeword out of range: some observation is >= M=%d (reference: IndexError)", h->M);
            return HMMB_ERR_RANGE;
        }
    }
    return HMMB_OK;
}

// ---- thin-state rescue, host side (device side: hmm_device.cuh / bw_kernels.cuh)
static double *rescue_base(hmmb_bw *h) { return h->d_accum + (size_t)h->W * h->astride + (size_t)h->world * h->W * 2; }

// log-space pass over the sequences of the words with flagged states (after the E-step, before the reduce)
static int launch_rescue(hmmb_bw *h) {
    if (h->n_slots == 0) return HMMB_OK;
    SeqSet &s = h->cur();
    double *own = rescue_base(h) + (size_t)h->rank * h->slot_cap * h->rstride;
    const int64_t n = h->slot_cap * h->rstride;
    HMMB_LAUNCH("bw_rescue", k_bw_rescue_init, (unsigned)std::min<int64_t>((n + 255) / 256, 1024), 256, 0, own, n);
    return with_codewords(s, [&](auto sym, auto blocked) -> int {
        HMMB_LAUNCH("bw_rescue", (k_bw_rescue<decltype(sym), decltype(blocked)::value>), h->exact_grid, BW_THREADS, 0, s.d_obs,
                    blocked() ? s.d_foff : s.d_off, s.d_len, s.d_word, s.R, h->N, h->M, h->d_pi, h->d_A, h->d_Bt, h->act_cur,
                    h->d_exact_scratch, h->exact_stride, h->d_thinmask, h->d_slot_of, own, h->rstride, SYM_MASK);
        return HMMB_OK;
    });
}

// Called after a stream synchronisation with the number of states the M-step has newly flagged: gives every flagged
// state a slot — numbered by (word, state), the same on every rank because the flags derive from the all-reduced
// sums — and grows the slot region behind the accumulators if needed.
static int bw_assign_slots(hmmb_bw *h) {
    Ctx &c = ctx();
    const int W = h->W, N = h->N;
    std::vector<uint32_t> mask((size_t)W);
    HMMB_CUDA(cudaMemcpy(mask.data(), h->d_thinmask, (size_t)W * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    std::vector<int32_t> slot_of((size_t)W * N, -1);
    int n = 0;
    for (int w = 0; w < W; ++w)
        for (int i = 0; i < N; ++i)
            if ((mask[w] >> i) & 1u) slot_of[(size_t)w * N + i] = n++;
    h->n_slots = n;
    h->n_thin_total = n;
    if (n > h->slot_cap) {
        h->slot_cap = ((int64_t)n + 15) & ~int64_t(15);
        HMMB_CUDA(cudaStreamSynchronize(c.stream));
        HMMB_TRY(bw_alloc_accum(h));
    }
    HMMB_CUDA(cudaMemcpy(h->d_slot_of, slot_of.data(), slot_of.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    HMMB_CUDA(cudaMemsetAsync(h->d_thin_new, 0, sizeof(int32_t), c.stream));
    return HMMB_OK;
}

// E-step (+ rescue pass) + reduce + all-reduce + M-step over the words of `mask`
static int bw_one_pass(hmmb_bw *h, int32_t *mask, double eps, int max_iter, int sync_each, int skip_new_thin) {
    Ctx &c = ctx();
    h->act_cur = mask;
    struct Restore { hmmb_bw *h; ~Restore() { h->act_cur = h->d_active; } } restore{h};
    for (int attempt = 0; attempt < 2; ++attempt) {
        HMMB_CUDA(cudaMemsetAsync(h->d_accum, 0, (size_t)h->accum_n * sizeof(double), c.stream));
        h->estep_reduced = false;
        HMMB_TRY(bw_estep(h));
        // (an E-step that already ran its collectives cannot be redone by one rank alone: backward-pass
        // hand-overs then only take effect from the next iteration, as with sync_each == 0)
        if (!sync_each || h->estep_reduced) break;
        // backward-pass hand-overs are discovered after their sequence already contributed:
        // redo this E-step once with them routed to the exact kernel (flags are sticky)
        int32_t nf = 0;
        HMMB_CUDA(cudaMemcpyAsync(&nf, h->d_newflags, sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
        HMMB_CUDA(cudaStreamSynchronize(c.stream));
        HMMB_TRY(bw_after_sync(h));
        if (nf == 0) break;
        h->n_backward_handover += nf;
        HMMB_CUDA(cudaMemsetAsync(h->d_newflags, 0, sizeof(int32_t), c.stream));
    }
    HMMB_TRY(launch_rescue(h));
    if (!h->estep_reduced) {
        const bool n4 = h->s.layout == LAYOUT_N4;  // the N = 4 E-step leaves per-CTA partials
        const dim3 rgrid((unsigned)h->W, n4 ? (unsigned)((h->nacc + RED_EX - 1) / RED_EX) : 1u);
        HMMB_LAUNCH("bw_reduce", k_bw_reduce, rgrid, RED_THREADS, 0, n4 ? h->d_partials : nullptr, h->pstride,
                    (n4 && h->estep_fine) ? h->d_cta_begin_fine : h->d_cta_begin, h->d_llseq, h->d_seq_begin, h->d_accum, h->astride, h->nacc,
                    h->d_accum + (size_t)h->W * h->astride, h->rank, h->W, mask);
        if (h->allreduce && h->world > 1) {
            static int pid_ar = -1;
            if (pid_ar < 0) pid_ar = phase_id("bw_allreduce");
            if (c.profiling) phase_begin(pid_ar);  // CUDA events around the collective on the launching stream
            int rc = h->allreduce(h->d_accum, h->accum_n, h->user);
            if (c.profiling) phase_end(pid_ar);
            if (rc != 0) { set_error("allreduce hook failed (%d)", rc); return HMMB_ERR_CUDA; }
        }
    } else if (h->n_slots > 0 && h->allreduce && h->world > 1) {
        // (the overlapping E-step has reduced the word slices and the statistics itself: the slot region is left)
        int rc = h->allreduce(rescue_base(h), (int64_t)h->world * h->slot_cap * h->rstride, h->user);
        if (rc == 0) rc = h->allreduce(nullptr, 0, h->user);
        if (rc != 0) { set_error("allreduce hook failed (%d)", rc); return HMMB_ERR_CUDA; }
    }
    HMMB_CUDA(cudaMemsetAsync(h->d_redo, 0, (size_t)h->W * sizeof(int32_t), c.stream));
    HMMB_LAUNCH("bw_mstep", k_bw_mstep, h->W, RED_THREADS, 0, h->d_accum, h->astride,
                h->d_accum + (size_t)h->W * h->astride, h->world, h->W, h->N, h->M, h->d_pi, h->d_A, h->d_Bt,
                mask, h->d_active, h->d_iters, h->d_prev, h->d_hist, h->hist_cap, eps, max_iter, h->d_any, h->d_bzero,
                h->d_thinmask, h->d_thin_new, h->d_redo, skip_new_thin, h->d_slot_of, rescue_base(h), h->slot_cap, h->rstride,
                THIN_LIMIT);
    return HMMB_OK;
}

int hmmb_bw_iterate(hmmb_bw_t *h, int n_iter, double eps, int max_iter, int sync_each) {
    HMMB_TRY(require_init());
    if (!h || !h->params_set) { set_error("hmmb_bw_iterate: parameters not set"); return HMMB_ERR_ARG; }
    Ctx &c = ctx();
    HMMB_TRY(bw_ensure_hist(h, std::min(std::max(max_iter, 1), 1 << 16)));  // history keeps at most 65536 iterations
    for (int it = 0; it < n_iter; ++it) {
        if (!h->any_active) break;
        HMMB_CUDA(cudaMemsetAsync(h->d_any, 0, sizeof(int32_t), c.stream));
        // with sync_each a word whose M-step finds a newly thin state is held back (its parameters, iteration count
        // and history untouched) and the iteration is repeated for those words with the state's slot in place
        HMMB_TRY(bw_one_pass(h, h->d_active, eps, max_iter, sync_each, sync_each ? 1 : 0));
        if (sync_each) {
            int32_t any = 0, nt = 0;
            HMMB_CUDA(cudaMemcpyAsync(&any, h->d_any, sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
            HMMB_CUDA(cudaMemcpyAsync(&nt, h->d_thin_new, sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
            HMMB_CUDA(cudaStreamSynchronize(c.stream));
            HMMB_TRY(bw_after_sync(h));
            // (a repeat can flag further states of the words it runs on — they are held back again; the flags only
            // grow, at most N per word, so this ends)
            for (int guard = 0; nt > 0 && guard <= HMMB_MAX_STATES; ++guard) {
                HMMB_TRY(bw_assign_slots(h));
                HMMB_CUDA(cudaMemcpyAsync(h->d_redo_in, h->d_redo, (size_t)h->W * sizeof(int32_t), cudaMemcpyDeviceToDevice, c.stream));
                HMMB_TRY(bw_one_pass(h, h->d_redo_in, eps, max_iter, sync_each, 1));
                HMMB_CUDA(cudaMemcpyAsync(&any, h->d_any, sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
                HMMB_CUDA(cudaMemcpyAsync(&nt, h->d_thin_new, sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
                HMMB_CUDA(cudaStreamSynchronize(c.stream));
                HMMB_TRY(bw_after_sync(h));
            }
            h->any_active = any != 0;
        }
    }
    if (!sync_each && n_iter > 0) {
        int32_t any = 0, nt = 0;
        HMMB_CUDA(cudaMemcpyAsync(&any, h->d_any, sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
        HMMB_CUDA(cudaMemcpyAsync(&nt, h->d_thin_new, sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
        HMMB_CUDA(cudaStreamSynchronize(c.stream));
        HMMB_TRY(bw_after_sync(h));
        h->any_active = any != 0;
        // states flagged while the iterations were queued: their slots exist from the next call on
        if (nt > 0) HMMB_TRY(bw_assign_slots(h));
    }
    return HMMB_OK;
}

int hmmb_bw_thin_states(hmmb_bw_t *h, int64_t *n_states) {
    HMMB_TRY(require_init());
    if (!h || !n_states) { set_error("hmmb_bw_thin_states: null argument"); return HMMB_ERR_ARG; }
    *n_states = h->n_thin_total;
    return HMMB_OK;
}

int hmmb_bw_get_params(hmmb_bw_t *h, int finalize, double *pi, double *A, double *B) {
    HMMB_TRY(require_init());
    if (!h || !h->params_set) { set_error("hmmb_bw_get_params: parameters not set"); return HMMB_ERR_ARG; }
    Ctx &c = ctx();
    const int W = h->W, N = h->N, M = h->M;
    const size_t nB = (size_t)W * N * M, nA = (size_t)W * N * N, nP = (size_t)W * N;
    double *tmp = nullptr;
    HMMB_TRY(dev_alloc_t(&tmp, nB + nA + nP));
    HMMB_LAUNCH("bw_finalize", k_bw_finalize, W, RED_THREADS, 0, h->d_pi, h->d_A, h->d_Bt, N, M, finalize, tmp + nB + nA,
                tmp + nB, tmp);
    if (B) HMMB_TRY(d2h_big(B, tmp, nB * sizeof(double), c.stream));
    if (A) HMMB_CUDA(cudaMemcpyAsync(A, tmp + nB, nA * sizeof(double), cudaMemcpyDeviceToHost, c.stream));
    if (pi) HMMB_CUDA(cudaMemcpyAsync(pi, tmp + nB + nA, nP * sizeof(double), cudaMemcpyDeviceToHost, c.stream));
    HMMB_CUDA(cudaStreamSynchronize(c.stream));
    dev_free(tmp);
    return HMMB_OK;
}

int hmmb_bw_get_history(hmmb_bw_t *h, double *ll_hist, int hist_cap, int32_t *iters) {
    HMMB_TRY(require_init());
    if (!h) { set_error("hmmb_bw_get_history: null handle"); return HMMB_ERR_ARG; }
    Ctx &c = ctx();
    if (ll_hist && hist_cap > 0) {
        for (int64_t e = 0; e < (int64_t)h->W * hist_cap; ++e) ll_hist[e] = NAN;
        const int ncopy = std::min(hist_cap, h->hist_cap);
        if (ncopy > 0 && h->d_hist)
            HMMB_CUDA(cudaMemcpy2DAsync(ll_hist, hist_cap * sizeof(double), h->d_hist, h->hist_cap * sizeof(double),
                                        ncopy * sizeof(double), h->W, cudaMemcpyDeviceToHost, c.stream));
    }
    if (iters) HMMB_CUDA(cudaMemcpyAsync(iters, h->d_iters, h->W * sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
    HMMB_CUDA(cudaStreamSynchronize(c.stream));
    return HMMB_OK;
}

int hmmb_bw_diagnostics(hmmb_bw_t *h, int64_t *exact_sequence_passes, int64_t *backward_handovers) {
    HMMB_TRY(require_init());
    if (!h) { set_error("hmmb_bw_diagnostics: null handle"); return HMMB_ERR_ARG; }
    Ctx &c = ctx();
    int64_t ne = 0;
    int32_t nf = 0;
    HMMB_CUDA(cudaMemcpyAsync(&ne, h->d_nexact, sizeof(int64_t), cudaMemcpyDeviceToHost, c.stream));
    HMMB_CUDA(cudaMemcpyAsync(&nf, h->d_newflags, sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
    HMMB_CUDA(cudaStreamSynchronize(c.stream));
    if (exact_sequence_passes) *exact_sequence_passes = ne;
    if (backward_handovers) *backward_handovers = h->n_backward_handover + nf;
    return HMMB_OK;
}

int hmmb_bw_get_seq_ll(hmmb_bw_t *h, double *ll_seq) {
    HMMB_TRY(require_init());
    if (!h || !ll_seq) { set_error("hmmb_bw_get_seq_ll: null argument"); return HMMB_ERR_ARG; }
    Ctx &c = ctx();
    std::vector<double> tmp((size_t)h->s.R);
    if (h->s.R > 0) {
        HMMB_CUDA(cudaMemcpyAsync(tmp.data(), h->d_llseq, h->s.R * sizeof(double), cudaMemcpyDeviceToHost, c.stream));
        HMMB_CUDA(cudaStreamSynchronize(c.stream));
    }
    const std::vector<int32_t> &order = h->cur().order;  // empty = identity
    for (int64_t i = 0; i < h->s.R; ++i) ll_seq[order.empty() ? i : order[i]] = tmp[i];
    return HMMB_OK;
}

int hmmb_bw_fit(const void *obs, int idx_bytes, const int64_t *offsets, const int32_t *word_of_seq, int64_t R, int W,
                int N, int M, const double *pi0, const double *A0, const double *B0, double eps, int max_iter,
                double *pi, double *A, double *B, double *ll_hist, int32_t *iters) {
    hmmb_bw_t *h = nullptr;
    if (!pi0 || !A0 || !B0) { set_error("hmmb_bw_fit: null parameters"); return HMMB_ERR_ARG; }
    HMMB_TRY(hmmb_bw_create_ex(&h, obs, idx_bytes, 0, offsets, word_of_seq, R, W, N, M, HMMB_BW_PIPELINE_UPLOAD, pi0, A0, B0));
    int rc = HMMB_OK;
    if (rc == HMMB_OK) rc = hmmb_bw_iterate(h, max_iter, eps, max_iter, 1);
    if (rc == HMMB_OK) rc = hmmb_bw_get_params(h, 1, pi, A, B);
    if (rc == HMMB_OK && (ll_hist || iters)) rc = hmmb_bw_get_history(h, ll_hist, std::max(max_iter, 1), iters);
    hmmb_bw_destroy(h);
    return rc;
}

// ---------------------------------------------------------------- recognition
// The sequence set and device buffers of one hmmb_score / hmmb_viterbi call, released however the call returns.
struct CallGuard {
    SeqSet &s;
    std::vector<void *> ptrs;
    ~CallGuard() { s.release(); for (void *p : ptrs) dev_free(p); }
};

template <int NP, typename SymT>
static int launch_score_generic(SeqSet &s, int W, const double *d_pi, const double *d_A, const double *d_Bt, double *d_ll, int32_t *d_nan) {
    const LanesGrid lg = lanes_grid(s.R, NP);
    dim3 g(lg.grid, (unsigned)W);
    HMMB_LAUNCH("score", (k_scoreG<NP, SymT>), g, BW_THREADS, 0, (const SymT *)s.d_obs, s.d_off, s.d_len, s.d_order, s.R,
                lg.per_group, s.N, s.M, W, d_pi, d_A, d_Bt, d_ll, d_nan);
    return HMMB_OK;
}

// N = 4 scorers over the blocks [b0, b1) (a stage of the pipelined scorer, or all of them); bidiag: every A is
// upper-bidiagonal
static int launch_score_special(SeqSet &s, bool bidiag, int W, const double *d_pi, const double *d_A, const double *d_Bt,
                                double *d_ll, int32_t *d_nan, int b0, int b1) {
    Ctx &c = ctx();
    const int nb = b1 - b0;
    if (nb <= 0) return HMMB_OK;
    // both scorers have one signature; [BIDIAG][VECB] picks the instance
    using Score4 = decltype(&k_score4<false, false>);
    const bool vecb = s.tmax_all > SCORE4_SCALAR_BOUND_MAX_T;
    if (s.M <= SCORE4R_MAX_M) {
        const Score4 k[2][2] = {{k_score4r<false, false>, k_score4r<false, true>}, {k_score4r<true, false>, k_score4r<true, true>}};
        // replicated-B scorer: 8 warps per CTA, 2 CTAs per SM, about six waves of CTAs
        int bpc = std::max(SCORE4R_WARPS, (int)(((int64_t)nb * W + c.sm_count * 12 - 1) / (c.sm_count * 12)));
        bpc = (bpc + SCORE4R_WARPS - 1) / SCORE4R_WARPS * SCORE4R_WARPS;
        bpc = std::min(bpc, 128);
        dim3 g((unsigned)((nb + bpc - 1) / bpc), (unsigned)W);
        const size_t smem = (size_t)SCORE4R_MAX_M * SCORE4R_REP * 2 * sizeof(double2) + (size_t)s.M * sizeof(double) + (size_t)((s.M + 15) & ~15);
        HMMB_CUDA(cudaFuncSetAttribute(k[bidiag][vecb], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        HMMB_LAUNCH("score", k[bidiag][vecb], g, SCORE4R_WARPS * 32, smem, s.d_blks + b0, nb, bpc, (const uint4 *)s.d_obs,
                    s.d_len, s.d_order, d_pi, d_A, d_Bt, s.M, W, d_ll, d_nan);
        return HMMB_OK;
    }
    const Score4 k[2][2] = {{k_score4<false, false>, k_score4<false, true>}, {k_score4<true, false>, k_score4<true, true>}};
    // each CTA re-uses one model's B for several 32-utterance blocks
    int bpc = std::max(BW_WARPS, (s.nblk * W + c.sm_count * 16 - 1) / (c.sm_count * 16));
    bpc = (bpc + BW_WARPS - 1) / BW_WARPS * BW_WARPS;
    bpc = std::min(bpc, 64);
    dim3 g((unsigned)((nb + bpc - 1) / bpc), (unsigned)W);
    const size_t smem = (size_t)s.M * 5 * sizeof(double) + (size_t)((s.M + 15) & ~15);
    HMMB_LAUNCH("score", k[bidiag][vecb], g, BW_THREADS, smem, s.d_blks + b0, nb, bpc, (const uint4 *)s.d_obs, s.d_len,
                s.d_order, d_pi, d_A, d_Bt, s.M, W, d_ll, d_nan);
    return HMMB_OK;
}

template <int NS>
static int launch_score_ltr(SeqSet &s, int W, const double *d_pi, const double *d_A, const double *d_Bt, double *d_ll, int32_t *d_nan) {
    if (s.ncta == 0) return HMMB_OK;
    const size_t smem = (size_t)s.M * NS * 8 + (size_t)s.M * 8 + (size_t)s.M * 2;
    HMMB_CUDA(cudaFuncSetAttribute(k_scoreL<NS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 g((unsigned)s.ncta, (unsigned)W);
    HMMB_LAUNCH("score", k_scoreL<NS>, g, LTR_THREADS, smem, s.d_work, s.d_blks, (const uint4 *)s.d_obs, s.d_len, s.d_order,
                d_pi, d_A, d_Bt, s.M, W, d_ll, d_nan);
    return HMMB_OK;
}

int hmmb_score(const void *obs, int idx_bytes, int obs_on_device, const int64_t *offsets, int64_t U, int W, int N, int M,
               const double *pi, const double *A, const double *B, double *ll_out, int32_t *argmax_out) {
    HMMB_TRY(require_init());
    Ctx &c = ctx();
    // the flag the scorers set when the precision guard marked a pair, and the count of pairs k_score_exact recomputed
    // (hmmb_score_diagnostics): one slot of the context, cleared together before anything can fail, so that the count
    // always describes this call
    if (!c.score_slot) HMMB_TRY(dev_alloc_t(&c.score_slot, 4));
    HMMB_CUDA(cudaMemsetAsync(c.score_slot, 0, 4 * sizeof(int32_t), c.stream));
    if (!pi || !A || !B || W <= 0 || W > 65535) { set_error("hmmb_score: bad arguments (W=%d)", W); return HMMB_ERR_ARG; }
    SeqSet s;
    CallGuard guard{s, {}};
    const Family fam = pick_family(N, M, A, W);
    const size_t nB = (size_t)W * N * M, nA = (size_t)W * N * N, nP = (size_t)W * N;
    double *tmp = nullptr, *d_pi = nullptr, *d_A = nullptr, *d_Bt = nullptr, *d_ll = nullptr;
    int32_t *d_arg = nullptr;
    int32_t *d_nan = c.score_slot;
    int64_t *d_npairs = reinterpret_cast<int64_t *>(c.score_slot + 2);
    bool models_up = false;
    // model parameters -> device.  In the pipelined scorer this runs inside seqset_build, between the first chunks and the rest
    // of the codeword upload and on the same DMA queue (see hmmb_bw_create_ex).
    std::function<int()> upload_models = [&]() -> int {
        models_up = true;
        if (U == 0) return HMMB_OK;
        HMMB_TRY(dev_alloc_t(&tmp, nB + nA + nP)); guard.ptrs.push_back(tmp);
        HMMB_TRY(dev_alloc_t(&d_pi, nP)); guard.ptrs.push_back(d_pi);
        HMMB_TRY(dev_alloc_t(&d_A, nA)); guard.ptrs.push_back(d_A);
        HMMB_TRY(dev_alloc_t(&d_Bt, nB)); guard.ptrs.push_back(d_Bt);
        HMMB_TRY(dev_alloc_t(&d_ll, (size_t)U * W)); guard.ptrs.push_back(d_ll);
        HMMB_TRY(dev_alloc_t(&d_arg, (size_t)U)); guard.ptrs.push_back(d_arg);
        HMMB_TRY(h2d_small(tmp, B, nB * sizeof(double)));
        HMMB_TRY(h2d_small(tmp + nB, A, nA * sizeof(double)));
        HMMB_TRY(h2d_small(tmp + nB + nA, pi, nP * sizeof(double)));
        HMMB_TRY(h2d_join());
        dim3 gb((unsigned)std::min((N * M + 255) / 256, 64), (unsigned)W);
        HMMB_LAUNCH("score_load", k_load_B, gb, 256, 0, tmp, N, M, d_Bt, (int32_t *)nullptr);
        HMMB_LAUNCH("score_load", k_load_clamped, (unsigned)std::min<size_t>((nA + 255) / 256, 1024), 256, 0, tmp + nB, (int64_t)nA, d_A);
        HMMB_LAUNCH("score_load", k_load_clamped, (unsigned)std::min<size_t>((nP + 255) / 256, 1024), 256, 0, tmp + nB + nA, (int64_t)nP, d_pi);
        return HMMB_OK;
    };
    // Pipelined scorer (N = 4, pinned codewords in length-descending order, small models): the stages of the
    // upload are repacked and scored as they land, and each stage's rows of the [U, W] matrix start their way back
    // to the host while the next stage is being scored.
    const bool pipeline = fam.layout() != LAYOUT_LTR && nB * sizeof(double) <= (size_t(4) << 20) && !getenv("HMMB_SCORE_NO_PIPELINE");
    HMMB_TRY(seqset_build(s, obs, idx_bytes, obs_on_device, offsets, nullptr, U, 1, N, M, fam.layout(), pipeline,
                          pipeline ? &upload_models : nullptr, score_stages(ll_out != nullptr)));
    if (U == 0) return HMMB_OK;
    if (!models_up) HMMB_TRY(upload_models());
    // [exact recompute of the pairs the precision guard marked,] argmax, results to the host
    auto finish = [&](bool recompute, bool send_ll) -> int {
        if (recompute) {
            const int64_t warps = std::min<int64_t>((int64_t)c.sm_count * 16, U);
            const int eg = (int)std::max<int64_t>(1, (warps + BW_WARPS - 1) / BW_WARPS);
            HMMB_TRY(with_codewords(s, [&](auto sym, auto blocked) -> int {
                HMMB_LAUNCH("score_exact", (k_score_exact<decltype(sym), decltype(blocked)::value>), eg, BW_THREADS, 0, s.d_obs,
                            blocked() ? s.d_foff : s.d_off, s.d_len, s.d_order, U, N, M, W, d_pi, d_A, d_Bt, d_ll, d_nan,
                            d_npairs);
                return HMMB_OK;
            }));
        }
        HMMB_LAUNCH("score_argmax", k_argmax_first, (unsigned)((U + 255) / 256), 256, 0, d_ll, U, W, d_arg);
        if (argmax_out) HMMB_CUDA(cudaMemcpyAsync(argmax_out, d_arg, (size_t)U * sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
        if (send_ll) HMMB_TRY(d2h_big(ll_out, d_ll, (size_t)U * W * sizeof(double), c.stream));
        HMMB_CUDA(cudaStreamSynchronize(c.stream));
        return HMMB_OK;
    };
    if (!s.pend) {
        if (s.layout == LAYOUT_N4) {
            HMMB_TRY(launch_score_special(s, fam.bidiag, W, d_pi, d_A, d_Bt, d_ll, d_nan, 0, s.nblk));
        } else if (s.layout == LAYOUT_LTR) {
            HMMB_TRY(N == 16 ? launch_score_ltr<16>(s, W, d_pi, d_A, d_Bt, d_ll, d_nan) : launch_score_ltr<8>(s, W, d_pi, d_A, d_Bt, d_ll, d_nan));
        } else {
            HMMB_TRY(with_lanes(s, [&](auto np, auto sym) {
                return launch_score_generic<decltype(np)::value, decltype(sym)>(s, W, d_pi, d_A, d_Bt, d_ll, d_nan);
            }));
        }
        // (k_score_exact returns at once when no pair was marked)
        return finish(true, ll_out != nullptr);
    }
    PendingPrepare &p = *s.pend;
    int bdone = 0;
    // a pageable result matrix cannot leave stage by stage (its copies would block the host between the
    // stages): it goes through the bounce buffers after the last stage
    const bool ll_pinned = ll_out && host_is_pinned(ll_out);
    cudaEvent_t scored = event_get();
    for (int j = 0; j < p.nstage; ++j) {
        HMMB_CUDA(cudaStreamWaitEvent(c.stream, p.up->ev[p.ev_index[j]], 0));
        HMMB_TRY(launch_repack_range(s, p.up->d_raw, p.idx_bytes, bdone, p.blk_end[j], s.d_bad));
        HMMB_TRY(launch_score_special(s, fam.bidiag, W, d_pi, d_A, d_Bt, d_ll, d_nan, bdone, p.blk_end[j]));
        if (ll_pinned) {
            // scoring has a single "word", so block b holds utterances [32 b, 32 b + 32) of the (identity) order
            const int64_t u0 = (int64_t)bdone * 32, u1 = std::min<int64_t>(U, (int64_t)p.blk_end[j] * 32);
            HMMB_CUDA(cudaEventRecord(scored, c.stream));
            HMMB_CUDA(cudaStreamWaitEvent(c.d2h_stream, scored, 0));
            HMMB_CUDA(cudaMemcpyAsync(ll_out + u0 * W, d_ll + u0 * W, (size_t)(u1 - u0) * W * sizeof(double),
                                      cudaMemcpyDeviceToHost, c.d2h_stream));
        }
        bdone = p.blk_end[j];
    }
    event_put(scored);
    int32_t flags[2] = {0, 0};  // a pair marked by the precision guard, a codeword out of range
    HMMB_CUDA(cudaMemcpyAsync(&flags[0], d_nan, sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
    HMMB_CUDA(cudaMemcpyAsync(&flags[1], s.d_bad, sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
    HMMB_TRY(finish(false, ll_out && !ll_pinned));
    HMMB_CUDA(cudaStreamSynchronize(c.d2h_stream));
    s.pend.reset();
    if (flags[1]) {
        set_error("codeword out of range: some observation is >= M=%d (reference: IndexError)", M);
        return HMMB_ERR_RANGE;
    }
    // rare: the precision guard marked pairs; recompute them in log space and send everything again
    if (flags[0]) return finish(true, ll_out != nullptr);
    return HMMB_OK;
}

int hmmb_score_diagnostics(int64_t *exact_pairs) {
    HMMB_TRY(require_init());
    if (!exact_pairs) { set_error("hmmb_score_diagnostics: null argument"); return HMMB_ERR_ARG; }
    Ctx &c = ctx();
    int64_t n = 0;
    if (c.score_slot) {
        HMMB_CUDA(cudaMemcpyAsync(&n, c.score_slot + 2, sizeof(int64_t), cudaMemcpyDeviceToHost, c.stream));
        HMMB_CUDA(cudaStreamSynchronize(c.stream));
    }
    *exact_pairs = n;
    return HMMB_OK;
}

// ---------------------------------------------------------------- Viterbi decoding
template <int NS, bool BIDIAG>
static int launch_viterbi_blocked(SeqSet &s, const double *d_lpi, const double *d_lA, const double *d_lBt, double *d_score,
                                  int8_t *d_last, void *d_bp) {
    if (s.ncta == 0) return HMMB_OK;
    const size_t smem = (size_t)s.M * NS * sizeof(double);
    HMMB_CUDA(cudaFuncSetAttribute((k_viterbiB<NS, BIDIAG>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // The work items are sized for the trainer's CTAs (about two per SM at N = 4, each for one 16-warp backward CTA);
    // one 8-warp Viterbi CTA per item would leave the SMs with a few warps each for a latency-bound per-thread
    // recursion, so every item is shared by enough CTAs for about eight per SM.
    const int split = std::max(1, std::min(BWD4_MAX_WARPS, (ctx().sm_count * 8 + s.ncta - 1) / s.ncta));
    dim3 g((unsigned)s.ncta, (unsigned)split);
    HMMB_LAUNCH("viterbi", (k_viterbiB<NS, BIDIAG>), g, VIT_THREADS, smem, s.d_work, s.d_blks, (const uint4 *)s.d_obs, s.d_len,
                s.d_order, d_lpi, d_lA, d_lBt, s.M, d_score, d_last, (VitRow<NS> *)d_bp);
    return HMMB_OK;
}

template <int NS>
static int launch_vit_backtrace_blocked(SeqSet &s, const int8_t *d_last, const void *d_bp, int8_t *d_path) {
    if (s.nblk == 0) return HMMB_OK;
    constexpr int WPB = VIT_THREADS / 32;
    HMMB_LAUNCH("viterbi_backtrace", k_vit_backtraceB<NS>, (s.nblk + WPB - 1) / WPB, VIT_THREADS, 0, s.d_blks, s.nblk, s.d_len,
                s.d_off, d_last, (const VitRow<NS> *)d_bp, d_path);
    return HMMB_OK;
}

template <int NP, typename SymT>
static int launch_viterbi_generic(SeqSet &s, const double *d_lpi, const double *d_lA, const double *d_lBt, double *d_score,
                                  int8_t *d_last, uint8_t *d_bp) {
    const LanesGrid g = lanes_grid(s.R, NP);
    HMMB_LAUNCH("viterbi", (k_viterbiG<NP, SymT>), g.grid, BW_THREADS, 0, (const SymT *)s.d_obs, s.d_off, s.d_len, s.d_word,
                s.d_order, s.d_foff, s.R, g.per_group, s.N, s.M, d_lpi, d_lA, d_lBt, d_score, d_last, d_bp);
    return HMMB_OK;
}

int hmmb_viterbi(const void *obs, int idx_bytes, int obs_on_device, const int64_t *offsets, int64_t U,
                 const int32_t *model_of_utt, int W, int N, int M, const double *pi, const double *A, const double *B,
                 double *score_out, int8_t *path_out) {
    HMMB_TRY(require_init());
    if (!pi || !A || !B || W <= 0 || W > 65535 || (U > 0 && !model_of_utt)) {
        set_error("hmmb_viterbi: bad arguments (W=%d)", W);
        return HMMB_ERR_ARG;
    }
    Ctx &c = ctx();
    SeqSet s;
    CallGuard guard{s, {}};
    // the layouts and kernel families of hmmb_score
    const Family fam = pick_family(N, M, A, W);
    HMMB_TRY(seqset_build(s, obs, idx_bytes, obs_on_device, offsets, model_of_utt, U, W, N, M, fam.layout()));
    if (U == 0) return HMMB_OK;
    const size_t nB = (size_t)W * N * M, nA = (size_t)W * N * N, nP = (size_t)W * N;
    double *tmp = nullptr, *d_lBt = nullptr, *d_lA = nullptr, *d_lpi = nullptr, *d_score = nullptr;
    HMMB_TRY(dev_alloc_t(&tmp, nB + nA + nP)); guard.ptrs.push_back(tmp);
    HMMB_TRY(dev_alloc_t(&d_lBt, nB + nA + nP)); guard.ptrs.push_back(d_lBt);
    d_lA = d_lBt + nB;
    d_lpi = d_lA + nA;
    HMMB_TRY(dev_alloc_t(&d_score, (size_t)U)); guard.ptrs.push_back(d_score);
    HMMB_CUDA(cudaMemcpyAsync(tmp, B, nB * sizeof(double), cudaMemcpyHostToDevice, c.stream));
    HMMB_CUDA(cudaMemcpyAsync(tmp + nB, A, nA * sizeof(double), cudaMemcpyHostToDevice, c.stream));
    HMMB_CUDA(cudaMemcpyAsync(tmp + nB + nA, pi, nP * sizeof(double), cudaMemcpyHostToDevice, c.stream));
    HMMB_LAUNCH("viterbi_load", k_vit_logs, (unsigned)std::min<size_t>((nB + nA + nP + 255) / 256, (size_t)c.sm_count * 8), 256, 0,
                tmp + 0, tmp + nB, tmp + nB + nA, W, N, M, d_lBt, d_lA, d_lpi);
    // backpointers: blocked layouts one packed row per step and lane (1 byte per frame at N = 4 / 8, 2 at N = 16);
    // generic layout one byte per state per frame
    const bool want_path = path_out != nullptr;
    int8_t *d_last = nullptr, *d_path = nullptr;
    void *d_bp = nullptr;
    if (want_path) {
        const size_t row_bytes = s.layout == LAYOUT_LTR && N == 16 ? 2 : 1;
        const size_t bp_bytes = s.blocked() ? (size_t)s.spill_steps * 32 * row_bytes : (size_t)s.frames * N;
        HMMB_TRY(dev_alloc(&d_bp, bp_bytes)); guard.ptrs.push_back(d_bp);
        HMMB_TRY(dev_alloc_t(&d_last, (size_t)U)); guard.ptrs.push_back(d_last);
        HMMB_TRY(dev_alloc_t(&d_path, (size_t)s.frames)); guard.ptrs.push_back(d_path);
    }
    if (s.layout == LAYOUT_N4) {
        HMMB_TRY((fam.bidiag ? launch_viterbi_blocked<4, true>(s, d_lpi, d_lA, d_lBt, d_score, d_last, d_bp)
                             : launch_viterbi_blocked<4, false>(s, d_lpi, d_lA, d_lBt, d_score, d_last, d_bp)));
        if (want_path) HMMB_TRY(launch_vit_backtrace_blocked<4>(s, d_last, d_bp, d_path));
    } else if (s.layout == LAYOUT_LTR) {
        HMMB_TRY((N == 16 ? launch_viterbi_blocked<16, true>(s, d_lpi, d_lA, d_lBt, d_score, d_last, d_bp)
                          : launch_viterbi_blocked<8, true>(s, d_lpi, d_lA, d_lBt, d_score, d_last, d_bp)));
        if (want_path)
            HMMB_TRY(N == 16 ? launch_vit_backtrace_blocked<16>(s, d_last, d_bp, d_path)
                             : launch_vit_backtrace_blocked<8>(s, d_last, d_bp, d_path));
    } else {
        uint8_t *bp8 = (uint8_t *)d_bp;
        HMMB_TRY(with_lanes(s, [&](auto np, auto sym) {
            return launch_viterbi_generic<decltype(np)::value, decltype(sym)>(s, d_lpi, d_lA, d_lBt, d_score, d_last, bp8);
        }));
        if (want_path)
            HMMB_LAUNCH("viterbi_backtrace", k_vit_backtraceG, (unsigned)((U + VIT_THREADS - 1) / VIT_THREADS), VIT_THREADS, 0, U, N,
                        s.d_len, s.d_off, s.d_foff, d_last, bp8, d_path);
    }
    if (score_out) HMMB_TRY(d2h_big(score_out, d_score, (size_t)U * sizeof(double), c.stream));
    if (want_path) HMMB_TRY(d2h_big(path_out, d_path, (size_t)s.frames, c.stream));
    HMMB_CUDA(cudaStreamSynchronize(c.stream));
    return HMMB_OK;
}

// ---------------------------------------------------------------- connected-word decoding
template <int SPT, typename SymT>
static int launch_words_generic(SeqSet &s, int W, int N, double log_penalty, const double *d_lpi, const double *d_lA,
                                const double *d_lE, double *d_score, int2 *d_rec) {
    Ctx &c = ctx();
    const int K = W * N;
    const int threads = (int)std::min<int64_t>(WORDS_MAX_THREADS, ((K + SPT - 1) / SPT + 31) / 32 * 32);
    const size_t smem = (size_t)K * 24 + 2 * 32 * sizeof(WordEnd);
    HMMB_CUDA(cudaFuncSetAttribute((k_wordsG<SPT, SymT>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    HMMB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (k_wordsG<SPT, SymT>), threads, smem));
    const unsigned grid = (unsigned)std::min<int64_t>(s.R, (int64_t)c.sm_count * std::max(per_sm, 1));
    HMMB_LAUNCH("words", (k_wordsG<SPT, SymT>), grid, threads, smem, (const SymT *)s.d_obs, s.d_off, s.d_len, s.d_order, s.R,
                W, N, d_lpi, d_lA, d_lE, log_penalty, d_score, d_rec);
    return HMMB_OK;
}

// the fewest states per thread that keep a CTA within WORDS_MAX_THREADS threads
template <typename SymT>
static int launch_words_spt(SeqSet &s, int W, int N, double log_penalty, const double *d_lpi, const double *d_lA,
                            const double *d_lE, double *d_score, int2 *d_rec) {
    const int K = W * N;
    if (K <= WORDS_MAX_THREADS) return launch_words_generic<1, SymT>(s, W, N, log_penalty, d_lpi, d_lA, d_lE, d_score, d_rec);
    if (K <= 2 * WORDS_MAX_THREADS) return launch_words_generic<2, SymT>(s, W, N, log_penalty, d_lpi, d_lA, d_lE, d_score, d_rec);
    if (K <= 4 * WORDS_MAX_THREADS) return launch_words_generic<4, SymT>(s, W, N, log_penalty, d_lpi, d_lA, d_lE, d_score, d_rec);
    return launch_words_generic<8, SymT>(s, W, N, log_penalty, d_lpi, d_lA, d_lE, d_score, d_rec);
}
static_assert(WORDS_MAX_STATES <= 8 * WORDS_MAX_THREADS, "launch_words_spt covers every W * N up to the bound");

// lane = word (W <= 32): G lanes per utterance, 32 / G utterances per warp; the log-emission table in shared memory
// when it fits the opt-in limit (the reference's shape: 256 x 10 x 4 x 8 B = 80 KB)
template <int NS, bool BIDIAG, typename SymT>
static int launch_words_blocked(SeqSet &s, int W, double log_penalty, const double *d_lpi, const double *d_lA,
                                const double *d_lE, double *d_score, int2 *d_rec) {
    Ctx &c = ctx();
    int G = 1;
    while (G < W) G <<= 1;
    const int64_t warps_needed = (s.R + 32 / G - 1) / (32 / G);
    const size_t tab = (size_t)s.M * W * NS * sizeof(double);
    const bool smem = tab <= (size_t)c.smem_optin;
    auto launch = [&](auto kern, size_t bytes) -> int {
        if (bytes) HMMB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        int per_sm = 0;
        HMMB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WORDSB_THREADS, bytes));
        const int64_t want = (warps_needed + WORDSB_THREADS / 32 - 1) / (WORDSB_THREADS / 32);
        const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)c.sm_count * std::max(per_sm, 1)));
        HMMB_LAUNCH("words", kern, grid, WORDSB_THREADS, bytes, (const SymT *)s.d_obs, s.d_off, s.d_len, s.d_order, s.R, W,
                    G, s.M, d_lpi, d_lA, d_lE, log_penalty, d_score, d_rec);
        return HMMB_OK;
    };
    return smem ? launch(k_wordsB<NS, BIDIAG, true, SymT>, tab) : launch(k_wordsB<NS, BIDIAG, false, SymT>, (size_t)0);
}

int hmmb_decode_words(const void *obs, int idx_bytes, int obs_on_device, const int64_t *offsets, int64_t U, int W, int N,
                      int M, const double *pi, const double *A, const double *B, double log_penalty, double *score_out,
                      int64_t *seg_offsets_out, int32_t *seg_word_out, int32_t *seg_start_out) {
    HMMB_TRY(require_init());
    if (!pi || !A || !B || W <= 0 || W > 65535 || !std::isfinite(log_penalty) || (!seg_word_out != !seg_start_out)) {
        set_error("hmmb_decode_words: bad arguments (W=%d, log_penalty=%g; seg_word_out and seg_start_out go together)", W,
                  log_penalty);
        return HMMB_ERR_ARG;
    }
    if (N >= 1 && N <= HMMB_MAX_STATES && (int64_t)W * N > WORDS_MAX_STATES) {
        set_error("hmmb_decode_words: W * N = %lld states above the limit of %d", (long long)W * N, WORDS_MAX_STATES);
        return HMMB_ERR_UNSUPPORTED;
    }
    Ctx &c = ctx();
    if (U == 0 && seg_offsets_out) seg_offsets_out[0] = 0;
    SeqSet s;
    CallGuard guard{s, {}};
    // one codeword stream in length-descending order (a single "word": every utterance meets every model) for either
    // kernel; the family decision of the scorer picks the lane-per-word kernel for the blocked shapes
    const Family fam = pick_family(N, M, A, W);
    const bool blocked = fam.layout() != LAYOUT_LANES && W <= 32;
    HMMB_TRY(seqset_build(s, obs, idx_bytes, obs_on_device, offsets, nullptr, U, 1, N, M, LAYOUT_LANES));
    if (U == 0) return HMMB_OK;
    const size_t nE = (size_t)W * N * M, nA = (size_t)W * N * N, nP = (size_t)W * N;
    double *tmp = nullptr, *d_lE = nullptr, *d_score = nullptr;
    HMMB_TRY(dev_alloc_t(&tmp, nE + nA + nP)); guard.ptrs.push_back(tmp);
    HMMB_TRY(dev_alloc_t(&d_lE, nE + nA + nP)); guard.ptrs.push_back(d_lE);
    double *d_lA = d_lE + nE, *d_lpi = d_lA + nA;
    HMMB_TRY(dev_alloc_t(&d_score, (size_t)U)); guard.ptrs.push_back(d_score);
    HMMB_CUDA(cudaMemcpyAsync(tmp, B, nE * sizeof(double), cudaMemcpyHostToDevice, c.stream));
    HMMB_CUDA(cudaMemcpyAsync(tmp + nE, A, nA * sizeof(double), cudaMemcpyHostToDevice, c.stream));
    HMMB_CUDA(cudaMemcpyAsync(tmp + nE + nA, pi, nP * sizeof(double), cudaMemcpyHostToDevice, c.stream));
    HMMB_LAUNCH("words_load", k_words_logs, (unsigned)std::min<size_t>((nE + nA + nP + 255) / 256, (size_t)c.sm_count * 8), 256, 0,
                tmp + 0, tmp + nE, tmp + nE + nA, W, N, M, d_lE, d_lA, d_lpi);
    // word-end records: one (word, first frame) pair per frame at the frame's input position
    const bool want_segments = seg_offsets_out || seg_word_out;
    int2 *d_rec = nullptr;
    if (want_segments) { HMMB_TRY(dev_alloc_t(&d_rec, (size_t)s.frames)); guard.ptrs.push_back(d_rec); }
    if (blocked) {
        auto run = [&](auto sym) -> int {
            using SymT = decltype(sym);
            if (N == 4) return fam.bidiag ? launch_words_blocked<4, true, SymT>(s, W, log_penalty, d_lpi, d_lA, d_lE, d_score, d_rec)
                                          : launch_words_blocked<4, false, SymT>(s, W, log_penalty, d_lpi, d_lA, d_lE, d_score, d_rec);
            return N == 8 ? launch_words_blocked<8, true, SymT>(s, W, log_penalty, d_lpi, d_lA, d_lE, d_score, d_rec)
                          : launch_words_blocked<16, true, SymT>(s, W, log_penalty, d_lpi, d_lA, d_lE, d_score, d_rec);
        };
        HMMB_TRY(s.sym_bytes == 1 ? run(uint8_t{}) : run(uint16_t{}));
    } else {
        HMMB_TRY(s.sym_bytes == 1 ? launch_words_spt<uint8_t>(s, W, N, log_penalty, d_lpi, d_lA, d_lE, d_score, d_rec)
                                  : launch_words_spt<uint16_t>(s, W, N, log_penalty, d_lpi, d_lA, d_lE, d_score, d_rec));
    }
    if (score_out) HMMB_TRY(d2h_big(score_out, d_score, (size_t)U * sizeof(double), c.stream));
    if (!want_segments) {
        HMMB_CUDA(cudaStreamSynchronize(c.stream));
        return HMMB_OK;
    }
    // segment counts -> host, prefix sum, offsets -> device, the segments written at them and copied back
    std::vector<int64_t> seg_off((size_t)U + 1);
    int64_t *d_segoff = nullptr;
    HMMB_TRY(dev_alloc_t(&d_segoff, (size_t)U + 1)); guard.ptrs.push_back(d_segoff);
    const unsigned bt_grid = (unsigned)((U + WORDS_BT_THREADS - 1) / WORDS_BT_THREADS);
    HMMB_LAUNCH("words_backtrace", k_words_count, bt_grid, WORDS_BT_THREADS, 0, U, s.d_off, s.d_len, s.d_order, d_score, d_rec,
                d_segoff + 1);
    HMMB_TRY(d2h_big(seg_off.data() + 1, d_segoff + 1, (size_t)U * sizeof(int64_t), c.stream));
    HMMB_CUDA(cudaStreamSynchronize(c.stream));
    seg_off[0] = 0;
    for (int64_t u = 0; u < U; ++u) seg_off[u + 1] += seg_off[u];
    const int64_t nseg = seg_off[U];
    if (seg_offsets_out) std::copy(seg_off.begin(), seg_off.end(), seg_offsets_out);
    if (!seg_word_out || nseg == 0) return HMMB_OK;
    int32_t *d_seg = nullptr;
    HMMB_TRY(dev_alloc_t(&d_seg, (size_t)nseg * 2)); guard.ptrs.push_back(d_seg);
    HMMB_CUDA(cudaMemcpyAsync(d_segoff, seg_off.data(), ((size_t)U + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, c.stream));
    HMMB_LAUNCH("words_backtrace", k_words_emit, bt_grid, WORDS_BT_THREADS, 0, U, s.d_off, s.d_len, s.d_order, d_segoff, d_rec,
                d_seg, d_seg + nseg);
    HMMB_TRY(d2h_big(seg_word_out, d_seg, (size_t)nseg * sizeof(int32_t), c.stream));
    HMMB_TRY(d2h_big(seg_start_out, d_seg + nseg, (size_t)nseg * sizeof(int32_t), c.stream));
    HMMB_CUDA(cudaStreamSynchronize(c.stream));
    return HMMB_OK;
}

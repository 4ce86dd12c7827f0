// Connected-word decoding (an extension: the reference recognises one word per recording): the best word sequence of
// every utterance over a free loop of W isolated-word models, by one-pass dynamic programming (Vintsyuk; Bridle, Brown
// and Chamberlain; Rabiner & Juang ch. 7).
//
// Semantics (shared with oracle/words_oracle.py and include/hmmb200.h), additions in exactly this order:
//   delta_0(w,j) = lpi[w][j] + lb[w][j](o_0)                              token_0(w,j) = 0
//   t >= 1:  in(w,j) = max_i (delta_t-1(w,i) + lA[w][i][j])    smallest i on ties (ascending scan, strict '>')
//            en(w,j) = E_t-1 + lpi[w][j]
//            delta_t(w,j) = (en > in ? en : in) + lb[w][j](o_t)
//            token_t(w,j) = en > in ? t : token_t-1(w, argmax i)
//   e_t = max_w delta_t(w, N-1) (smallest w on ties),  E_t = e_t + log_penalty,  record_t = (argmax w, its token)
//   score = E_T-1
// A word is entered in any state and left only from its last state.  The backtrace reads record_t = (w, s) at
// t = T-1, which is "word w on frames [s, t]", and continues at t = s - 1.
//
// Like the Viterbi decoder the recursion only adds and compares log values, so it needs no precision guard.
//
//   k_words_logs   linear pi / A / B -> log pi, log A and the codeword-major log emission table [M][W][N]: the W * N
//                  states of one codeword are one contiguous row, read coalesced by the threads of a frame.
//   k_wordsB       lane = word on the blocked shapes (N = 4; left-to-right N = 8 / 16) with W <= 32: G = the next power
//                  of two >= W lanes per utterance, 32 / G utterances per warp, delta and tokens in registers, the
//                  word-end max by xor shuffles within the group; no barrier.
//   k_wordsG       one CTA per utterance (grid-stride over the length-sorted order), threads over the states
//                  k = w * N + j, delta and tokens double-buffered in shared memory, one barrier per frame.
//   k_words_count / k_words_emit   one thread per utterance walks its word-end records (K steps for K words): the
//                  segment count, then the segments in time order at their prefix offsets.
#pragma once

#include "viterbi_kernels.cuh"

namespace hmmb {

constexpr int WORDS_MAX_STATES = 8192;   // W * N: 24 B of shared memory per state (2 x delta + 2 x token) = 192 KB
constexpr int WORDS_MAX_THREADS = 1024;
constexpr int WORDS_BT_THREADS = 256;
constexpr int WORDSB_THREADS = 256;

// raw linear B [W][N][M], A [W][N][N], pi [W][N] -> log B as [M][W][N], log A, log pi
__global__ void k_words_logs(const double *__restrict__ B, const double *__restrict__ A, const double *__restrict__ pi,
                             int W, int N, int M, double *__restrict__ lE, double *__restrict__ lA, double *__restrict__ lpi) {
    const int64_t K = (int64_t)W * N, nE = K * M, nA = K * N, nP = K;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nE + nA + nP; e += (int64_t)gridDim.x * blockDim.x) {
        if (e < nE) {  // B read in its own layout (coalesced), the table written scattered
            const int64_t k = e / M, sym = e - k * M;
            lE[sym * K + k] = vit_log(B[e]);
        } else if (e < nE + nA) {
            lA[e - nE] = vit_log(A[e - nE]);
        } else {
            lpi[e - nE - nA] = vit_log(pi[e - nE - nA]);
        }
    }
}

// A word-end candidate: the larger value wins, the smaller word on equal values (a total order, so any reduction tree
// gives the same winner).
struct WordEnd {
    double v;
    int w, tok;
};
__device__ __forceinline__ bool word_end_better(double v, int w, const WordEnd &b) { return v > b.v || (v == b.v && w < b.w); }

// SPT states per thread (state k = threadIdx.x + q * blockDim.x); dynamic shared memory: delta [2][K] fp64, token
// [2][K] int32, word-end partials [2][32].  rec == nullptr: score only (no records).
template <int SPT, typename SymT>
__global__ void __launch_bounds__(WORDS_MAX_THREADS)
k_wordsG(const SymT *__restrict__ obs, const int64_t *__restrict__ off_sorted, const int32_t *__restrict__ len_sorted,
         const int32_t *__restrict__ order, int64_t U, int W, int N, const double *__restrict__ lpi,
         const double *__restrict__ lA, const double *__restrict__ lE, double log_penalty, double *__restrict__ score_out,
         int2 *__restrict__ rec) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int K = W * N;
    double *sd = reinterpret_cast<double *>(smem_raw);
    int32_t *stok = reinterpret_cast<int32_t *>(sd + 2 * K);
    WordEnd *red = reinterpret_cast<WordEnd *>(smem_raw + (size_t)K * 24);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    // ph: the buffer this frame writes, flipped every frame over all utterances of the CTA, so that the single barrier
    // per frame also separates a frame's reads of the partials from the writes two frames later
    int ph = 0;
    for (int64_t r = blockIdx.x; r < U; r += gridDim.x) {
        const int T = len_sorted[r];
        const SymT *o = obs + off_sorted[r];
        int2 *rr = rec ? rec + off_sorted[r] : nullptr;
        double lb[SPT];
        {
            const double *row = lE + (size_t)o[0] * K;
#pragma unroll
            for (int q = 0; q < SPT; ++q) lb[q] = tid + q * (int)blockDim.x < K ? __ldg(row + tid + q * blockDim.x) : neg_inf();
        }
        double E = neg_inf();
        for (int t = 0; t < T; ++t, ph ^= 1) {
            double nb[SPT];  // the next frame's emissions, loaded ahead
            if (t + 1 < T) {
                const double *row = lE + (size_t)o[t + 1] * K;
#pragma unroll
                for (int q = 0; q < SPT; ++q) nb[q] = tid + q * (int)blockDim.x < K ? __ldg(row + tid + q * blockDim.x) : neg_inf();
            }
            const double *dprev = sd + (ph ^ 1) * K;
            const int32_t *tprev = stok + (ph ^ 1) * K;
            WordEnd best{neg_inf(), INT_MAX, 0};
#pragma unroll
            for (int q = 0; q < SPT; ++q) {
                const int k = tid + q * (int)blockDim.x;
                if (k >= K) continue;
                const int w = k / N, j = k - w * N;
                const double lp = __ldg(lpi + k);
                double v;
                int tok;
                if (t == 0) {
                    v = lp + lb[q];
                    tok = 0;
                } else {
                    const double *dw = dprev + w * N;
                    const double *la = lA + (size_t)w * N * N + j;
                    double in = dw[0] + __ldg(la);
                    int arg = 0;
                    for (int i = 1; i < N; ++i) {
                        const double c = dw[i] + __ldg(la + (size_t)i * N);
                        if (c > in) { in = c; arg = i; }
                    }
                    const double en = E + lp;
                    if (en > in) {
                        v = en + lb[q];
                        tok = t;
                    } else {
                        v = in + lb[q];
                        tok = tprev[w * N + arg];
                    }
                }
                sd[ph * K + k] = v;
                stok[ph * K + k] = tok;
                if (j == N - 1 && word_end_better(v, w, best)) best = WordEnd{v, w, tok};
            }
#pragma unroll
            for (int s = 16; s > 0; s >>= 1) {
                const double ov = __shfl_xor_sync(0xffffffffu, best.v, s);
                const int ow = __shfl_xor_sync(0xffffffffu, best.w, s);
                const int ot = __shfl_xor_sync(0xffffffffu, best.tok, s);
                if (word_end_better(ov, ow, best)) best = WordEnd{ov, ow, ot};
            }
            if (lane == 0) red[ph * 32 + warp] = best;
            __syncthreads();
            best = red[ph * 32];
            for (int x = 1; x < nwarps; ++x) {
                const WordEnd c = red[ph * 32 + x];
                if (word_end_better(c.v, c.w, best)) best = c;
            }
            E = best.v + log_penalty;
            if (rr && tid == 0) rr[t] = make_int2(best.w, best.tok);
#pragma unroll
            for (int q = 0; q < SPT; ++q) lb[q] = nb[q];
        }
        if (tid == 0) score_out[order[r]] = E;
    }
}

// G lanes per utterance (lane % G = word, lanes with word >= W idle), utterance r = group index, grid-stride over the
// warps of the length-descending order; a warp runs to the longest T of its groups.  SMEM: the [M][W][NS] log-emission
// table is staged in dynamic shared memory, else read with __ldg.  rec == nullptr: score only.
template <int NS, bool BIDIAG, bool SMEM, typename SymT>
__global__ void __launch_bounds__(WORDSB_THREADS)
k_wordsB(const SymT *__restrict__ obs, const int64_t *__restrict__ off_sorted, const int32_t *__restrict__ len_sorted,
         const int32_t *__restrict__ order, int64_t U, int W, int G, int M, const double *__restrict__ lpi,
         const double *__restrict__ lA, const double *__restrict__ lE, double log_penalty, double *__restrict__ score_out,
         int2 *__restrict__ rec) {
    static_assert(NS == 4 || (BIDIAG && (NS == 8 || NS == 16)), "blocked word decoder: N = 4, or left-to-right N = 8 / 16");
    constexpr int CPR = NS / 2;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const double2 *tab = reinterpret_cast<const double2 *>(lE);
    if (SMEM) {
        double2 *st = reinterpret_cast<double2 *>(smem_raw);
        const int n = M * W * CPR;
        for (int e = threadIdx.x; e < n; e += WORDSB_THREADS) st[e] = __ldg(tab + e);
        __syncthreads();
        tab = st;
    }
    const int lane = threadIdx.x & 31;
    const int g = lane % G, gpw = 32 / G;
    const bool live = g < W;
    const int w = live ? g : 0;
    // dense: la[i * NS + j] = log a_ij; left-to-right: la[i] = log a_ii, la[NS + i] = log a_i,i+1
    double la[BIDIAG ? 2 * NS : NS * NS], lp[NS];
    const double *lAw = lA + (size_t)w * NS * NS;
#pragma unroll
    for (int i = 0; i < NS; ++i) {
        lp[i] = live ? __ldg(lpi + w * NS + i) : neg_inf();
        if (BIDIAG) {
            la[i] = __ldg(lAw + i * NS + i);
            la[NS + i] = (i + 1 < NS) ? __ldg(lAw + i * NS + i + 1) : neg_inf();
        } else {
#pragma unroll
            for (int j = 0; j < NS; ++j) la[i * NS + j] = __ldg(lAw + i * NS + j);
        }
    }
    const int64_t warps = (int64_t)gridDim.x * (WORDSB_THREADS / 32);
    for (int64_t wb = (int64_t)blockIdx.x * (WORDSB_THREADS / 32) + (threadIdx.x >> 5); wb * gpw < U; wb += warps) {
        const int64_t r = wb * gpw + lane / G;
        const int T = r < U ? len_sorted[r] : 0;
        const int Tw = warp_max_int(T);
        const SymT *o = obs + (T > 0 ? off_sorted[r] : 0);
        int2 *rr = (rec && T > 0) ? rec + off_sorted[r] : nullptr;
        double d[NS];
        int tk[NS];
        double E = neg_inf();
        unsigned sym_next = T > 0 ? (unsigned)o[0] : 0u;
        for (int t = 0; t < Tw; ++t) {
            const bool act = t < T;
            const unsigned sym = sym_next;
            if (t + 1 < T) sym_next = (unsigned)o[t + 1];
            double lb[NS];
            const double2 *row = tab + ((size_t)sym * W + w) * CPR;
#pragma unroll
            for (int q = 0; q < CPR; ++q) {
                const double2 x = (act && live) ? (SMEM ? row[q] : __ldg(row + q)) : make_double2(neg_inf(), neg_inf());
                lb[2 * q] = x.x;
                lb[2 * q + 1] = x.y;
            }
            if (t == 0) {
#pragma unroll
                for (int j = 0; j < NS; ++j) {
                    d[j] = lp[j] + lb[j];
                    tk[j] = 0;
                }
            } else if (act) {
                if (BIDIAG) {
                    // candidates i = j - 1 (scanned first) and i = j: the stay wins only if strictly larger
#pragma unroll
                    for (int j = NS - 1; j >= 0; --j) {
                        double in = d[j] + la[j];
                        int from = tk[j];
                        if (j > 0) {
                            const double mv = d[j - 1] + la[NS + j - 1];
                            if (!(in > mv)) { in = mv; from = tk[j - 1]; }
                        }
                        const double en = E + lp[j];
                        d[j] = (en > in ? en : in) + lb[j];
                        tk[j] = en > in ? t : from;
                    }
                } else {
                    double nd[NS];
                    int nt[NS];
#pragma unroll
                    for (int j = 0; j < NS; ++j) {
                        double in = d[0] + la[j];
                        int from = tk[0];
#pragma unroll
                        for (int i = 1; i < NS; ++i) {
                            const double c = d[i] + la[i * NS + j];
                            if (c > in) { in = c; from = tk[i]; }
                        }
                        const double en = E + lp[j];
                        nd[j] = (en > in ? en : in) + lb[j];
                        nt[j] = en > in ? t : from;
                    }
#pragma unroll
                    for (int j = 0; j < NS; ++j) { d[j] = nd[j]; tk[j] = nt[j]; }
                }
            }
            // word-end max over the group: (value, word, token), the smallest word on equal values
            WordEnd best{live ? d[NS - 1] : neg_inf(), live ? g : INT_MAX, tk[NS - 1]};
            for (int s = G >> 1; s > 0; s >>= 1) {
                const double ov = __shfl_xor_sync(0xffffffffu, best.v, s);
                const int ow = __shfl_xor_sync(0xffffffffu, best.w, s);
                const int ot = __shfl_xor_sync(0xffffffffu, best.tok, s);
                if (word_end_better(ov, ow, best)) best = WordEnd{ov, ow, ot};
            }
            if (act) {
                E = best.v + log_penalty;
                if (rr && g == 0) rr[t] = make_int2(best.w, best.tok);
            }
        }
        if (T > 0 && g == 0) score_out[order[r]] = E;
    }
}

// one thread per utterance (sorted order): the number of segments of its best word sequence (0 if it is impossible)
__global__ void __launch_bounds__(WORDS_BT_THREADS)
k_words_count(int64_t U, const int64_t *__restrict__ off_sorted, const int32_t *__restrict__ len_sorted,
              const int32_t *__restrict__ order, const double *__restrict__ score, const int2 *__restrict__ rec,
              int64_t *__restrict__ count) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= U) return;
    const int u = order[r];
    int64_t n = 0;
    if (score[u] > neg_inf()) {
        const int2 *rr = rec + off_sorted[r];
        for (int t = len_sorted[r] - 1; t >= 0; t = rr[t].y - 1) ++n;
    }
    count[u] = n;
}

// the second walk: the segments of utterance u go to [seg_off[u], seg_off[u + 1]), in time order
__global__ void __launch_bounds__(WORDS_BT_THREADS)
k_words_emit(int64_t U, const int64_t *__restrict__ off_sorted, const int32_t *__restrict__ len_sorted,
             const int32_t *__restrict__ order, const int64_t *__restrict__ seg_off, const int2 *__restrict__ rec,
             int32_t *__restrict__ seg_word, int32_t *__restrict__ seg_start) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= U) return;
    const int u = order[r];
    int64_t pos = seg_off[u + 1];
    if (pos == seg_off[u]) return;
    const int2 *rr = rec + off_sorted[r];
    for (int t = len_sorted[r] - 1; t >= 0; t = rr[t].y - 1) {
        --pos;
        seg_word[pos] = rr[t].x;
        seg_start[pos] = rr[t].y;
    }
}

}  // namespace hmmb

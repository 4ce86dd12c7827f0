// Viterbi decoding (an extension: the reference has no Viterbi): the most likely state path of every utterance under
// the model it is assigned to, and that path's log-probability.
//
// Semantics (shared with oracle/viterbi_oracle.py):
//   delta_0(j) = log pi_j + log b_j(o_0)
//   delta_t(j) = (max_i (delta_t-1(i) + log a_ij)) + log b_j(o_t)          (additions in exactly this order)
//   psi_t(j)   = the smallest i that reaches the max (ascending scan, strict '>')
//   last state = the smallest j that reaches max_j delta_T-1(j); the score is that max.
// An utterance whose score is -inf gets -1 for every frame.
//
// The recursion only adds and compares log values, so unlike the scaled linear forward pass it needs no precision
// guard: -inf marks a structural zero, and -inf + x = -inf never produces a NaN.  These kernels are exact as they are.
//
//   k_vit_logs        linear pi / A / B (non-positive or NaN entries = structural zeros) -> log pi, log A, log B^T.
//   k_viterbiB        one utterance per THREAD on the blocked layouts (N = 4; N = 8 / 16 upper-bidiagonal): log B^T of
//                     the work item's model in shared memory, delta in registers, one packed backpointer row per step
//                     interleaved by lane: step t of block b at row (Blk::spill_base + t), 32 lanes per row.
//   k_viterbiG        lanes = states on the generic layout (every other shape): the max over i by shuffles, one
//                     backpointer byte per state per frame at the sequence's frame prefix.
//   k_vit_backtrace*  the lanes of a block / one thread per sequence walk t from the end down; the path goes to the
//                     input frame order.
#pragma once

#include <type_traits>

#include "bwltr_kernels.cuh"

namespace hmmb {

constexpr int VIT_THREADS = 256;

// log of the clamped linear value (HMM/hmm_training.py:46-54's safe_log); log(), not a fast-math approximation
__device__ __forceinline__ double vit_log(double v) { return v > 0.0 ? log(v) : neg_inf(); }

// raw linear B [W][N][M], A [W][N][N], pi [W][N] -> log B^T [W][M][N], log A, log pi
__global__ void k_vit_logs(const double *__restrict__ B, const double *__restrict__ A, const double *__restrict__ pi,
                           int W, int N, int M, double *__restrict__ lBt, double *__restrict__ lA, double *__restrict__ lpi) {
    const int64_t nB = (int64_t)W * M * N, nA = (int64_t)W * N * N, nP = (int64_t)W * N;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nB + nA + nP; e += (int64_t)gridDim.x * blockDim.x) {
        if (e < nB) {
            const int64_t w = e / ((int64_t)M * N), r = e - w * M * N;
            const int64_t k = r / N, j = r - k * N;
            lBt[e] = vit_log(B[(w * N + j) * M + k]);
        } else if (e < nB + nA) {
            lA[e - nB] = vit_log(A[e - nB]);
        } else {
            lpi[e - nB - nA] = vit_log(pi[e - nB - nA]);
        }
    }
}

// Packed backpointer row of one step and lane on the blocked layouts.  N = 4: psi_t(j) in bits [2j, 2j + 2) (one byte).
// Left-to-right N = 8 / 16: bit j set <=> psi_t(j) = j - 1, clear <=> psi_t(j) = j (one / two bytes).
template <int NS>
using VitRow = typename std::conditional<NS == 16, uint16_t, uint8_t>::type;

template <int NS>
__device__ __forceinline__ int vit_prev(unsigned row, int s) {
    if (NS == 4) return (int)((row >> (2 * s)) & 3u);
    return s - (int)((row >> s) & 1u);
}

// chunk c of row `row` of a [rows][NS] fp64 table stored as double2[rows * NS / 2], XOR-swizzled as Ltr<NS>::swz so that
// the random rows of 32 lanes spread over the banks
template <int NS>
__device__ __forceinline__ int vit_swz(unsigned row, int c) {
    constexpr int CPR = NS / 2;
    return (int)row * CPR + (c ^ (int)((row / (8 / CPR)) & (CPR - 1)));
}

// The path of one sequence, written from its last frame down: bytes are gathered into 32-bit words so that the
// scattered per-lane stores are four times fewer.  `p` (the path buffer) is 4-byte aligned.
struct PathWriter {
    int8_t *p;
    uint32_t acc = 0;
    int n = 0;
    __device__ __forceinline__ void put(int64_t q, int8_t v) {  // q = position of this frame, descending by one per call
        acc = (acc << 8) | (uint8_t)v;
        ++n;
        if ((q & 3) == 0) flush(q);
    }
    __device__ __forceinline__ void flush(int64_t q) {  // the n gathered bytes belong at [q, q + n)
        if (n == 4) {
            *reinterpret_cast<uint32_t *>(p + q) = acc;
        } else {
            for (int k = 0; k < n; ++k) p[q + k] = (int8_t)(acc >> (8 * k));
        }
        acc = 0;
        n = 0;
    }
};

// ---------------------------------------------------------------- one utterance per thread (blocked layouts)
// grid = (CTA work items (one model each), CTAs per item); B^T of the item's model in shared memory ([M][NS] fp64 log
// values).
// bp == nullptr: score only (no backpointers, no last state).
template <int NS, bool BIDIAG>
__global__ void __launch_bounds__(VIT_THREADS)
k_viterbiB(const CtaWork *__restrict__ work, const Blk *__restrict__ blks, const uint4 *__restrict__ obs_blk,
           const int32_t *__restrict__ len_sorted, const int32_t *__restrict__ order, const double *__restrict__ lpi,
           const double *__restrict__ lA, const double *__restrict__ lBt, int M, double *__restrict__ score_out,
           int8_t *__restrict__ last_out, VitRow<NS> *__restrict__ bp) {
    static_assert(NS == 4 || (BIDIAG && (NS == 8 || NS == 16)), "blocked Viterbi: N = 4, or left-to-right N = 8 / 16");
    using S16 = Sym<uint16_t>;
    constexpr int CPR = NS / 2;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double2 *sB = reinterpret_cast<double2 *>(smem_raw);
    const CtaWork cw = work[blockIdx.x];
    const int w = cw.word;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    {
        const double2 *src = reinterpret_cast<const double2 *>(lBt + (size_t)w * M * NS);
        for (int e = threadIdx.x; e < M * CPR; e += VIT_THREADS) sB[vit_swz<NS>((unsigned)(e / CPR), e % CPR)] = __ldg(src + e);
    }
    // dense: la[i * NS + j] = log a_ij; left-to-right: la[i] = log a_ii, la[NS + i] = log a_i,i+1
    double la[BIDIAG ? 2 * NS : NS * NS];
    const double *lAw = lA + (size_t)w * NS * NS;
#pragma unroll
    for (int i = 0; i < NS; ++i) {
        if (BIDIAG) {
            la[i] = __ldg(lAw + i * NS + i);
            la[NS + i] = (i + 1 < NS) ? __ldg(lAw + i * NS + i + 1) : neg_inf();
        } else {
#pragma unroll
            for (int j = 0; j < NS; ++j) la[i * NS + j] = __ldg(lAw + i * NS + j);
        }
    }
    const double *lpiw = lpi + (size_t)w * NS;
    __syncthreads();
    constexpr int NW = VIT_THREADS / 32;
    // the item's blocks are shared by gridDim.y CTAs (every split-th block: equal shares of the length-sorted blocks),
    // and each CTA's warps take theirs in serpentine order, as in k_bw_fwdL
    const int split = gridDim.y, nk = (cw.blk_end - cw.blk_begin - (int)blockIdx.y + split - 1) / split;
    for (int rb = 0, rnd = 0; rb < nk; rb += NW, ++rnd) {
        const int k = rb + ((rnd & 1) ? NW - 1 - warp : warp);
        if (k >= nk) continue;
        const Blk bk = blks[cw.blk_begin + k * split + (int)blockIdx.y];
        const int T = lane < bk.nseq ? len_sorted[bk.first + lane] : 0;
        VitRow<NS> *bpl = bp ? bp + (size_t)bk.spill_base * 32 + lane : nullptr;
        const uint4 *op = obs_blk + bk.obs_base + lane;
        double d[NS];
#pragma unroll
        for (int j = 0; j < NS; ++j) d[j] = neg_inf();
        const int nch = (bk.tmax + SPC4 - 1) / SPC4;
        uint4 wnext = nch > 0 ? __ldg(op) : make_uint4(0, 0, 0, 0);
        for (int c = 0; c < nch; ++c) {
            uint4 wc = wnext;
            if (c + 1 < nch) wnext = __ldg(op + (size_t)(c + 1) * 32);
#pragma unroll 1
            for (int s = 0; s < SPC4; ++s) {
                const int t = c * SPC4 + s;
                const unsigned sym = S16::pop_front(wc) & SYM_MASK;
                if (t >= T) continue;
                double lb[NS];
#pragma unroll
                for (int q = 0; q < CPR; ++q) {
                    const double2 x = sB[vit_swz<NS>(sym, q)];
                    lb[2 * q] = x.x;
                    lb[2 * q + 1] = x.y;
                }
                if (t == 0) {
#pragma unroll
                    for (int j = 0; j < NS; ++j) d[j] = __ldg(lpiw + j) + lb[j];
                    continue;
                }
                unsigned row = 0u;
                if (BIDIAG) {
                    // candidates i = j - 1 (scanned first) and i = j: the stay wins only if strictly larger
#pragma unroll
                    for (int j = NS - 1; j > 0; --j) {
                        const double mv = d[j - 1] + la[NS + j - 1], st = d[j] + la[j];
                        const bool stay = st > mv;
                        if (NS == 4) row |= (unsigned)(stay ? j : j - 1) << (2 * j);
                        else row |= (stay ? 0u : 1u) << j;
                        d[j] = (stay ? st : mv) + lb[j];
                    }
                    d[0] = (d[0] + la[0]) + lb[0];
                } else {
                    double nd[NS];
#pragma unroll
                    for (int j = 0; j < NS; ++j) {
                        double best = d[0] + la[j];
                        unsigned arg = 0u;
#pragma unroll
                        for (int i = 1; i < NS; ++i) {
                            const double v = d[i] + la[i * NS + j];
                            if (v > best) { best = v; arg = (unsigned)i; }
                        }
                        row |= arg << (2 * j);
                        nd[j] = best + lb[j];
                    }
#pragma unroll
                    for (int j = 0; j < NS; ++j) d[j] = nd[j];
                }
                if (bpl) bpl[(size_t)t * 32] = (VitRow<NS>)row;
            }
        }
        if (lane < bk.nseq) {
            double best = d[0];
            int arg = 0;
#pragma unroll
            for (int j = 1; j < NS; ++j)
                if (d[j] > best) { best = d[j]; arg = j; }
            score_out[order[bk.first + lane]] = best;
            if (last_out) last_out[bk.first + lane] = (int8_t)(best > neg_inf() ? arg : -1);
        }
    }
}

// one warp per 32-sequence block, lane = sequence: every step's row read is one coalesced 32- / 64-byte load
template <int NS>
__global__ void __launch_bounds__(VIT_THREADS)
k_vit_backtraceB(const Blk *__restrict__ blks, int nblk, const int32_t *__restrict__ len_sorted,
                 const int64_t *__restrict__ off_sorted, const int8_t *__restrict__ last, const VitRow<NS> *__restrict__ bp,
                 int8_t *__restrict__ path) {
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * (VIT_THREADS / 32) + (threadIdx.x >> 5);
    if (b >= nblk) return;
    const Blk bk = blks[b];
    if (lane >= bk.nseq) return;
    const int64_t i = (int64_t)bk.first + lane;
    const int T = len_sorted[i];
    const int64_t off = off_sorted[i];
    const VitRow<NS> *bpl = bp + (size_t)bk.spill_base * 32 + lane;
    int st = last[i];
    PathWriter pw{path};
    for (int t = T - 1; t >= 0; --t) {
        pw.put(off + t, (int8_t)st);
        if (t > 0 && st >= 0) st = vit_prev<NS>((unsigned)bpl[(size_t)t * 32], st);
    }
    if (pw.n) pw.flush(off);
}

// ---------------------------------------------------------------- lanes = states (generic layout)
// NP lanes per sequence (lane j = state j), 32 / NP sequences per warp; sequence r is decoded against model word[r].
template <int NP, typename SymT>
__global__ void __launch_bounds__(BW_THREADS)
k_viterbiG(const SymT *__restrict__ obs, const int64_t *__restrict__ off_sorted, const int32_t *__restrict__ len_sorted,
           const int32_t *__restrict__ word_sorted, const int32_t *__restrict__ order, const int64_t *__restrict__ foff,
           int64_t U, int64_t per_group, int N, int M, const double *__restrict__ lpi, const double *__restrict__ lA,
           const double *__restrict__ lBt, double *__restrict__ score_out, int8_t *__restrict__ last_out,
           uint8_t *__restrict__ bp) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int GPW = 32 / NP;
    const int j = lane % NP, gbase = lane - j;
    const int64_t group = ((int64_t)blockIdx.x * BW_WARPS + warp) * GPW + lane / NP;
    for (int64_t k = 0; k < per_group; ++k) {
        const int64_t r = group * per_group + k;
        const int T = r < U ? len_sorted[r] : 0;
        const int Tw = warp_max_int(T);
        if (Tw == 0) continue;
        const int w = T > 0 ? word_sorted[r] : 0;
        const bool st = T > 0 && j < N;
        double lcol[NP];  // log a_ij of this lane's state j
#pragma unroll
        for (int i = 0; i < NP; ++i) lcol[i] = (st && i < N) ? __ldg(lA + ((size_t)w * N + i) * N + j) : neg_inf();
        const SymT *o = obs + (T > 0 ? off_sorted[r] : 0);
        const double *lBw = lBt + (size_t)w * M * N;
        uint8_t *bpr = (bp && st) ? bp + (size_t)foff[r] * N + j : nullptr;
        double d = neg_inf();
        for (int t = 0; t < Tw; ++t) {
            const double lb = (st && t < T) ? __ldg(lBw + (size_t)o[t] * N + j) : neg_inf();
            if (t == 0) {
                d = st ? __ldg(lpi + (size_t)w * N + j) + lb : neg_inf();
                continue;
            }
            double best = __shfl_sync(0xffffffffu, d, gbase) + lcol[0];
            int arg = 0;
#pragma unroll
            for (int i = 1; i < NP; ++i) {
                const double v = __shfl_sync(0xffffffffu, d, gbase + i) + lcol[i];
                if (v > best) { best = v; arg = i; }
            }
            if (st && t < T) {
                d = best + lb;
                if (bpr) bpr[(size_t)t * N] = (uint8_t)arg;
            }
        }
        // last state: the smallest j with the largest delta (pairs (value, state) reduced over the group)
        double best = st ? d : neg_inf();
        int arg = j;
#pragma unroll
        for (int o2 = NP / 2; o2 > 0; o2 >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, best, o2);
            const int oa = __shfl_xor_sync(0xffffffffu, arg, o2);
            if (ov > best || (ov == best && oa < arg)) { best = ov; arg = oa; }
        }
        if (T > 0 && j == 0) {
            score_out[order[r]] = best;
            if (last_out) last_out[r] = (int8_t)(best > neg_inf() ? arg : -1);
        }
    }
}

// one thread per sequence
__global__ void __launch_bounds__(VIT_THREADS)
k_vit_backtraceG(int64_t U, int N, const int32_t *__restrict__ len_sorted, const int64_t *__restrict__ off_sorted,
                 const int64_t *__restrict__ foff, const int8_t *__restrict__ last, const uint8_t *__restrict__ bp,
                 int8_t *__restrict__ path) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= U) return;
    const int T = len_sorted[r];
    const int64_t off = off_sorted[r];
    const uint8_t *bpr = bp + (size_t)foff[r] * N;
    int st = last[r];
    PathWriter pw{path};
    for (int t = T - 1; t >= 0; --t) {
        pw.put(off + t, (int8_t)st);
        if (t > 0 && st >= 0) st = bpr[(size_t)t * N + st];
    }
    if (pw.n) pw.flush(off);
}

}  // namespace hmmb

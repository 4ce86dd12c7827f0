// Left-to-right Baum-Welch E-step kernels for N = 8 / 16 states (BASELINE config 4: 1000
// words, N = 16, M = 1024): one sequence per THREAD, 32 same-word sequences per warp in
// lock-step, for models whose transition matrix is upper-bidiagonal (a_ij > 0 only for
// j = i or j = i + 1 — the reference's left-to-right topology, HMM/hmm_training.py:307-312,
// which re-estimation preserves because zeros of A stay zeros, :450-455).
//
// Why not lanes = states (bw_kernels.cuh)?  With 16 lanes per sequence every reduction over
// states is a shuffle tree and a warp-step moves only 2 frames: the generic kernels execute
// ~140 warp-instructions per frame (ncu, profiles/r1e_*).  With a thread per sequence the
// bidiagonal mat-vec is 31 register FMAs, every reduction is in registers, and a warp-step
// moves 32 frames: ~6-10 warp-instructions per frame.
//
//   k_bw_fwdL   scaled forward pass; B^T of the CTA's word in shared memory ([M][NS] fp64,
//               16-byte chunks XOR-swizzled so that 32 random rows spread over all banks);
//               alpha-hat spilled [block][t][chunk][lane] as coalesced 16-byte streaming stores.
//   k_bw_bwdL   backward pass fused with gamma / xi / emission-count accumulation.  Each lane's
//               gamma_t row (NS fp64 = 128 B at NS = 16) is staged in shared memory (padded
//               rows, conflict-free), re-read with lanes = states and added to the word's count
//               row in the global accumulator with coalesced fp64 REDs (the L2 atomic units),
//               which frees the shared memory a [M][NS] count table would need for B^T.
//               Measured on B200 (scripts/microbench2.cu, clk per row per SM): coalesced RED
//               rows with lanes = states 7.8, one TMA bulk reduction per lane
//               (cp.reduce.async.bulk .add.f64) 7.6, shared table + row locks 8.9, shared CAS
//               atomics 11.8, per-element global RED 24.4.  The TMA instruction takes its
//               operands from uniform registers, so a warp issues its 32 reductions in a serial
//               ELECT / R2UR / UBLKRED loop (ncu, profiles/r1i_*: 42 % of the kernel's
//               instructions): config 4 backward 5.55 ms with it against 4.54 ms with the RED
//               rows.  That variant was removed; it is in the history at commit 03a55a2.
//
// Numerics are those of the N = 4 kernels (bw4_kernels.cuh): exact power-of-two rescale,
// smallest-denormal FMA addends that keep "value > 0 <=> the reference's log value is
// finite", structural alive-masks, scalar error bound with hand-over to the exact log-space
// kernel, careful out-of-line step for everything unusual.
#pragma once

#include "bw4_kernels.cuh"

namespace hmmb {

constexpr int LTR_WARPS = 8;
constexpr int LTR_THREADS = LTR_WARPS * 32;
constexpr int LTR_MAX_SYM = 1 << SYM_BITS;   // codewords share the packed u16 layout of the N = 4 path
// steps ahead of use for the alpha-hat L2 prefetch (3 / 6 / 12 and an extra L1 prefetch measured
// within 6 % of each other on config 4: the backward pass is not waiting on the spill)
constexpr int BWDL_L2_PREFETCH = 6;

template <int NS>
struct Ltr {
    static_assert(NS == 8 || NS == 16, "left-to-right kernels are instantiated for 8 and 16 states");
    static constexpr int CPR = NS / 2;                  // 16-byte chunks per row
    static constexpr unsigned FULL = (1u << NS) - 1u;
    static constexpr int ROWB = NS * 8 + 16;            // padded staging row (bytes): conflict-free per quarter-warp
    // chunk c of row `row` of a [rows][NS] fp64 table stored as double2[rows * CPR]
    static __device__ __forceinline__ int swz(unsigned row, int c) {
        return (int)row * CPR + (c ^ (int)((row / (8 / CPR)) & (CPR - 1)));
    }
};

template <int N>
__device__ __forceinline__ double tree_sum(const double (&x)[N]) {
    double t[N / 2];
#pragma unroll
    for (int i = 0; i < N / 2; ++i) t[i] = x[i] + x[i + N / 2];
#pragma unroll
    for (int s = N / 4; s > 0; s >>= 1) {
#pragma unroll
        for (int i = 0; i < s; ++i) t[i] += t[i + s];
    }
    return t[0];
}

// all NS non-negative doubles strictly positive? (integer pipe)
template <int N>
__device__ __forceinline__ bool all_posN(const double (&x)[N]) {
    unsigned m = 0xffffffffu;
#pragma unroll
    for (int i = 0; i < N; ++i) m = min(m, (unsigned)__double2hiint(x[i]) | (unsigned)__double2loint(x[i]));
    return m != 0u;
}

// largest high word of NS non-negative doubles: max_hiN(x) >= hi(c) <=> some x_i >= c (c a power of two)
template <int N>
__device__ __forceinline__ unsigned max_hiN(const double (&x)[N]) {
    unsigned m = 0u;
#pragma unroll
    for (int i = 0; i < N; ++i) m = max(m, (unsigned)__double2hiint(x[i]));
    return m;
}

// Exponent-split products (see exact_products4): out_j = n_j*b_j * 2^-E.  Arrays in local memory.
template <int NS>
__device__ __noinline__ int exact_productsN(const double *nn, const double *bb, double *out, int *E_out) {
    double m[NS];
    int e[NS];
    int E = INT_MIN;
    for (int j = 0; j < NS; ++j) {
        m[j] = 0.0;
        e[j] = INT_MIN;
        out[j] = 0.0;
        if (nn[j] > 0.0 && bb[j] > 0.0) {
            frexp_prod(nn[j], bb[j], m[j], e[j]);
            E = max(E, e[j]);
        }
    }
    *E_out = 0;
    if (E == INT_MIN) return 0;
    int code = 1;
    for (int j = 0; j < NS; ++j) {
        if (e[j] != INT_MIN) {
            double v = ldexp(m[j], max(e[j] - E, -1200));
            if (v == 0.0) v = tiny_pos();
            out[j] = v;
            if (e[j] >= E - 64 && nn[j] < SUBNORMAL_LIMIT) code = 2;
        }
    }
    *E_out = E;
    return code;
}

// ---------------------------------------------------------------- forward
// One sequence per lane.  as[i] = a_ii, an[i] = a_i,i+1 (an[NS-1] = 0); piw = the word's pi in
// global memory (read at t = 0 only); sB = swizzled B^T, sBmax[sym] = max_j b_j(sym),
// sBmask[sym] = {j : b_j(sym) > 0}; selfm / nextm = {i : a_ii > 0} / {i : a_i,i+1 > 0}.
// Replaces calculate_log_alpha (HMM/hmm_training.py:122-160) and the alpha init (:357-360);
// returns log P(O|lambda) (:376-377), -inf if structurally impossible, NaN = hand over to the
// exact log-space kernel.  allfull = every step had all NS states alive and a scale >= 1, i.e.
// every spilled alpha-hat is strictly positive (the backward pass then skips that test).
// PERSTATE = false (first pass): the scalar error bound of fwd4_run, ~5 instructions per step; rigorous but loose — it
// assumes the error sits in the most probable state, so over a few thousand frames of peaked emissions it drifts
// up to the limit although nothing is wrong.  A lane that trips it is simply run again with PERSTATE = true: per-state
// bounds e_j following the exact linear recursion of the values, kept in local memory (volatile: no registers in the
// common path), born only where a zero / denormal value is actually produced.  Only what that pass marks goes to the
// exact log-space kernel.
template <int NS, bool SPILL, bool PERSTATE = false>
__device__ __forceinline__ double fwdL_run(int T, int tmax, const uint4 *__restrict__ op,
                                           const double2 *__restrict__ sB, const double *__restrict__ sBmax,
                                           const unsigned short *__restrict__ sBmask, const double (&as)[NS],
                                           const double (&an)[NS], const double *__restrict__ piw, double rmax,
                                           unsigned selfm, unsigned nextm, unsigned pmask, double2 *__restrict__ sp,
                                           bool &allfull) {
    using L = Ltr<NS>;
    using S16 = Sym<uint16_t>;
    double al[NS];
#pragma unroll
    for (int j = 0; j < NS; ++j) al[j] = 0.0;
    double E = 0.0;          // !PERSTATE: scalar error bound, units of 2^-1000
    volatile double ev[NS];  // PERSTATE: per-state bounds, only touched once a denormal was born (`tainted`)
    bool tainted = false;
    long long esum = 0;
    unsigned m = 0u;
    bool stop = false, allf = true;
    double ll = neg_inf();
    const double tiny = tiny_pos();
    const int nch = (tmax + SPC4 - 1) / SPC4;
    uint4 wnext = nch > 0 ? __ldg(op) : make_uint4(0, 0, 0, 0);
    for (int c = 0; c < nch; ++c) {
        uint4 w = wnext;
        if (c + 1 < nch) wnext = __ldg(op + (size_t)(c + 1) * 32);
#pragma unroll 1
        for (int s = 0; s < SPC4; ++s) {
            const int t = c * SPC4 + s;
            const unsigned sym = S16::pop_front(w) & SYM_MASK;
            if (t < T && !stop) {
                double b[NS];
#pragma unroll
                for (int q = 0; q < L::CPR; ++q) {
                    const double2 x = sB[L::swz(sym, q)];
                    b[2 * q] = x.x;
                    b[2 * q + 1] = x.y;
                }
                const unsigned r = (t == 0) ? pmask : (((m & selfm) | ((m & nextm) << 1)) & L::FULL);
                m = r & (unsigned)sBmask[sym];
                double at[NS];
                unsigned subm = 0u;  // alive states whose value came out zero / denormal: an absolute error is born here
                if (m == L::FULL && t > 0) {
                    // ---- every state alive (the usual case)
                    at[0] = fma(fma(al[0], as[0], tiny), b[0], tiny);
#pragma unroll
                    for (int j = 1; j < NS; ++j) at[j] = fma(fma(al[j], as[j], fma(al[j - 1], an[j - 1], tiny)), b[j], tiny);
                    if (PERSTATE) {
#pragma unroll
                        for (int j = 0; j < NS; ++j) subm |= is_sub(at[j]) ? (1u << j) : 0u;
                    }
                } else if (m == 0u) {
                    stop = true;  // no state can emit o_t: log P = -inf (:155-160)
                    allf = false;
#pragma unroll
                    for (int j = 0; j < NS; ++j) at[j] = 0.0;
                } else {
                    // ---- first step, or some states structurally dead: masked addends keep them exactly 0
                    allf = allf && (m == L::FULL);
#pragma unroll
                    for (int j = 0; j < NS; ++j) {
                        double n;
                        if (t == 0) n = __ldg(piw + j);
                        else if (j == 0) n = fma(al[0], as[0], tiny_if(r, 0));
                        else n = fma(al[j], as[j], fma(al[j - 1], an[j - 1], tiny_if(r, j)));
                        at[j] = fma(n, b[j], tiny_if(m, j));
                        if (PERSTATE && t > 0 && ((m >> j) & 1u) && is_sub(at[j])) subm |= 1u << j;  // (pi * b at t = 0 is one exact product)
                    }
                }
                double ssum = tree_sum<NS>(at);
                if (!stop && !(ssum >= TINY_STEP)) {
                    // ---- the whole step is tiny: exponent-split products (rare; arrays in local memory)
                    double tn[NS], tb[NS], to[NS];
                    for (int j = 0; j < NS; ++j) {
                        double n;
                        if (t == 0) n = __ldg(piw + j);
                        else if (j == 0) n = fma(al[0], as[0], tiny_if(r, 0));
                        else n = fma(al[j], as[j], fma(al[j - 1], an[j - 1], tiny_if(r, j)));
                        tn[j] = n;
                        tb[j] = b[j];
                    }
                    int Ex;
                    const int code = exact_productsN<NS>(tn, tb, to, &Ex);
                    if (code == 0) {
                        stop = true;
                    } else if ((code == 2 && t > 0) || tainted || E > 0.0) {
                        stop = true;  // the surviving states had lost their bits: exact path
                        ll = nan_mark();
                    } else {
                        esum += Ex;
#pragma unroll
                        for (int j = 0; j < NS; ++j) at[j] = to[j];
                        ssum = tree_sum<NS>(at);
                    }
                    allf = false;
                }
                if (!stop) {
                    const double sc = pow2_rescale(ssum, esum);
                    allf = allf && (__double2hiint(sc) >= 0x3ff00000);  // scale >= 1: a denormal alpha cannot be flushed
#pragma unroll
                    for (int j = 0; j < NS; ++j) al[j] = at[j] * sc;
                    if (!PERSTATE) {
                        E = fma(E, rmax * sBmax[sym], (double)NS * ERR_UNIT) * sc;
                        if (!(E <= ERR_LIMIT)) {
                            stop = true;
                            ll = nan_mark();
                        }
                    } else if (subm != 0u || tainted) {
                        // e'_j = (b_j(o_t) * (e_j a_jj + e_j-1 a_j-1,j) + seed_j) * scale, seed_j = 2^-1074 where a denormal was born
                        if (!tainted) {
#pragma unroll
                            for (int j = 0; j < NS; ++j) ev[j] = 0.0;
                            tainted = true;
                        }
                        double etot = 0.0, eprev = 0.0;
#pragma unroll
                        for (int q = 0; q < L::CPR; ++q) {
                            const double2 x = sB[L::swz(sym, q)];  // (re-read: b[] is not kept alive for this rare path)
#pragma unroll
                            for (int h = 0; h < 2; ++h) {
                                const int j = 2 * q + h;
                                const double ej = ev[j];
                                const double f = fma(ej, as[j], j > 0 ? eprev * an[j > 0 ? j - 1 : 0] : 0.0);
                                eprev = ej;
                                const double en = fma(f, h ? x.y : x.x, ((subm >> j) & 1u) ? ERR_UNIT : 0.0) * sc;
                                ev[j] = en;
                                etot += en;
                            }
                        }
                        if (!(etot <= ERR_LIMIT)) {
                            stop = true;
                            ll = nan_mark();
                        }
                    }
                    if (t == T - 1 && !stop) ll = log(tree_sum<NS>(al)) + (double)esum * LN2;
                }
                // a stopped sequence is skipped by the backward pass: nothing more to spill
                if (SPILL && !stop) {
#pragma unroll
                    for (int q = 0; q < L::CPR; ++q)
                        __stcs(sp + ((size_t)t * L::CPR + q) * 32, make_double2(al[2 * q], al[2 * q + 1]));
                }
            }
        }
    }
    allfull = allf && !stop;
    return ll;
}

// CTA prologue: B^T of word w -> swizzled shared memory, for the forward pass together with the
// per-codeword max / support mask (CPR consecutive threads hold one row).
template <int NS, bool WANT_MAX>
__device__ __forceinline__ void load_BtL(const double *__restrict__ Btw, int M, double2 *sB, double *sBmax,
                                         unsigned short *sBmask) {
    using L = Ltr<NS>;
    const int tid = threadIdx.x;
    const double2 *src = reinterpret_cast<const double2 *>(Btw);
    const int total = M * L::CPR;
    for (int e0 = 0; e0 < total; e0 += LTR_THREADS) {
        const int e = e0 + tid;
        const bool valid = e < total;
        const unsigned row = (unsigned)(e / L::CPR);
        const int c = e % L::CPR;
        double2 x = make_double2(0.0, 0.0);
        if (valid) {
            x = __ldg(src + e);
            sB[L::swz(row, c)] = x;
        }
        if (WANT_MAX) {
            double mx = fmax(x.x, x.y);
            unsigned mk = (x.x > 0.0 ? 1u : 0u) << (2 * c) | (x.y > 0.0 ? 1u : 0u) << (2 * c + 1);
#pragma unroll
            for (int o = L::CPR / 2; o > 0; o >>= 1) {
                mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
                mk |= __shfl_xor_sync(0xffffffffu, mk, o);
            }
            if (valid && c == 0) { sBmax[row] = mx; sBmask[row] = (unsigned short)mk; }
        }
    }
}

// a_ii / a_i,i+1 of one model into registers with the largest row sum and the support masks
template <int NS>
__device__ __forceinline__ void load_modelL(const double *__restrict__ Aw, const double *__restrict__ piw, double (&as)[NS],
                                            double (&an)[NS], double &rmax, unsigned &selfm, unsigned &nextm,
                                            unsigned &pmask) {
    rmax = 0.0;
    selfm = nextm = pmask = 0u;
#pragma unroll
    for (int i = 0; i < NS; ++i) {
        as[i] = __ldg(Aw + i * NS + i);
        an[i] = (i + 1 < NS) ? __ldg(Aw + i * NS + i + 1) : 0.0;
        rmax = fmax(rmax, as[i] + an[i]);
        selfm |= (as[i] > 0.0 ? 1u : 0u) << i;
        nextm |= (an[i] > 0.0 ? 1u : 0u) << i;
        pmask |= (__ldg(piw + i) > 0.0 ? 1u : 0u) << i;
    }
}

template <int NS>
__global__ void __launch_bounds__(LTR_THREADS, NS == 8 ? 2 : 1)
k_bw_fwdL(const CtaWork *__restrict__ work, const Blk *__restrict__ blks, const uint4 *__restrict__ obs_blk,
          const int32_t *__restrict__ len_sorted, const double *__restrict__ pi, const double *__restrict__ A,
          const double *__restrict__ Bt, int M, double2 *__restrict__ spill, double *__restrict__ ll_seq,
          const int32_t *__restrict__ active, uint8_t *__restrict__ flag, uint8_t *__restrict__ allfull) {
    using L = Ltr<NS>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double2 *sB = reinterpret_cast<double2 *>(smem_raw);                      // [M * CPR] swizzled B^T
    double *sBmax = reinterpret_cast<double *>(sB + (size_t)M * L::CPR);      // [M]
    unsigned short *sBmask = reinterpret_cast<unsigned short *>(sBmax + M);   // [M]
    const CtaWork cw = work[blockIdx.x];
    if (!active[cw.word]) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    load_BtL<NS, true>(Bt + (size_t)cw.word * M * NS, M, sB, sBmax, sBmask);
    const double *piw = pi + (size_t)cw.word * NS;
    double as[NS], an[NS];
    double rmax;
    unsigned selfm, nextm, pmask;
    load_modelL<NS>(A + (size_t)cw.word * NS * NS, piw, as, an, rmax, selfm, nextm, pmask);
    __syncthreads();
    // blocks are sorted by length: warps take them in serpentine order (0..7, 7..0, ...) so that every warp of the CTA
    // gets about the same number of steps (plain striding gave warp 0 the longest block of every round: with four
    // rounds per CTA the last warp idled for a tenth of the kernel at the CTA's final barrier)
    for (int rb = cw.blk_begin, rnd = 0; rb < cw.blk_end; rb += LTR_WARPS, ++rnd) {
        const int b = rb + ((rnd & 1) ? LTR_WARPS - 1 - warp : warp);
        if (b >= cw.blk_end) continue;
        const Blk bk = blks[b];
        int T = lane < bk.nseq ? len_sorted[bk.first + lane] : 0;
        if (T > 0 && flag[bk.first + lane]) T = 0;  // handled by the exact log-space kernel
        bool af = false;
        double ll = fwdL_run<NS, true>(T, bk.tmax, obs_blk + bk.obs_base + lane, sB, sBmax, sBmask, as, an, piw, rmax,
                                       selfm, nextm, pmask, spill + (size_t)bk.spill_base * L::CPR * 32 + lane, af);
        if (__any_sync(0xffffffffu, T > 0 && ll != ll)) {  // (rare) the marked lanes again, with per-state bounds
            bool af2 = false;
            const double ll2 = fwdL_run<NS, true, true>((T > 0 && ll != ll) ? T : 0, bk.tmax, obs_blk + bk.obs_base + lane, sB, sBmax,
                                                        sBmask, as, an, piw, rmax, selfm, nextm, pmask,
                                                        spill + (size_t)bk.spill_base * L::CPR * 32 + lane, af2);
            if (T > 0 && ll != ll) { ll = ll2; af = af2; }
        }
        if (T > 0) {
            ll_seq[bk.first + lane] = ll;
            allfull[bk.first + lane] = af ? 1 : 0;
            if (ll != ll) raise_flag(flag, bk.first + lane);  // precision guard: hand over (sticky)
        }
    }
}

// Recognition with left-to-right models (replaces calculate_log_likelihood, HMM/hmm_testing.py:49-104):
// grid = (utterance work items, models); the CTA keeps one model's B^T in shared memory and
// scores its 32-utterance blocks with the forward recursion above (no spill).
template <int NS>
__global__ void __launch_bounds__(LTR_THREADS, NS == 8 ? 2 : 1)
k_scoreL(const CtaWork *__restrict__ work, const Blk *__restrict__ blks, const uint4 *__restrict__ obs_blk,
         const int32_t *__restrict__ len_sorted, const int32_t *__restrict__ order, const double *__restrict__ pi,
         const double *__restrict__ A, const double *__restrict__ Bt, int M, int W, double *__restrict__ ll_out,
         int32_t *__restrict__ any_nan) {
    using L = Ltr<NS>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double2 *sB = reinterpret_cast<double2 *>(smem_raw);
    double *sBmax = reinterpret_cast<double *>(sB + (size_t)M * L::CPR);
    unsigned short *sBmask = reinterpret_cast<unsigned short *>(sBmax + M);
    const CtaWork cw = work[blockIdx.x];
    const int w = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    load_BtL<NS, true>(Bt + (size_t)w * M * NS, M, sB, sBmax, sBmask);
    const double *piw = pi + (size_t)w * NS;
    double as[NS], an[NS];
    double rmax;
    unsigned selfm, nextm, pmask;
    load_modelL<NS>(A + (size_t)w * NS * NS, piw, as, an, rmax, selfm, nextm, pmask);
    __syncthreads();
    for (int b = cw.blk_begin + warp; b < cw.blk_end; b += LTR_WARPS) {
        const Blk bk = blks[b];
        const int T = lane < bk.nseq ? len_sorted[bk.first + lane] : 0;
        bool af;
        double ll = fwdL_run<NS, false>(T, bk.tmax, obs_blk + bk.obs_base + lane, sB, sBmax, sBmask, as, an, piw, rmax,
                                        selfm, nextm, pmask, nullptr, af);
        if (__any_sync(0xffffffffu, T > 0 && ll != ll)) {  // (rare) the marked lanes again, with per-state bounds
            const double ll2 = fwdL_run<NS, false, true>((T > 0 && ll != ll) ? T : 0, bk.tmax, obs_blk + bk.obs_base + lane, sB, sBmax,
                                                         sBmask, as, an, piw, rmax, selfm, nextm, pmask, nullptr, af);
            if (T > 0 && ll != ll) ll = ll2;
        }
        if (lane < bk.nseq) {
            ll_out[(size_t)order[bk.first + lane] * W + w] = ll;
            if (ll != ll) *any_nan = 1;  // precision guard marked this pair: k_score_exact has work to do
        }
    }
}

// ---------------------------------------------------------------- backward + accumulate
template <int NS>
struct BwdLState {
    double v[NS];           // v_j = b_j(o_{t+1}) * beta-hat_{t+1}(j)
    double Xs[NS], Xn[NS];  // sum_t u_i v_i and sum_t u_i v_{i+1} (a_ii / a_i,i+1 applied at the flush)
    unsigned seenS, seenN;  // states i for which a finite xi_t(i,i) / xi_t(i,i+1) term existed
    bool imprecise, vpos;
};

// Careful version of one backward step (all clamps, structural tests, precision hand-over) on
// a copy of the lane's state in local memory; generic-N restatement of bwd4_step_slow.
// sA = {a_ii [NS], a_i,i+1 [NS]} in shared memory.  Writes gamma_t to g[].
template <int NS>
__device__ __noinline__ void bwdL_step_slow(BwdLState<NS> &st, const double *__restrict__ sA,
                                            const double2 *__restrict__ sB, unsigned sym, bool last, const double *al,
                                            double *g) {
    using L = Ltr<NS>;
    double h[NS], w[NS];
    if (last) {
        for (int i = 0; i < NS; ++i) { h[i] = 1.0; w[i] = 0.0; }  // log beta_{T-1} = 0 (:363)
    } else {
        // un-normalised beta_t(i) = sum_j a_ij b_j(o_{t+1}) beta_{t+1}(j)  (:163-199)
        double q[NS], qs = 0.0;
        for (int i = 0; i < NS; ++i) {
            const double a_s = sA[i], a_n = (i + 1 < NS) ? sA[NS + i] : 0.0;
            const double v_s = st.v[i], v_n = (i + 1 < NS) ? st.v[i + 1] : 0.0;
            double x = a_s * v_s + a_n * v_n;
            if (x == 0.0 && ((a_s > 0.0 && v_s > 0.0) || (a_n > 0.0 && v_n > 0.0))) x = tiny_pos();
            q[i] = x;
            qs += x;
        }
        const double sc = qs > 0.0 ? pow2_rescale_noacc(qs) : 1.0;
        for (int i = 0; i < NS; ++i) {
            h[i] = q[i] * sc;
            if (h[i] == 0.0 && q[i] > 0.0) h[i] = tiny_pos();  // (sc < 1 must not flush a denormal marker: bw4_kernels.cuh)
            w[i] = st.v[i] * sc;
        }
    }
    // gamma_t(i) = alpha_t(i) beta_t(i) / sum_i alpha_t(i) beta_t(i)   (:389-394)
    double u[NS], norm = 0.0;
    for (int i = 0; i < NS; ++i) { u[i] = al[i]; g[i] = al[i] * h[i]; norm += g[i]; }
    double r;
    if (!(norm >= TINY_STEP)) {
        // forward and backward mass on (almost) disjoint states: redo 2^1000 larger, hand over
        st.imprecise = true;
        const double big = 0x1p500;
        norm = 0.0;
        for (int i = 0; i < NS; ++i) {
            u[i] = al[i] * big;
            g[i] = u[i] * (h[i] * big);
            w[i] *= big;
            norm += g[i];
        }
        r = norm > 0.0 ? 1.0 / norm : 0.0;
    } else {
        r = 1.0 / norm;
    }
    for (int i = 0; i < NS; ++i) {
        g[i] *= r;
        if (g[i] == 0.0 && al[i] > 0.0 && h[i] > 0.0) g[i] = tiny_pos();
    }
    if (!last) {
        // xi_t(i,j) = alpha_t(i) a_ij b_j(o_{t+1}) beta_{t+1}(j) / norm   (:397-410), j = i, i+1
        for (int i = 0; i < NS; ++i) {
            const double ui = u[i] * r;
            st.Xs[i] = fma(ui, w[i], st.Xs[i]);
            if (i + 1 < NS) st.Xn[i] = fma(ui, w[i + 1], st.Xn[i]);
            if (al[i] > 0.0) {
                if (st.v[i] > 0.0) st.seenS |= 1u << i;
                if (i + 1 < NS && st.v[i + 1] > 0.0) st.seenN |= 1u << i;
            }
        }
    }
    // v_j = b_j(o_t) beta-hat_t(j) for step t-1
    double b[NS], vs = 0.0;
    for (int q = 0; q < L::CPR; ++q) {
        const double2 x = sB[L::swz(sym, q)];
        b[2 * q] = x.x;
        b[2 * q + 1] = x.y;
    }
    for (int i = 0; i < NS; ++i) { st.v[i] = b[i] * h[i]; vs += st.v[i]; }
    if (!(vs >= TINY_STEP)) {
        // tiny emission column: exponent-split products (the scale of v is free)
        double o[NS];
        int E;
        if (exact_productsN<NS>(h, b, o, &E) == 2) st.imprecise = true;
        for (int i = 0; i < NS; ++i) st.v[i] = o[i];
    } else {
        for (int i = 0; i < NS; ++i)
            if (st.v[i] == 0.0 && b[i] > 0.0 && h[i] > 0.0) st.v[i] = tiny_pos();
    }
    bool vp = true;
    for (int i = 0; i < NS; ++i) vp = vp && (st.v[i] > 0.0);
    st.vpos = vp;
}

// Accumulator layout per word: [pi N][xi N*N][cnt M*N] (fp64, L2 atomics), N == NS.
template <int NS>
__global__ void __launch_bounds__(LTR_THREADS, NS == 8 ? 2 : 1)
k_bw_bwdL(const CtaWork *__restrict__ work, const Blk *__restrict__ blks, const uint4 *__restrict__ obs_blk,
          const int32_t *__restrict__ len_sorted, const double *__restrict__ A, const double *__restrict__ Bt, int M,
          const double2 *__restrict__ spill, const double *__restrict__ ll_seq, const int32_t *__restrict__ active,
          const int32_t *__restrict__ b_has_zero, const uint8_t *__restrict__ allfull, double *__restrict__ accum,
          int64_t astride, uint8_t *__restrict__ flag, int32_t *__restrict__ new_flags) {
    using L = Ltr<NS>;
    using S16 = Sym<uint16_t>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double2 *sB = reinterpret_cast<double2 *>(smem_raw);                                  // [M * CPR] swizzled B^T
    unsigned char *sStage = reinterpret_cast<unsigned char *>(sB + (size_t)M * L::CPR);    // [warps][32][ROWB]
    double *sA = reinterpret_cast<double *>(sStage + (size_t)LTR_WARPS * 32 * L::ROWB);   // a_ii [NS], a_i,i+1 [NS]
    double *sRed = sA + 2 * NS;                                                            // [warps][2 * NS]
    __shared__ unsigned sSeen[2];

    const CtaWork cw = work[blockIdx.x];
    if (!active[cw.word]) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    load_BtL<NS, false>(Bt + (size_t)cw.word * M * NS, M, sB, nullptr, nullptr);
    const double *Aw = A + (size_t)cw.word * NS * NS;
    if (tid < NS) {
        sA[tid] = __ldg(Aw + tid * NS + tid);
        sA[NS + tid] = (tid + 1 < NS) ? __ldg(Aw + tid * NS + tid + 1) : 0.0;
    }
    if (tid == 0) sSeen[0] = sSeen[1] = 0u;
    __syncthreads();
    // lean path precondition (structure only): B > 0 everywhere, every state has an outgoing
    // transition; whether every alpha-hat is positive comes from the forward pass (allfull)
    bool rows_ok = true;
#pragma unroll
    for (int i = 0; i < NS; ++i) rows_ok = rows_ok && (sA[i] > 0.0 || sA[NS + i] > 0.0);
    const bool lean_ok = (b_has_zero[cw.word] == 0) && rows_ok;
    const double tiny = tiny_pos();
    double *accw = accum + (size_t)cw.word * astride;
    double *acc_cnt = accw + NS + NS * NS;
    unsigned char *stage = sStage + (size_t)warp * 32 * L::ROWB + (size_t)lane * L::ROWB;
    // count flush with lanes = states: lane (fo, jj) reads state jj of staged rows fo, fo + FPI, ...
    const int flush_jj = lane % NS, flush_fo = lane / NS;
    const unsigned char *flush_src = sStage + (size_t)warp * 32 * L::ROWB + (size_t)flush_fo * L::ROWB + flush_jj * 8;
    const int flush_sym_off = NS * 8 - flush_jj * 8;  // from the lane's element to the row's padding word
    double *flush_dst = acc_cnt + flush_jj;

    double v[NS], Xs[NS], Xn[NS];
#pragma unroll
    for (int i = 0; i < NS; ++i) Xs[i] = Xn[i] = 0.0;
    unsigned seenS = 0u, seenN = 0u;

    for (int rb = cw.blk_begin, rnd = 0; rb < cw.blk_end; rb += LTR_WARPS, ++rnd) {
        const int b = rb + ((rnd & 1) ? LTR_WARPS - 1 - warp : warp);
        if (b >= cw.blk_end) continue;
        const Blk bk = blks[b];
        int T = 0;
        bool apos = false;
        if (lane < bk.nseq) {
            T = len_sorted[bk.first + lane];
            if (!(ll_seq[bk.first + lane] > neg_inf())) T = 0;  // impossible sequence: contributes nothing (:391-394)
            if (flag[bk.first + lane]) T = 0;                   // exact log-space kernel did this one
            apos = allfull[bk.first + lane] != 0;
        }
#pragma unroll
        for (int i = 0; i < NS; ++i) v[i] = 0.0;
        bool imprecise = false, vpos = false;
        const uint4 *op = obs_blk + bk.obs_base + lane;
        const double2 *sp = spill + (size_t)bk.spill_base * L::CPR * 32 + lane;
        const char *sp_line = reinterpret_cast<const char *>(spill + (size_t)bk.spill_base * L::CPR * 32) + (size_t)lane * 128;
        const int nch = (bk.tmax + SPC4 - 1) / SPC4;
        uint4 wnext = __ldg(op + (size_t)(nch - 1) * 32);
        if (T < bk.tmax) {  // this lane sits out the block's first steps (or all of them): its staged row reads as zero
            double2 *sg = reinterpret_cast<double2 *>(stage);
#pragma unroll
            for (int p = 0; p < L::CPR; ++p) sg[p] = make_double2(0.0, 0.0);
            *reinterpret_cast<unsigned *>(stage + NS * 8) = 0u;
        }
        // alpha-hat of the step to come.  Every step loads its successor's row into these registers right after its
        // own last use of them, so that the load (an L2 hit thanks to the prefetch below) is in flight during the
        // count flush and the next step's q = A v, instead of being waited for at the first product with q (that
        // wait was 14 % of the kernel's stall samples).  Unconditional: a row at or beyond a lane's own T lies
        // inside the block's spill and is never used.
        double al[NS];
        double rref = 1.0;  // 1 / sum_i alpha-hat_{T-1}(i): reference of the division-free normalisation (bw4_kernels.cuh)
#pragma unroll
        for (int q = 0; q < L::CPR; ++q) {
            const double2 x = __ldcs(sp + ((size_t)(bk.tmax - 1) * L::CPR + q) * 32);
            al[2 * q] = x.x;
            al[2 * q + 1] = x.y;
        }
        for (int c = nch - 1; c >= 0; --c) {
            uint4 w = wnext;
            if (c > 0) wnext = __ldg(op + (size_t)(c - 1) * 32);
            int s = SPC4 - 1;
            // the top chunk's unused entries are dropped here, so that the step loop has no skip branch.  (ptxas waits
            // for the alpha-hat loads of the previous iteration at the first instruction group of the loop body whatever
            // the first use is — 7-8 % of the kernel's stall samples sit there; moving the first use behind q = A v,
            // taking the all-positive test from the forward pass, or sending the rows through cp.async staging did not
            // shorten the step: DESIGN.md section 6.)
            if (c == nch - 1)
                for (const int s0 = bk.tmax - 1 - c * SPC4; s > s0; --s) S16::pop_back(w);
#pragma unroll 1
            for (; s >= 0; --s) {
                const int t = c * SPC4 + s;
                const unsigned sym = S16::pop_back(w) & SYM_MASK;
                const bool act = t < T;
                // pull the spill towards L2 well ahead
                prefetch_l2_if(sp_line + (size_t)(t - BWDL_L2_PREFETCH) * (NS * 8 * 32), t >= BWDL_L2_PREFETCH && lane * 128 < NS * 8 * 32);
                if (act) {
                    bool done = false;
                    if (lean_ok && (apos || all_posN<NS>(al))) {
                        double2 *sg = reinterpret_cast<double2 *>(stage);
                        if (t == T - 1) {
                            // first step of the recursion: beta_{T-1} = 1 (:363); gamma = alpha / sum(alpha), v = b(o_t)
                            double nv[NS];
#pragma unroll
                            for (int p = 0; p < L::CPR; ++p) {
                                const double2 x = sB[L::swz(sym, p)];
                                nv[2 * p] = x.x;
                                nv[2 * p + 1] = x.y;
                            }
                            if (max_hiN<NS>(nv) >= LEAN_MIN_HI) {
                                const double r = 1.0 / tree_sum<NS>(al);  // the one true division of the sequence
                                rref = r;
#pragma unroll
                                for (int p = 0; p < L::CPR; ++p)
                                    sg[p] = make_double2(fma(al[2 * p], r, tiny), fma(al[2 * p + 1], r, tiny));
#pragma unroll
                                for (int i = 0; i < NS; ++i) v[i] = nv[i];
                                vpos = true;
                                done = true;
                            }
                        } else if (vpos) {
                            // lean step: beta_t(i) ~ q_i = a_ii v_i + a_i,i+1 v_{i+1} (:163-199); gamma_t(i) = al_i q_i / norm
                            // (:389-394); xi_t(i,j) = al_i a_ij v_j / norm (:397-410); norm = sum_i al_i q_i.  The denormal
                            // addends keep a finite-but-underflowed log value (barely) positive.  Nothing is committed
                            // (v, Xs, Xn, the count REDs) before the three magnitude tests have passed.
                            double q[NS];
#pragma unroll
                            for (int i = 0; i < NS - 1; ++i) q[i] = fma(sA[NS + i], v[i + 1], fma(sA[i], v[i], tiny));
                            q[NS - 1] = fma(sA[NS - 1], v[NS - 1], tiny);
                            const double qs = tree_sum<NS>(q);
                            double n0 = 0.0, n1 = 0.0, n2 = 0.0, n3 = 0.0;
#pragma unroll
                            for (int i = 0; i < NS; i += 4) {
                                n0 = fma(al[i], q[i], n0);
                                n1 = fma(al[i + 1], q[i + 1], n1);
                                n2 = fma(al[i + 2], q[i + 2], n2);
                                n3 = fma(al[i + 3], q[i + 3], n3);
                            }
                            const double norm = (n0 + n1) + (n2 + n3);
                            // 1 / norm from the reference by exponent arithmetic; the same identity (sum_i alpha_t(i)
                            // beta_t(i) = P(O) at every t) is the backward pass's precision check
                            const double r = recip_from_ref(norm, rref);
                            if ((norm >= LEAN_MIN) & (qs >= LEAN_MIN) & norm_consistent(norm, r)) {
                                const double sc = pow2_rescale_noacc(qs);
#pragma unroll
                                for (int p = 0; p < L::CPR; ++p)  // gamma_t, staged (not yet issued)
                                    sg[p] = make_double2(fma(al[2 * p] * r, q[2 * p], tiny), fma(al[2 * p + 1] * r, q[2 * p + 1], tiny));
#pragma unroll
                                for (int p = 0; p < L::CPR; ++p) {  // q becomes v_j = b_j(o_t) beta-hat_t(j) in place
                                    const double2 x = sB[L::swz(sym, p)];
                                    q[2 * p] = fma(x.x, q[2 * p] * sc, tiny);
                                    q[2 * p + 1] = fma(x.y, q[2 * p + 1] * sc, tiny);
                                }
                                if (max_hiN<NS>(q) >= LEAN_MIN_HI) {
#pragma unroll
                                    for (int i = 0; i < NS; ++i) {
                                        const double ui = al[i] * r;
                                        Xs[i] = fma(ui, v[i], Xs[i]);
                                        if (i + 1 < NS) Xn[i] = fma(ui, v[i + 1], Xn[i]);
                                    }
#pragma unroll
                                    for (int i = 0; i < NS; ++i) v[i] = q[i];
                                    seenS = L::FULL;
                                    seenN = L::FULL >> 1;
                                    done = true;
                                }
                            }
                        }
                    }
                    if (!done) {
                        // the careful step works on a copy so that v / Xs / Xn never have their address taken
                        BwdLState<NS> tmp;
                        double g[NS], alc[NS];
#pragma unroll
                        for (int i = 0; i < NS; ++i) { tmp.v[i] = v[i]; tmp.Xs[i] = Xs[i]; tmp.Xn[i] = Xn[i]; alc[i] = al[i]; }
                        tmp.seenS = seenS; tmp.seenN = seenN; tmp.imprecise = imprecise; tmp.vpos = vpos;
                        bwdL_step_slow<NS>(tmp, sA, sB, sym, t == T - 1, alc, g);
                        if (t == T - 1) rref = 1.0 / tree_sum<NS>(al);
#pragma unroll
                        for (int i = 0; i < NS; ++i) { v[i] = tmp.v[i]; Xs[i] = tmp.Xs[i]; Xn[i] = tmp.Xn[i]; }
                        seenS = tmp.seenS; seenN = tmp.seenN; imprecise = tmp.imprecise; vpos = tmp.vpos;
                        double2 *sg = reinterpret_cast<double2 *>(stage);
#pragma unroll
                        for (int p = 0; p < L::CPR; ++p) sg[p] = make_double2(g[2 * p], g[2 * p + 1]);
                    }
                }
                {  // alpha-hat of step t - 1 (at t = 0: row 0 once more, unused)
                    const int tp = t > 0 ? t - 1 : 0;
#pragma unroll
                    for (int q = 0; q < L::CPR; ++q) {
                        const double2 x = __ldcs(sp + ((size_t)tp * L::CPR + q) * 32);
                        al[2 * q] = x.x;
                        al[2 * q + 1] = x.y;
                    }
                }
                // emission-count numerators (:460-500) and, at t = 0, the pi sums (:415-426): the staged
                // gamma rows are re-read with lanes = states (NS lanes per row, 32 / NS rows per
                // instruction) and added to the word's accumulator rows with coalesced fp64 REDs
                if (act) *reinterpret_cast<unsigned *>(stage + NS * 8) = sym;  // the row's codeword, in the row padding
                __syncwarp();
                {
                    // lane (fo, jj) of iteration k handles state jj of staged row k * FPI + fo; everything but
                    // the codeword is a compile-time offset from per-lane bases set up before the time loop
                    const unsigned actmask = __ballot_sync(0xffffffffu, act);
                    constexpr int FPI = 32 / NS;  // frames (rows) per warp instruction
                    if (actmask == 0xffffffffu) {
#pragma unroll
                        for (int k = 0; k < NS; ++k) {
                            const unsigned char *row = flush_src + (size_t)k * FPI * L::ROWB;
                            const unsigned sf = *reinterpret_cast<const unsigned *>(row + flush_sym_off);
                            atomicAdd(flush_dst + (size_t)sf * NS, *reinterpret_cast<const double *>(row));
                        }
                    } else {
                        // rows of lanes that are not active (yet) hold zeros and codeword 0 (written at the top of the
                        // block): an instruction is skipped when none of its rows is active — a warp-uniform test —
                        // and adds + 0.0 for the others.  (Per-lane tests here made the last, partly filled block of a
                        // word a quarter slower than a full one, and the CTA's other warps waited for it.)
#pragma unroll
                        for (int k = 0; k < NS; ++k) {
                            if ((actmask >> (k * FPI)) & ((1u << FPI) - 1u)) {
                                const unsigned char *row = flush_src + (size_t)k * FPI * L::ROWB;
                                const unsigned sf = *reinterpret_cast<const unsigned *>(row + flush_sym_off);
                                atomicAdd(flush_dst + (size_t)sf * NS, *reinterpret_cast<const double *>(row));
                            }
                        }
                    }
                    if (t == 0) {  // warp-uniform
#pragma unroll 2
                        for (int k = 0; k < NS; ++k) {
                            if ((actmask >> (k * FPI + flush_fo)) & 1u)
                                atomicAdd(accw + flush_jj, *reinterpret_cast<const double *>(flush_src + (size_t)k * FPI * L::ROWB));
                        }
                    }
                }
                __syncwarp();
            }
        }
        if (imprecise) {  // sticky hand-over; the host redoes this E-step once (hmmb_bw_iterate)
            raise_flag(flag, bk.first + lane);
            atomicAdd(new_flags, 1);
        }
    }

    // ---- CTA flush of the xi sums: warp shuffle tree, then one fp64 RED per entry
    double *red = sRed + (size_t)warp * 2 * NS;
#pragma unroll
    for (int i = 0; i < NS; ++i) {
        double x = Xs[i], y = Xn[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            x += __shfl_xor_sync(0xffffffffu, x, o);
            y += __shfl_xor_sync(0xffffffffu, y, o);
        }
        if (lane == 0) { red[i] = x; red[NS + i] = y; }
    }
    const unsigned sS = __reduce_or_sync(0xffffffffu, seenS), sN = __reduce_or_sync(0xffffffffu, seenN);
    if (lane == 0) { atomicOr(&sSeen[0], sS); atomicOr(&sSeen[1], sN); }
    __syncthreads();
    if (tid < 2 * NS) {
        double x = 0.0;
#pragma unroll
        for (int wq = 0; wq < LTR_WARPS; ++wq) x += sRed[wq * 2 * NS + tid];
        const int i = tid < NS ? tid : tid - NS, j = tid < NS ? i : i + 1;
        if (j < NS) {
            const double aij = sA[tid];
            double val = aij > 0.0 ? aij * x : 0.0;  // impossible transitions: ignore whatever piled up
            if (val == 0.0 && aij > 0.0 && ((sSeen[tid < NS ? 0 : 1] >> i) & 1u)) val = tiny_pos();
            if (val > 0.0) atomicAdd(accw + NS + (size_t)i * NS + j, val);
        }
    }
}

}  // namespace hmmb

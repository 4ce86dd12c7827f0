// Device-side building blocks of the scaled forward / backward recursions.
//
// Maths (SURVEY.md App. A): the reference works in log space and treats -inf as a
// structural zero that is dropped from every log-sum-exp (HMM/hmm_training.py:122-199).
// The fast kernels run the recursions in the linear domain with an exact power-of-two
// rescale per step and the invariant
//        value > 0   <=>   the reference's log value is finite,
// kept by clamping positive-but-underflowed products to the smallest denormal in rarely
// taken slow paths.  gamma_t and xi_t are normalised per step by
// norm_t = sum_i alpha_t(i) beta_t(i), so the scale factors never need to be stored; only
// sum_t log2(scale) (the sequence log-likelihood) leaves the forward pass.
//
// Precision guard.  One common scale per time step cannot represent states whose probability
// is more than ~1e-308 below the step's largest one; log space can.  That only matters when
// such a state later carries the sequence (the dominant states die on a zero / denormal
// emission) — typical for an utterance scored against a foreign word's model.  The forward
// pass therefore propagates a rigorous bound on the absolute error introduced by every
// denormal / clamped value (the same linear recursion, in units of 2^-1000) and, when the
// bound exceeds 1e-12 of the step's mass, marks the sequence (NaN log-likelihood).  Marked
// sequences are recomputed by the exact log-space routines at the end of this file, which
// restate the reference's algorithm literally.
#pragma once

#include <climits>

#include "common.cuh"

namespace hmmb {

// 32-sequence block of the N = 4 path: one sequence per lane, all of the same word.
struct Blk {
    int32_t word;
    int32_t nseq;        // <= 32 live lanes
    int32_t tmax;        // longest sequence in the block
    int32_t first;       // index of lane 0's sequence in the sorted order
    int64_t obs_base;    // uint4 index of the block's first 16-byte symbol chunk row
    int64_t spill_base;  // first time step of the block in the alpha spill (x 64 double2)
};

// CTA work item: blocks [blk_begin, blk_end) all belong to `word`.
struct CtaWork {
    int32_t word;
    int32_t blk_begin;
    int32_t blk_end;
    int32_t seq_begin;  // unused by the kernels; kept for debugging
};

constexpr double LN2 = 0.693147180559945309417232121458;

// A per-step total below 2^-960 means the step's factors are so small that plain products
// lose bits or underflow; the kernels then use exponent-split products (frexp / ldexp).
constexpr double TINY_STEP = 0x1p-960;
// error bounds are carried multiplied by 2^1000 so that they do not underflow themselves
constexpr double ERR_UNIT = 0x1p-74;              // smallest denormal (2^-1074) * 2^1000
constexpr double ERR_LIMIT = 1e-12 * 0x1p1000;    // relative bound 1e-12 in the same units
constexpr double SUBNORMAL_LIMIT = 0x1p-1021;

// Per-sequence hand-over flags (sticky, uint8 [R]) carry a 16-byte header in front of the array whose first int is
// "some flag is set": the exact kernel, launched every iteration, returns at once while it is zero instead of
// scanning R flags.
constexpr int FLAG_HDR = 16;
__device__ __forceinline__ void raise_flag(uint8_t *flag, int64_t i) {
    flag[i] = 1;
    *reinterpret_cast<volatile int *>(flag - FLAG_HDR) = 1;
}
__device__ __forceinline__ bool any_flag_raised(const uint8_t *flag) {
    return *reinterpret_cast<const volatile int *>(flag - FLAG_HDR) != 0;
}

__device__ __forceinline__ double nan_mark() { return __longlong_as_double(0x7ff8000000000000LL); }
// zero or denormal (non-negative input): exponent field is 0
__device__ __forceinline__ bool is_sub(double x) { return (unsigned)__double2hiint(x) < 0x00100000u; }

// x*y for positive doubles as mantissa in [0.25, 1) and a separate exponent: cannot underflow
__device__ __forceinline__ void frexp_prod(double x, double y, double &m, int &e) {
    int ex, ey;
    const double mx = frexp(x, &ex), my = frexp(y, &ey);
    m = mx * my;
    e = ex + ey;
}

// Exponent-split products for the N = 4 kernels: out_j = n_j*b_j * 2^-E with E the largest
// product exponent, so the largest out_j is in [0.25, 1).  Returns 0 if no product is
// positive, 2 if a product within 2^-64 of the largest comes from a sub-normal n_j (its bits
// are already lost), else 1.  Positive products that still underflow are held at the
// smallest denormal.
__device__ __noinline__ int exact_products4(double n0, double n1, double n2, double n3, double b0, double b1,
                                            double b2, double b3, double *out, int *E_out) {
    const double nn[4] = {n0, n1, n2, n3}, bb[4] = {b0, b1, b2, b3};
    double m[4];
    int e[4];
    int E = INT_MIN;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        m[j] = 0.0;
        e[j] = INT_MIN;
        if (nn[j] > 0.0 && bb[j] > 0.0) {
            frexp_prod(nn[j], bb[j], m[j], e[j]);
            E = max(E, e[j]);
        }
    }
    out[0] = out[1] = out[2] = out[3] = 0.0;
    *E_out = 0;
    if (E == INT_MIN) return 0;
    int code = 1;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
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

// ---------------------------------------------------------------- symbol shift registers
// A lane keeps 16 bytes of codewords (16 x u8 or 8 x u16) in a uint4 and pops one symbol
// per time step from the front (forward pass) or the back (backward pass).
template <typename SymT> struct Sym;
template <> struct Sym<uint8_t> {
    static constexpr int SPC = 16;
    static __device__ __forceinline__ unsigned pop_front(uint4 &w) {
        unsigned s = w.x & 0xffu;
        w.x = __funnelshift_r(w.x, w.y, 8);
        w.y = __funnelshift_r(w.y, w.z, 8);
        w.z = __funnelshift_r(w.z, w.w, 8);
        w.w >>= 8;
        return s;
    }
    static __device__ __forceinline__ unsigned pop_back(uint4 &w) {
        unsigned s = w.w >> 24;
        w.w = __funnelshift_l(w.z, w.w, 8);
        w.z = __funnelshift_l(w.y, w.z, 8);
        w.y = __funnelshift_l(w.x, w.y, 8);
        w.x <<= 8;
        return s;
    }
};
template <> struct Sym<uint16_t> {
    static constexpr int SPC = 8;
    static __device__ __forceinline__ unsigned pop_front(uint4 &w) {
        unsigned s = w.x & 0xffffu;
        w.x = __funnelshift_r(w.x, w.y, 16);
        w.y = __funnelshift_r(w.y, w.z, 16);
        w.z = __funnelshift_r(w.z, w.w, 16);
        w.w >>= 16;
        return s;
    }
    static __device__ __forceinline__ unsigned pop_back(uint4 &w) {
        unsigned s = w.w >> 16;
        w.w = __funnelshift_l(w.z, w.w, 16);
        w.z = __funnelshift_l(w.y, w.z, 16);
        w.y = __funnelshift_l(w.x, w.y, 16);
        w.x <<= 16;
        return s;
    }
};

// ---------------------------------------------------------------- generic-N helpers
template <int NP>
__device__ __forceinline__ double group_sum(double v) {
#pragma unroll
    for (int o = NP / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
template <int NP>
__device__ __forceinline__ double group_sum_masked(unsigned gm, double v) {
#pragma unroll
    for (int o = NP / 2; o > 0; o >>= 1) v += __shfl_xor_sync(gm, v, o);
    return v;
}

__device__ __forceinline__ int warp_max_int(int v) { return __reduce_max_sync(0xffffffffu, v); }

// Generic forward pass for one sequence handled by NP lanes (lane j = state j).
// stage: per-warp double-buffered [2][32] shared scratch (+[2][32] for the error bounds).
// All 32 lanes of the warp call this together (groups whose sequence is shorter idle on
// `t < T`), Tw = warp-wide max T.  Same return convention as fwd4_run.
template <int NP, typename SymT, bool SPILL>
__device__ __forceinline__ double fwdG_run(int T, int Tw, int N, int j, int gbase, int lane,
                                           const SymT *__restrict__ obs, const double *__restrict__ Btw,
                                           const double (&acol)[NP], double pj, double *__restrict__ spill,
                                           double *stage) {
    const unsigned gm = ((NP == 32) ? 0xffffffffu : ((1u << NP) - 1u)) << gbase;
    double *estage = stage + 64;
    double al = 0.0, er = 0.0;
    long long esum = 0;
    bool stop = false, tainted = false;
    double ll = neg_inf();
    int par = 0;
    // software pipeline of the two dependent loads: codeword two steps ahead, B one step ahead
    unsigned sym_n = (T > 1) ? (unsigned)obs[1] : 0u;                                 // o_{t+1}
    double b_n = (T > 0 && j < N) ? __ldg(Btw + (size_t)obs[0] * N + j) : 0.0;          // b_j(o_t)
    for (int t = 0; t < Tw; ++t) {
        const bool act = t < T && !stop;
        double at = 0.0, b = 0.0, n = 0.0;
        if (t < T) {
            b = b_n;
            if (t + 1 < T) {
                b_n = (j < N) ? __ldg(Btw + (size_t)sym_n * N + j) : 0.0;
                if (t + 2 < T) sym_n = obs[t + 2];
            }
        }
        if (act) {
            if (t == 0) {
                n = pj;
            } else {
                const double *prev = stage + par * 32 + gbase;
                const double2 *prev2 = reinterpret_cast<const double2 *>(prev);  // (gbase is a multiple of NP >= 4; stage is 16-byte aligned)
                double n0 = 0.0, n1 = 0.0, n2 = 0.0, n3 = 0.0;  // four chains: shorter dependency
#pragma unroll
                for (int i = 0; i < NP; i += 4) {
                    const double2 x = prev2[i / 2], y = prev2[i / 2 + 1];
                    n0 = fma(x.x, acol[i], n0);
                    n1 = fma(x.y, acol[i + 1], n1);
                    n2 = fma(y.x, acol[i + 2], n2);
                    n3 = fma(y.y, acol[i + 3], n3);
                }
                n = (n0 + n1) + (n2 + n3);
                if (n == 0.0) {  // keep "n > 0 <=> structurally reachable"
                    bool reach = false;
                    for (int i = 0; i < NP; ++i) reach |= (prev[i] > 0.0 && acol[i] > 0.0);
                    if (reach) n = tiny_pos();
                }
            }
            at = n * b;
        }
        double ssum = group_sum<NP>(at);
        double ea = 0.0;
        if (act) {
            if (!(ssum >= TINY_STEP)) {
                // tiny (or impossible) step: exponent-split products, group-wide max exponent
                double m = 0.0;
                int e = INT_MIN;
                if (n > 0.0 && b > 0.0) frexp_prod(n, b, m, e);
                int E = e;
#pragma unroll
                for (int o = NP / 2; o > 0; o >>= 1) E = max(E, __shfl_xor_sync(gm, E, o));
                const bool lost = (e != INT_MIN) && (e >= E - 64) && (n < SUBNORMAL_LIMIT) && t > 0;
                const bool anylost = (__ballot_sync(gm, lost) != 0u);
                if (E == INT_MIN) {
                    stop = true;
                } else if (anylost || tainted) {
                    stop = true;
                    ll = nan_mark();
                } else {
                    at = 0.0;
                    if (e != INT_MIN) {
                        at = ldexp(m, max(e - E, -1200));
                        if (at == 0.0) at = tiny_pos();
                    }
                    esum += E;
                    ssum = group_sum_masked<NP>(gm, at);
                }
            } else {
                double seed = 0.0;
                if (n > 0.0 && b > 0.0 && is_sub(at)) {
                    if (at == 0.0) at = tiny_pos();
                    seed = ERR_UNIT;
                }
                const bool anyseed = (__ballot_sync(gm, seed > 0.0) != 0u);
                if (tainted || anyseed) {
                    if (t > 0) {
                        const double *eprev = estage + par * 32 + gbase;
                        double en = 0.0;
#pragma unroll
                        for (int i = 0; i < NP; ++i) en = fma(eprev[i], acol[i], en);
                        ea = en * b;
                    }
                    ea += seed;
                    tainted = true;
                }
            }
            if (!stop) {
                const double sc = pow2_rescale(ssum, esum);
                al = at * sc;
                if (tainted) {
                    er = ea * sc;
                    const double etot = group_sum_masked<NP>(gm, er);
                    if (!(etot <= ERR_LIMIT)) {
                        stop = true;
                        ll = nan_mark();
                    }
                }
                if (t == T - 1 && !stop) ll = log(ssum * sc) + (double)esum * LN2;
            }
            if (stop) al = 0.0;
            if (SPILL && j < N) spill[(size_t)t * N + j] = al;
        }
        par ^= 1;
        stage[par * 32 + lane] = al;
        estage[par * 32 + lane] = er;
        __syncwarp();
    }
    return ll;
}

// ================================================================ exact log-space routines
// Literal restatement of the reference's log-space recursions for the (rare) sequences the
// precision guard hands over.  One warp per sequence, lane = state (N <= 32).
__device__ __forceinline__ double safe_log_d(double x) { return x > 0.0 ? log(x) : neg_inf(); }

__device__ __forceinline__ double warp_lse(double x, bool valid) {
    // log_sum_exp over the lanes with valid && x finite (HMM/hmm_training.py:66-79)
    double v = (valid && x > neg_inf()) ? x : neg_inf();
    double m = v;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (!(m > neg_inf())) return neg_inf();
    double s = (v > neg_inf()) ? exp(v - m) : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    return m + log(s);
}

// codeword accessors: linear stream (generic path) or the blocked layout of the N = 4 path
template <typename SymT>
struct LinObs {
    const SymT *p;
    __device__ __forceinline__ unsigned operator[](int t) const { return p[t]; }
};
template <typename SymT>
struct BlkObs {
    const uint4 *p;  // chunk row of this sequence's lane: obs_blk + blk.obs_base + lane
    unsigned mask = 0x7ffu;  // the 11 codeword bits of a packed entry (bw4_kernels.cuh)
    __device__ __forceinline__ unsigned operator[](int t) const {
        // blocked layout: 8 packed u16 per uint4, codeword in the low bits (bw4_kernels.cuh)
        const unsigned short *c = reinterpret_cast<const unsigned short *>(p + (size_t)(t / 8) * 32);
        return (unsigned)c[t % 8] & mask;
    }
};

// log alpha recursion (:122-160, :357-360).  scratch (nullable) receives log alpha [t][N].
// Returns log P(O|lambda) (:376-377).  lane = state j; all 32 lanes participate.
template <typename ObsT>
__device__ __noinline__ double exact_forward(int T, int N, int lane, const ObsT obs,
                                             const double *__restrict__ piw, const double *__restrict__ Aw,
                                             const double *__restrict__ Btw, double *__restrict__ scratch) {
    const int j = lane;
    const bool st = j < N;
    double la = neg_inf();
    for (int t = 0; t < T; ++t) {
        const unsigned sym = obs[t];
        const double lb = st ? safe_log_d(__ldg(Btw + (size_t)sym * N + j)) : neg_inf();
        double cur;
        if (t == 0) {
            cur = st ? safe_log_d(__ldg(piw + j)) + lb : neg_inf();
        } else {
            // LSE_i [ la_i + log a_ij ] over finite terms, two passes (max, then sum of exp)
            double m = neg_inf();
            for (int i = 0; i < N; ++i) {
                const double lai = __shfl_sync(0xffffffffu, la, i);
                const double x = st ? lai + safe_log_d(__ldg(Aw + (size_t)i * N + j)) : neg_inf();
                m = fmax(m, x);
            }
            double s = 0.0;
            for (int i = 0; i < N; ++i) {
                const double lai = __shfl_sync(0xffffffffu, la, i);
                const double x = st ? lai + safe_log_d(__ldg(Aw + (size_t)i * N + j)) : neg_inf();
                if (x > neg_inf()) s += exp(x - m);
            }
            cur = (m > neg_inf() && lb > neg_inf()) ? m + log(s) + lb : neg_inf();
        }
        la = cur;
        if (scratch && st) scratch[(size_t)t * N + j] = la;
    }
    return warp_lse(la, st);
}

// Exact E-step contribution of one sequence (:363-410 and the sums of :415-500): log beta
// recursion, gamma / xi in log space, exp'ed into the fp64 accumulators with atomics.
// acc layout: [pi N][xi N*N][cnt M*N].  Requires log alpha in scratch and finite logP.
template <typename ObsT>
__device__ __noinline__ void exact_backward_accumulate(int T, int N, int lane, const ObsT obs,
                                                       const double *__restrict__ Aw, const double *__restrict__ Btw,
                                                       const double *__restrict__ scratch, double logP,
                                                       double *__restrict__ acc) {
    const int i = lane;
    const bool st = i < N;
    double lbeta = st ? 0.0 : neg_inf();  // log beta_{T-1} = 0
    for (int t = T - 1; t >= 0; --t) {
        const unsigned sym = obs[t];
        const double la = st ? scratch[(size_t)t * N + i] : neg_inf();
        if (t < T - 1) {
            // term_j = log b_j(o_{t+1}) + log beta_{t+1}(j), held by lane j
            const unsigned sym1 = obs[t + 1];
            const double lbj = st ? safe_log_d(__ldg(Btw + (size_t)sym1 * N + i)) : neg_inf();
            const double term = (lbj > neg_inf() && lbeta > neg_inf()) ? lbj + lbeta : neg_inf();
            double m = neg_inf();
            for (int j = 0; j < N; ++j) {
                const double tj = __shfl_sync(0xffffffffu, term, j);
                const double laij = st ? safe_log_d(__ldg(Aw + (size_t)i * N + j)) : neg_inf();
                const double x = (tj > neg_inf() && laij > neg_inf()) ? laij + tj : neg_inf();
                m = fmax(m, x);
                // xi_t(i,j) = alpha_t(i) a_ij b_j(o_{t+1}) beta_{t+1}(j) / P   (:397-410)
                if (x > neg_inf() && la > neg_inf()) {
                    double xi = exp(la + x - logP);
                    if (xi == 0.0) xi = tiny_pos();
                    atomicAdd(acc + N + (size_t)i * N + j, xi);
                }
            }
            double s = 0.0;
            for (int j = 0; j < N; ++j) {
                const double tj = __shfl_sync(0xffffffffu, term, j);
                const double laij = st ? safe_log_d(__ldg(Aw + (size_t)i * N + j)) : neg_inf();
                const double x = (tj > neg_inf() && laij > neg_inf()) ? laij + tj : neg_inf();
                if (x > neg_inf()) s += exp(x - m);
            }
            lbeta = (m > neg_inf()) ? m + log(s) : neg_inf();
            if (!st) lbeta = neg_inf();
        }
        // gamma_t(i) (:389-394)
        if (st && la > neg_inf() && lbeta > neg_inf()) {
            double g = exp(la + lbeta - logP);
            if (g == 0.0) g = tiny_pos();
            atomicAdd(acc + N + (size_t)N * N + (size_t)sym * N + i, g);
            if (t == 0) atomicAdd(acc + i, g);
        }
    }
}

// ================================================================ thin-state rescue (log-space accumulators)
// The linear-domain accumulators hold POSTERIORS (gamma, xi in [0, 1]); a state whose whole posterior mass over the
// training set — over the steps that count for a row: t < T - 1 for A (HMM/hmm_training.py:429-457) — is below
// ~1e-308 has no representable sums, while the reference, which keeps log sums, still forms the RATIOS that become
// its A / B row (found by the property tests: a 16-state model on a 15-frame sequence, whose state 13 is only
// entered before the last step with posterior 1e-340, keeps a_13,13 = 0.394 in the reference).  Rows whose linear
// denominator falls below THIN_LIMIT are therefore re-accumulated in LOG space: the M-step flags the state (sticky),
// and from then on k_bw_rescue runs the reference's log-space recursions over the word's sequences and keeps, per
// flagged state i, log sum_t xi_t(i, j) and log sum_{t: o_t = k} gamma_t(i) in a slot of its own rank behind the
// accumulators (slots of other ranks stay 0, so the sum-all-reduce gathers them); the M-step combines the ranks'
// slots with log_sum_exp and overrides row i of A and B from them.
constexpr double THIN_LIMIT = 0x1p-200;

// *addr = log(exp(*addr) + exp(x)) atomically (x finite; *addr may be -inf)
__device__ __forceinline__ void atomic_lse(double *addr, double x) {
    unsigned long long *a = reinterpret_cast<unsigned long long *>(addr);
    unsigned long long old = *a, assumed;
    do {
        assumed = old;
        const double cur = __longlong_as_double((long long)assumed);
        double nv;
        if (!(cur > neg_inf())) nv = x;
        else nv = fmax(cur, x) + log1p(exp(-fabs(cur - x)));
        old = atomicCAS(a, assumed, (unsigned long long)__double_as_longlong(nv));
    } while (old != assumed);
}

// Backward pass in log space for ONE sequence (one warp, lane = state; scratch holds log alpha from exact_forward),
// adding only the rows of the states in `mask` to their slots: slot_of[i] >= 0 indexes [N log-xi | M log-gamma]
// rows of `rstride` doubles at `slots` (this rank's region).
template <typename ObsT>
__device__ __noinline__ void exact_backward_rescue(int T, int N, int M, int lane, const ObsT obs,
                                                   const double *__restrict__ Aw, const double *__restrict__ Btw,
                                                   const double *__restrict__ scratch, double logP, unsigned mask,
                                                   const int32_t *__restrict__ slot_of, double *__restrict__ slots,
                                                   int64_t rstride) {
    const int i = lane;
    const bool st = i < N;
    const bool mine = st && ((mask >> i) & 1u) && slot_of[i] >= 0;
    double *row = mine ? slots + (size_t)slot_of[i] * rstride : nullptr;
    double lbeta = st ? 0.0 : neg_inf();  // log beta_{T-1} = 0
    for (int t = T - 1; t >= 0; --t) {
        const unsigned sym = obs[t];
        const double la = st ? scratch[(size_t)t * N + i] : neg_inf();
        if (t < T - 1) {
            const unsigned sym1 = obs[t + 1];
            const double lbj = st ? safe_log_d(__ldg(Btw + (size_t)sym1 * N + i)) : neg_inf();
            const double term = (lbj > neg_inf() && lbeta > neg_inf()) ? lbj + lbeta : neg_inf();
            double m = neg_inf();
            for (int j = 0; j < N; ++j) {
                const double tj = __shfl_sync(0xffffffffu, term, j);
                const double laij = st ? safe_log_d(__ldg(Aw + (size_t)i * N + j)) : neg_inf();
                const double x = (tj > neg_inf() && laij > neg_inf()) ? laij + tj : neg_inf();
                m = fmax(m, x);
                // log xi_t(i,j) = log alpha_t(i) + log a_ij + log b_j(o_{t+1}) + log beta_{t+1}(j) - log P   (:397-410)
                if (mine && x > neg_inf() && la > neg_inf()) atomic_lse(row + j, la + x - logP);
            }
            double s = 0.0;
            for (int j = 0; j < N; ++j) {
                const double tj = __shfl_sync(0xffffffffu, term, j);
                const double laij = st ? safe_log_d(__ldg(Aw + (size_t)i * N + j)) : neg_inf();
                const double x = (tj > neg_inf() && laij > neg_inf()) ? laij + tj : neg_inf();
                if (x > neg_inf()) s += exp(x - m);
            }
            lbeta = (m > neg_inf()) ? m + log(s) : neg_inf();
            if (!st) lbeta = neg_inf();
        }
        // log gamma_t(i) (:389-394), by codeword
        if (mine && la > neg_inf() && lbeta > neg_inf()) atomic_lse(row + N + sym, la + lbeta - logP);
    }
    (void)M;
}

}  // namespace hmmb

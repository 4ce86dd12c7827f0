// N = 4 Baum-Welch E-step kernels (the reference's hard-coded state count,
// HMM/hmm_training.py:226): one sequence per thread, 32 same-word sequences per warp in
// lock-step.
//
//   k_repack_blocks4  ragged codewords -> blocked u16 layout [block][chunk of 8 steps][lane];
//                     each entry = codeword (11 bits) | conflict rank (5 bits): the number of
//                     lower lanes of the warp that see the same codeword at the same step.
//                     Codewords never change during training, so the conflict schedule of
//                     the emission-count update is computed once here instead of with
//                     MATCH.ANY every step (measured 1 MATCH per ~55 cycles per SM on B200).
//   k_bw_fwd4         scaled forward pass, alpha-hat spilled to HBM [block][t][half][lane] as
//                     coalesced 16-byte streaming stores (even steps, and odd steps that were not
//                     plain: see fwd4_plain), B^T of the CTA's word in shared memory.
//   k_bw_bwd4         backward pass fused with the gamma / xi / emission-count accumulation
//                     (beta never leaves registers; the plain odd-step alpha-hat rows rebuilt from
//                     the even ones); counts go to warp-private shared-memory
//                     copies with plain read-modify-writes in precomputed rank order (no
//                     atomics, deterministic); one partial per CTA.
//
// BIDIAG = true specialises both kernels for an upper-bidiagonal transition matrix (the
// reference's left-to-right default, :307-312 — zeros of A stay zeros under re-estimation,
// :450-455): 7 instead of 16 products in every mat-vec and 7 instead of 16 xi accumulators.
// Skipped terms are exact zeros, so the results are bit-identical to the dense kernel.
#pragma once

#include <type_traits>

#include "hmm_device.cuh"

namespace hmmb {

constexpr int BW_THREADS = 128;  // 4 warps per CTA in every E-step kernel
constexpr int BW_WARPS = BW_THREADS / 32;
constexpr int SPC4 = 8;          // packed u16 entries per uint4
constexpr unsigned SYM_MASK = 0x7ffu;
constexpr int SYM_BITS = 11;
constexpr int BW4_MAX_M = 512;   // warp-private count copies must fit in shared memory
// CTA work items of the N = 4 path are sized for ONE fat backward CTA per SM (up to BWD4_MAX_WARPS warps sharing one
// copy of the word's B^T); the forward kernel keeps its 4-warp CTAs and splits every work item over FWD4_SPLIT CTAs.
constexpr int BWD4_MAX_WARPS = 16;
constexpr int FWD4_SPLIT = 4;
constexpr int BWD4_REP = 8;  // replicas of B^T in the backward kernel when they fit (M <= 256), see fwd4_run

// ---------------------------------------------------------------- repack
// One warp per (block, chunk of 8 steps), lane = sequence.  The conflict rank of a lane at a step
// (number of lower lanes of the block with the same codeword) comes from SYM_BITS ballots: the
// lanes that agree with me on every bit are my peers.  No shared memory, no barriers; the output
// row of the chunk is one coalesced 512-byte store.
constexpr int REPACK_WARPS = 8;
// Lanes of the warp whose bit `bit` agrees with this lane's: the bit is sign-extended to a mask once (bfe.s32) and feeds both
// the ballot and the combination.  Written as `__ballot_sync((sym >> bit) & 1)` plus `?:` on the same expression, ptxas spent
// six to seven ALU instructions per bit, and the repack ran at 92 % of the ALU pipe.
__device__ __forceinline__ unsigned lanes_with_my_bit(unsigned sym, int bit) {
    int mine;
    asm("bfe.s32 %0, %1, %2, 1;" : "=r"(mine) : "r"(sym), "r"(bit));
    const unsigned set = __ballot_sync(0xffffffffu, mine != 0);
    return ~(set ^ (unsigned)mine);
}
template <typename InT>
__global__ void __launch_bounds__(REPACK_WARPS * 32)
k_repack_blocks4(const InT *__restrict__ obs, const int64_t *__restrict__ off_sorted,
                 const int32_t *__restrict__ len_sorted, const Blk *__restrict__ blks, int blk_base, int nblk,
                 uint4 *__restrict__ obs_blk, int M, int *__restrict__ bad) {
    const int b = blk_base + blockIdx.x;
    if (b >= nblk) return;
    const Blk bk = blks[b];
    const int nch = (bk.tmax + SPC4 - 1) / SPC4;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int T = 0;
    const InT *src = obs;
    if (lane < bk.nseq) {
        T = len_sorted[bk.first + lane];
        src = obs + off_sorted[bk.first + lane];
    }
    const unsigned lt = (1u << lane) - 1u;
    // one-byte codewords whose sequence starts on an 8-byte boundary are fetched a chunk (8 steps) at a time
    const bool wide = sizeof(InT) == 1 && ((reinterpret_cast<uintptr_t>(src) & 7u) == 0u);
    const bool small_m = M <= 256;  // (a codeword >= M is replaced by 0 before it is ranked)
    for (int c = warp; c < nch; c += REPACK_WARPS) {
        unsigned r[4] = {0u, 0u, 0u, 0u};
        unsigned long long chunk8 = 0ull;
        if (sizeof(InT) == 1 && wide && c * SPC4 + SPC4 <= T)
            chunk8 = __ldg(reinterpret_cast<const unsigned long long *>(src + c * SPC4));
#pragma unroll
        for (int s = 0; s < SPC4; ++s) {
            const int t = c * SPC4 + s;
            const bool have = t < T;
            unsigned sym = 0u;
            if (have) {
                unsigned long long v;
                if (sizeof(InT) == 1 && wide && c * SPC4 + SPC4 <= T) v = (chunk8 >> (8 * s)) & 0xffull;
                else v = (unsigned long long)src[t];
                if (v >= (unsigned long long)M) { atomicOr(bad, 1); v = 0; }
                sym = (unsigned)v;
            }
            // the lanes that hold the same codeword at this step: one ballot per codeword bit (eight for alphabets up to
            // 256, eleven otherwise; a single MATCH.ANY instead measured a third slower: 1.48 vs 1.08 ms for config 3's
            // 200 M frames); lanes without a frame are nobody's peer
            unsigned peers = __ballot_sync(0xffffffffu, have);
            if (small_m) {
#pragma unroll
                for (int bit = 0; bit < 8; ++bit) peers &= lanes_with_my_bit(sym, bit);
            } else {
#pragma unroll
                for (int bit = 0; bit < SYM_BITS; ++bit) peers &= lanes_with_my_bit(sym, bit);
            }
            const unsigned rank = __popc(peers & lt);
            const unsigned packed = have ? (sym | (rank << SYM_BITS)) : 0u;
            r[s >> 1] |= packed << ((s & 1) * 16);
        }
        obs_blk[bk.obs_base + (size_t)c * 32 + lane] = make_uint4(r[0], r[1], r[2], r[3]);
    }
}

// ---------------------------------------------------------------- forward
// zero-or-denormal test for four non-negative doubles at once (integer pipe)
__device__ __forceinline__ bool any_sub4(double x0, double x1, double x2, double x3) {
    const unsigned m = min(min((unsigned)__double2hiint(x0), (unsigned)__double2hiint(x1)),
                           min((unsigned)__double2hiint(x2), (unsigned)__double2hiint(x3)));
    return m < 0x00100000u;
}

// a[] holds A row-major (dense) or {a00,a11,a22,a33,a01,a12,a23} (BIDIAG).
template <bool BIDIAG>
__device__ __forceinline__ void matvec_fwd(const double *a, double al0, double al1, double al2, double al3, double &n0,
                                           double &n1, double &n2, double &n3) {
    if (BIDIAG) {
        n0 = al0 * a[0];
        n1 = al0 * a[4] + al1 * a[1];
        n2 = al1 * a[5] + al2 * a[2];
        n3 = al2 * a[6] + al3 * a[3];
    } else {
        n0 = al0 * a[0] + al1 * a[4] + al2 * a[8] + al3 * a[12];
        n1 = al0 * a[1] + al1 * a[5] + al2 * a[9] + al3 * a[13];
        n2 = al0 * a[2] + al1 * a[6] + al2 * a[10] + al3 * a[14];
        n3 = al0 * a[3] + al1 * a[7] + al2 * a[11] + al3 * a[15];
    }
}
// A[i][j] from either representation (slow paths only)
template <bool BIDIAG>
__device__ __forceinline__ double a_at(const double *a, int i, int j) {
    if (BIDIAG) return (j == i) ? a[i] : ((j == i + 1) ? a[4 + i] : 0.0);
    return a[i * 4 + j];
}

// Structural masks of a 4-state model (which log values are finite), kept as 4-bit sets:
//   rowmask[i]   = { j : a_ij > 0 }
//   lutF(m)      = union of rowmask[i] over i in m          (states reachable from the set m)
//   lutB(m)      = { i : rowmask[i] meets m }               (states that can continue into m)
// packed as sixteen 4-bit entries in a 64-bit word.
struct Masks4 {
    unsigned long long lutF, lutB;
    unsigned pmask;
};
__device__ __forceinline__ unsigned lut4(unsigned long long lut, unsigned m) {
    return (unsigned)(lut >> (m * 4u)) & 0xFu;
}
__device__ __forceinline__ Masks4 make_masks4(const double *__restrict__ Aw, const double *__restrict__ piw) {
    unsigned row[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        row[i] = 0u;
#pragma unroll
        for (int j = 0; j < 4; ++j) row[i] |= (__ldg(Aw + i * 4 + j) > 0.0) ? (1u << j) : 0u;
    }
    Masks4 mk;
    mk.lutF = mk.lutB = 0ull;
    for (unsigned m = 0; m < 16; ++m) {
        unsigned f = 0u, b = 0u;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if ((m >> i) & 1u) f |= row[i];
            if (row[i] & m) b |= 1u << i;
        }
        mk.lutF |= (unsigned long long)f << (m * 4u);
        mk.lutB |= (unsigned long long)b << (m * 4u);
    }
    mk.pmask = 0u;
    if (piw) {
#pragma unroll
        for (int j = 0; j < 4; ++j) mk.pmask |= (__ldg(piw + j) > 0.0) ? (1u << j) : 0u;
    }
    return mk;
}
// smallest denormal if bit `j` of `m` is set, else +0.0 (integer pipe)
__device__ __forceinline__ double tiny_if(unsigned m, int j) { return __hiloint2double(0, (int)((m >> j) & 1u)); }

// One PLAIN forward step: every state alive and t > 0, the common case of fwd4_run.  The smallest denormal is the
// addend of every chain, n = A^T al + tiny and at = b(o_t) .* n + tiny.  k_bw_bwd4 rebuilds the odd-step alpha-hat of
// such steps from the even-step row with this same function (fwd4_rebuild), so it is written with explicit fma() only:
// both kernels must get the same bits, not the same value to rounding.
template <bool BIDIAG>
__device__ __forceinline__ void fwd4_plain(const double *a, double al0, double al1, double al2, double al3, double2 b01,
                                           double2 b23, double tiny, double &n0, double &n1, double &n2, double &n3,
                                           double &at0, double &at1, double &at2, double &at3) {
    if (BIDIAG) {
        n0 = fma(al0, a[0], tiny);
        n1 = fma(al1, a[1], fma(al0, a[4], tiny));
        n2 = fma(al2, a[2], fma(al1, a[5], tiny));
        n3 = fma(al3, a[3], fma(al2, a[6], tiny));
    } else {
        n0 = fma(al3, a[12], fma(al2, a[8], fma(al1, a[4], fma(al0, a[0], tiny))));
        n1 = fma(al3, a[13], fma(al2, a[9], fma(al1, a[5], fma(al0, a[1], tiny))));
        n2 = fma(al3, a[14], fma(al2, a[10], fma(al1, a[6], fma(al0, a[2], tiny))));
        n3 = fma(al3, a[15], fma(al2, a[11], fma(al1, a[7], fma(al0, a[3], tiny))));
    }
    at0 = fma(n0, b01.x, tiny); at1 = fma(n1, b01.y, tiny);
    at2 = fma(n2, b23.x, tiny); at3 = fma(n3, b23.y, tiny);
}
// alpha-hat_t of a plain step from alpha-hat_{t-1} (in place): fwd4_plain, then the rescale of fwd4_run, which is
// the step's sum, pow2_rescale of it and at * sc.  Each product is rounded on its own (__dmul_rn), as the value
// fwd4_run spills is, so that no later sum can take it into an FMA.
template <bool BIDIAG>
__device__ __forceinline__ void fwd4_rebuild(const double *a, double2 &x01, double2 &x23, double2 b01, double2 b23,
                                             double tiny) {
    double n0, n1, n2, n3, at0, at1, at2, at3;
    fwd4_plain<BIDIAG>(a, x01.x, x01.y, x23.x, x23.y, b01, b23, tiny, n0, n1, n2, n3, at0, at1, at2, at3);
    const double sc = pow2_rescale_noacc((at0 + at1) + (at2 + at3));
    x01 = make_double2(__dmul_rn(at0, sc), __dmul_rn(at1, sc));
    x23 = make_double2(__dmul_rn(at2, sc), __dmul_rn(at3, sc));
}

// One sequence per lane.  p[j] = pi[j]; B^T of the word in shared memory as two arrays of
// double2, sB01[sym] = (b_0, b_1)(sym) and sB23[sym] = (b_2, b_3)(sym) — 16-byte rows give a
// random gather 8 distinct bank slots instead of 4 with 32-byte rows; sBmax[sym] =
// max_j B[j][sym], sBmask[sym] = {j : B[j][sym] > 0}, rmax = largest row sum of A.  op / sp
// include the lane offset.  Replaces calculate_log_alpha (HMM/hmm_training.py:122-160) and
// the alpha init (:357-360); returns log P(O|lambda) (:376-377), -inf for a structurally
// impossible sequence, or NaN when the precision guard asks for the exact log-space path.
//
// Which alpha_t(j) are finite in the reference is pure structure: m_t = lutF(m_{t-1}) &
// bmask(o_t), a handful of integer operations per step.  The arithmetic keeps
// "alpha-hat_t(j) > 0 <=> j in m_t" without any test by feeding the smallest denormal into the
// FMA chains as the addend of every alive state: a product that underflows stays (barely)
// positive, a normal value is unchanged.
//
// Precision guard: each step adds 2^-1074 per state (worst-case absolute error of a denormal /
// clamped value) to an error bound that is propagated along with the values (units of 2^-1000);
// when its total exceeds 1e-12 of the step's mass the sequence is handed over.
//   VECB (default): per state, e' = (b(o_t) .* (A^T e) + seeds) * scale — the exact linear recursion of the
//     errors.  It stays ~1e-320 of the mass unless the states that carried the sequence die, for any T.
//   !VECB: scalar E' = (E * rmax * max_j b_j(o_t) + seeds) * scale >= sum_j e'_j, 10 instructions cheaper per
//     step but loose: it assumes the error sits in the most probable state, so at every left-to-right
//     transition it grows by ~1 / a_i,i+1 against the true mass; fine for utterance lengths (used by the
//     issue-bound scorer when no utterance exceeds SCORE4_SCALAR_BOUND_MAX_T), trips after a few thousand
//     frames with peaked emissions.
//
// SPILL: alpha-hat_t goes to sp[t * 64] for every even t, and for an odd t only if the step was not plain (see
// fwd4_plain: an alive set still growing or cut by a zero of B, or the exponent-split branch), or if `full` asks for
// every row.  k_bw_bwd4 rebuilds the other odd rows; oddmask[t] (odd t < tmax) records which lanes wrote row t.
//
// REP = 8: B^T is stored eight times, entry (sym, r) at index sym * 8 + r, and a lane reads replica r = lane & 7:
// the eight lanes of a quarter-warp then always hit eight different 16-byte bank slots, so the gather is free of
// bank conflicts whatever the codewords are (used by the scorer, whose only shared-memory traffic it is).
template <bool BIDIAG, bool SPILL, bool VECB = true, int REP = 1>
__device__ __forceinline__ double fwd4_run(int T, int tmax, const uint4 *__restrict__ op,
                                           const double2 *__restrict__ sB01, const double2 *__restrict__ sB23,
                                           const double *__restrict__ sBmax,
                                           const unsigned char *__restrict__ sBmask, const double *a,
                                           const double (&p)[4], double rmax, const Masks4 &mk,
                                           double2 *__restrict__ sp, bool &allfull, int slot = 0,
                                           unsigned symmask = SYM_MASK, unsigned *__restrict__ oddmask = nullptr,
                                           bool full = false) {
    using S16 = Sym<uint16_t>;
    double al0 = 0.0, al1 = 0.0, al2 = 0.0, al3 = 0.0;
    double e0 = 0.0, e1 = 0.0, e2 = 0.0, e3 = 0.0;  // error bounds, units of 2^-1000: per state (VECB) or e0 = their sum
    long long esum = 0;
    unsigned m = 0u;    // alive set
    bool stop = false;  // dead (impossible) or flagged for the exact path
    bool allf = true;   // every step so far had all four states alive and a scale >= 1: every alpha-hat > 0
    double ll = neg_inf();
    const double tiny = tiny_pos();
    const int nch = (tmax + SPC4 - 1) / SPC4;
    uint4 wnext = nch > 0 ? __ldg(op) : make_uint4(0, 0, 0, 0);
    for (int c = 0; c < nch; ++c) {
        uint4 w = wnext;
        if (c + 1 < nch) wnext = __ldg(op + (size_t)(c + 1) * 32);  // prefetch the next 8 codewords
#pragma unroll 2
        for (int s = 0; s < SPC4; ++s) {
            const int t = c * SPC4 + s;
            const unsigned sym = S16::pop_front(w) & symmask;
            bool plain = false, wrote = false;
            if (t < T && !stop) {
                const double2 b01 = sB01[sym * REP + slot], b23 = sB23[sym * REP + slot];
                const unsigned r = (t == 0) ? mk.pmask : lut4(mk.lutF, m);  // reachable before emission
                m = r & (unsigned)sBmask[sym];
                double n0, n1, n2, n3, at0, at1, at2, at3;
                plain = m == 0xFu && t > 0;
                if (plain) {
                    // ---- every state alive (the usual case; the first step takes the masked branch)
                    fwd4_plain<BIDIAG>(a, al0, al1, al2, al3, b01, b23, tiny, n0, n1, n2, n3, at0, at1, at2, at3);
                } else if (m == 0u) {
                    stop = true;  // no state can emit o_t: log P = -inf (:155-160)
                    n0 = n1 = n2 = n3 = at0 = at1 = at2 = at3 = 0.0;
                } else {
                    // ---- first step, or some states structurally dead: masked addends keep them exactly 0
                    allf = allf && (m == 0xFu);
                    const double r0 = tiny_if(r, 0), r1 = tiny_if(r, 1), r2 = tiny_if(r, 2), r3 = tiny_if(r, 3);
                    if (t == 0) {
                        n0 = p[0]; n1 = p[1]; n2 = p[2]; n3 = p[3];
                    } else {
                        n0 = fma(al3, a_at<BIDIAG>(a, 3, 0), fma(al2, a_at<BIDIAG>(a, 2, 0), fma(al1, a_at<BIDIAG>(a, 1, 0), fma(al0, a_at<BIDIAG>(a, 0, 0), r0))));
                        n1 = fma(al3, a_at<BIDIAG>(a, 3, 1), fma(al2, a_at<BIDIAG>(a, 2, 1), fma(al1, a_at<BIDIAG>(a, 1, 1), fma(al0, a_at<BIDIAG>(a, 0, 1), r1))));
                        n2 = fma(al3, a_at<BIDIAG>(a, 3, 2), fma(al2, a_at<BIDIAG>(a, 2, 2), fma(al1, a_at<BIDIAG>(a, 1, 2), fma(al0, a_at<BIDIAG>(a, 0, 2), r2))));
                        n3 = fma(al3, a_at<BIDIAG>(a, 3, 3), fma(al2, a_at<BIDIAG>(a, 2, 3), fma(al1, a_at<BIDIAG>(a, 1, 3), fma(al0, a_at<BIDIAG>(a, 0, 3), r3))));
                    }
                    at0 = fma(n0, b01.x, tiny_if(m, 0)); at1 = fma(n1, b01.y, tiny_if(m, 1));
                    at2 = fma(n2, b23.x, tiny_if(m, 2)); at3 = fma(n3, b23.y, tiny_if(m, 3));
                }
                double ssum = (at0 + at1) + (at2 + at3);
                if (!stop && !(ssum >= TINY_STEP)) {
                    // ---- the whole step is tiny: exponent-split products (rare)
                    double o[4];
                    int Ex;
                    const int code = exact_products4(n0, n1, n2, n3, b01.x, b01.y, b23.x, b23.y, o, &Ex);
                    if (code == 0) {
                        stop = true;
                    } else if ((code == 2 && t > 0) || ((e0 + e1) + (e2 + e3)) > 0.0) {
                        stop = true;  // the surviving states had lost their bits: exact path
                        ll = nan_mark();
                    } else {
                        esum += Ex;
                        at0 = o[0]; at1 = o[1]; at2 = o[2]; at3 = o[3];
                        ssum = (at0 + at1) + (at2 + at3);
                    }
                    allf = false;
                    plain = false;
                }
                if (!stop) {
                    const double sc = pow2_rescale(ssum, esum);
                    allf = allf && (__double2hiint(sc) >= 0x3ff00000);  // scale >= 1 cannot flush a denormal alpha
                    al0 = at0 * sc; al1 = at1 * sc; al2 = at2 * sc; al3 = at3 * sc;
                    if (!VECB) {
                        e0 = fma(e0, rmax * sBmax[sym], 4.0 * ERR_UNIT) * sc;  // scalar bound (see above)
                    } else {
                    // error bounds follow the same linear recursion as the values (t = 0: pi is exact), plus the
                    // worst-case rounding of one denormal / clamped value per state
                    double f0 = 0.0, f1 = 0.0, f2 = 0.0, f3 = 0.0;
                    if (t > 0) {
                        if (BIDIAG) {
                            f0 = e0 * a[0];
                            f1 = fma(e1, a[1], e0 * a[4]);
                            f2 = fma(e2, a[2], e1 * a[5]);
                            f3 = fma(e3, a[3], e2 * a[6]);
                        } else {
                            f0 = fma(e3, a[12], fma(e2, a[8], fma(e1, a[4], e0 * a[0])));
                            f1 = fma(e3, a[13], fma(e2, a[9], fma(e1, a[5], e0 * a[1])));
                            f2 = fma(e3, a[14], fma(e2, a[10], fma(e1, a[6], e0 * a[2])));
                            f3 = fma(e3, a[15], fma(e2, a[11], fma(e1, a[7], e0 * a[3])));
                        }
                    }
                    e0 = fma(f0, b01.x, ERR_UNIT) * sc;
                    e1 = fma(f1, b01.y, ERR_UNIT) * sc;
                    e2 = fma(f2, b23.x, ERR_UNIT) * sc;
                    e3 = fma(f3, b23.y, ERR_UNIT) * sc;
                    }
                    if (!(((e0 + e1) + (e2 + e3)) <= ERR_LIMIT)) {
                        stop = true;
                        ll = nan_mark();
                    }
                    if (t == T - 1 && !stop) ll = log((al0 + al1) + (al2 + al3)) + (double)esum * LN2;
                }
                // a stopped sequence (impossible, or handed to the exact kernel) is skipped by the backward
                // pass, so nothing of it needs to be spilled from here on; the row of a plain odd step is rebuilt
                // there from the even row before it (fwd4_rebuild)
                if (SPILL && !stop && (!(t & 1) || !plain || full)) {
                    __stcs(sp + (size_t)t * 64, make_double2(al0, al1));
                    __stcs(sp + (size_t)t * 64 + 32, make_double2(al2, al3));
                    wrote = true;
                }
            }
            if (SPILL && (t & 1)) {
                // which lanes wrote this odd row: one word per (block, odd step), all zeros on data without zeros
                const unsigned wm = __ballot_sync(0xffffffffu, wrote);
                if ((threadIdx.x & 31) == 0 && t < tmax) oddmask[t] = wm;
            }
        }
    }
    allfull = allf && !stop;
    return ll;
}

// ---------------------------------------------------------------- lean forward pass of the scorer
// calculate_log_likelihood (HMM/hmm_testing.py:49-104) for models whose B has no zero and whose alive set becomes
// all four states within the first three frames (every left-to-right model entered in state 0, and every model
// with positive pi): from frame tstar on, "alpha_t(j) is finite" holds for every j and needs no bookkeeping.
//
// No error bound is carried.  Instead every step checks, on the integer pipe, that all four alpha_t(j) b_j(o_t) are
// NORMAL doubles within 2^900 of each other.  While that holds no value was ever denormal or clamped, every
// operation rounded a normal result (an underflowing addend inside a normal sum changes it by less than half an
// ulp), so the values carry only the ordinary relative error ~t * 2^-52 and the log-likelihood meets the 1e-9
// contract by eight orders.  The first step that fails the check marks the lane; marked lanes are redone by
// fwd4_run with the full structural / precision logic.  The rescale is an exponent subtraction (exact, integer
// pipe): al_j = at_j * 2^-e with e the exponent of the largest of the four.
template <bool BIDIAG, int REP>
__device__ __forceinline__ double score4_lean_run(int T, int tmax, const uint4 *__restrict__ op,
                                                  const double2 *__restrict__ b01row, const double2 *__restrict__ b23row,
                                                  const double *a, const double (&p)[4], const Masks4 &mk, int tstar,
                                                  bool &bad_out) {
    // b01row / b23row = the lane's replica column: entry of codeword sym at [sym * REP]
    using S16 = Sym<uint16_t>;
    double al0 = 0.0, al1 = 0.0, al2 = 0.0, al3 = 0.0;
    int esum = 0;
    bool bad = false;
    unsigned m = 0u;
    // one time step; MASKED (first chunk only): the alive set is still growing, dead states are exact zeros
    auto step = [&](auto masked, int t, unsigned sym) {
        constexpr bool MASKED = decltype(masked)::value;
        const double2 b01 = b01row[sym * REP], b23 = b23row[sym * REP];
        double n0, n1, n2, n3;
        if (MASKED && t == 0) {
            n0 = p[0]; n1 = p[1]; n2 = p[2]; n3 = p[3];
        } else {
            matvec_fwd<BIDIAG>(a, al0, al1, al2, al3, n0, n1, n2, n3);
        }
        const double at0 = n0 * b01.x, at1 = n1 * b01.y, at2 = n2 * b23.x, at3 = n3 * b23.y;
        unsigned h0 = (unsigned)__double2hiint(at0), h1 = (unsigned)__double2hiint(at1);
        unsigned h2 = (unsigned)__double2hiint(at2), h3 = (unsigned)__double2hiint(at3);
        const unsigned hmax = max(max(h0, h1), max(h2, h3));
        const bool growing = MASKED && t < tstar;  // (warp-uniform)
        if (growing) {  // leave the structurally dead states out of the minimum
            m = (t == 0) ? mk.pmask : lut4(mk.lutF, m);
            h0 = (m & 1u) ? h0 : hmax; h1 = (m & 2u) ? h1 : hmax;
            h2 = (m & 4u) ? h2 : hmax; h3 = (m & 8u) ? h3 : hmax;
        }
        const unsigned hmin = min(min(h0, h1), min(h2, h3));
        // all four normal, finite, and within 2^900 of the largest
        bad = bad || (hmin < 0x00100000u) || (hmax >= 0x7fe00000u) || (hmax - hmin > (900u << 20));
        const int eb = (int)(hmax & 0x7ff00000u) - 0x3ff00000;
        esum += eb >> 20;
        // exact scale by 2^-e: subtract from the exponent field
        al0 = __hiloint2double(__double2hiint(at0) - eb, __double2loint(at0));
        al1 = __hiloint2double(__double2hiint(at1) - eb, __double2loint(at1));
        al2 = __hiloint2double(__double2hiint(at2) - eb, __double2loint(at2));
        al3 = __hiloint2double(__double2hiint(at3) - eb, __double2loint(at3));
        if (growing) {  // exact zeros of the dead states stay zeros
            al0 = (m & 1u) ? al0 : 0.0; al1 = (m & 2u) ? al1 : 0.0;
            al2 = (m & 4u) ? al2 : 0.0; al3 = (m & 8u) ? al3 : 0.0;
        }
    };
    const int nch = (tmax + SPC4 - 1) / SPC4;
    uint4 wnext = nch > 0 ? __ldg(op) : make_uint4(0, 0, 0, 0);
    for (int c = 0; c < nch; ++c) {
        uint4 w = wnext;
        if (c + 1 < nch) wnext = __ldg(op + (size_t)(c + 1) * 32);
        if (c == 0) {
#pragma unroll 1
            for (int s = 0; s < SPC4; ++s) {
                const unsigned sym = S16::pop_front(w) & SYM_MASK;
                if (s < T) step(std::true_type{}, s, sym);
            }
        } else {
#pragma unroll 4
            for (int s = 0; s < SPC4; ++s) {
                const unsigned sym = S16::pop_front(w) & SYM_MASK;
                if (c * SPC4 + s < T) step(std::false_type{}, c * SPC4 + s, sym);
            }
        }
    }
    bad_out = bad;
    return log((al0 + al1) + (al2 + al3)) + (double)esum * LN2;
}

// A and pi of word w -> registers, rmax = largest row sum of A, structural masks.
template <bool BIDIAG>
__device__ __forceinline__ void load_Api4(const double *__restrict__ pi, const double *__restrict__ A, int w, double *a,
                                          double (&p)[4], double &rmax, Masks4 &mk) {
    const double *Aw = A + (size_t)w * 16;
    rmax = 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i)
        rmax = fmax(rmax, (__ldg(Aw + i * 4) + __ldg(Aw + i * 4 + 1)) + (__ldg(Aw + i * 4 + 2) + __ldg(Aw + i * 4 + 3)));
    if (BIDIAG) {
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = __ldg(Aw + i * 5);
#pragma unroll
        for (int i = 0; i < 3; ++i) a[4 + i] = __ldg(Aw + i * 5 + 1);
    } else {
#pragma unroll
        for (int q = 0; q < 16; ++q) a[q] = __ldg(Aw + q);
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) p[q] = __ldg(pi + (size_t)w * 4 + q);
    mk = make_masks4(Aw, pi + (size_t)w * 4);
}

// CTA prologue shared by the forward-type kernels: B^T of word w -> shared memory with the
// per-codeword max_j b_j and support mask, A and pi -> registers, rmax = largest row sum of A.
template <bool BIDIAG>
__device__ __forceinline__ void load_model4(const double *__restrict__ pi, const double *__restrict__ A,
                                            const double *__restrict__ Bt, int w, int M, double *sB, double *sBmax,
                                            unsigned char *sBmask, double *a, double (&p)[4], double &rmax,
                                            Masks4 &mk) {
    const int tid = threadIdx.x;
    const double2 *src = reinterpret_cast<const double2 *>(Bt + (size_t)w * M * 4);
    double2 *dst = reinterpret_cast<double2 *>(sB);
    for (int e = tid; e < M; e += BW_THREADS) {
        const double2 x = __ldg(src + 2 * e), y = __ldg(src + 2 * e + 1);
        dst[e] = x;      // sB01
        dst[M + e] = y;  // sB23
        sBmax[e] = fmax(fmax(x.x, x.y), fmax(y.x, y.y));
        sBmask[e] = (unsigned char)((x.x > 0.0 ? 1 : 0) | (x.y > 0.0 ? 2 : 0) | (y.x > 0.0 ? 4 : 0) | (y.y > 0.0 ? 8 : 0));
    }
    load_Api4<BIDIAG>(pi, A, w, a, p, rmax, mk);
}

template <bool BIDIAG>
__device__ __forceinline__ void load_A4(const double *__restrict__ Aw, double *a) {
    if (BIDIAG) {
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = __ldg(Aw + i * 5);
#pragma unroll
        for (int i = 0; i < 3; ++i) a[4 + i] = __ldg(Aw + i * 5 + 1);
    } else {
#pragma unroll
        for (int q = 0; q < 16; ++q) a[q] = __ldg(Aw + q);
    }
}

// 4 CTAs per SM: with 5 (96 registers) the forward pass measured 8 % slower on config 3
constexpr int FWD4_MIN_CTAS = 4;
template <bool BIDIAG>
__global__ void __launch_bounds__(BW_THREADS, FWD4_MIN_CTAS)
k_bw_fwd4(const CtaWork *__restrict__ work, const Blk *__restrict__ blks, const uint4 *__restrict__ obs_blk,
          const int32_t *__restrict__ len_sorted, const double *__restrict__ pi, const double *__restrict__ A,
          const double *__restrict__ Bt, int M, double2 *__restrict__ spill, double *__restrict__ ll_seq,
          const int32_t *__restrict__ active, uint8_t *__restrict__ flag, uint8_t *__restrict__ allfull, int split,
          unsigned symmask, unsigned *__restrict__ oddmask, bool full_spill) {
    extern __shared__ double sB[];  // [M][4] B^T, [M] per-codeword max, [M] support masks (u8)
    double *sBmax = sB + (size_t)M * 4;
    unsigned char *sBmask = reinterpret_cast<unsigned char *>(sBmax + M);
    CtaWork cw = work[blockIdx.x / split];
    if (!active[cw.word]) return;
    {   // this CTA's share of the work item's blocks (the item is sized for one fat backward CTA)
        const int nb = cw.blk_end - cw.blk_begin, part = blockIdx.x % split;
        const int lo = cw.blk_begin + (int)((int64_t)nb * part / split);
        cw.blk_end = cw.blk_begin + (int)((int64_t)nb * (part + 1) / split);
        cw.blk_begin = lo;
        if (cw.blk_begin >= cw.blk_end) return;
    }
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double a[BIDIAG ? 7 : 16], p[4], rmax;
    Masks4 mk;
    load_model4<BIDIAG>(pi, A, Bt, cw.word, M, sB, sBmax, sBmask, a, p, rmax, mk);
    __syncthreads();
    for (int b = cw.blk_begin + warp; b < cw.blk_end; b += BW_WARPS) {
        const Blk bk = blks[b];
        int T = lane < bk.nseq ? len_sorted[bk.first + lane] : 0;
        if (T > 0 && flag[bk.first + lane]) T = 0;  // handled by the exact log-space kernel
        bool af = false;
        const double ll = fwd4_run<BIDIAG, true>(T, bk.tmax, obs_blk + bk.obs_base + lane, reinterpret_cast<const double2 *>(sB),
                                                 reinterpret_cast<const double2 *>(sB) + M, sBmax, sBmask, a, p, rmax,
                                                 mk, spill + bk.spill_base * 64 + lane, af, 0, symmask,
                                                 oddmask + bk.spill_base, full_spill);
        if (T > 0) {
            ll_seq[bk.first + lane] = ll;
            allfull[bk.first + lane] = af ? 1 : 0;
            if (ll != ll) raise_flag(flag, bk.first + lane);  // precision guard: hand over (sticky)
        }
    }
}

// ---------------------------------------------------------------- backward + accumulate
// Warp-private emission-count update in precomputed rank order (see k_repack_blocks4): one
// conflict-free read-modify-write round per rank, rank 0 (distinct codewords) being the bulk.
// Round 0 and round 1 (taken on ~93 % of the steps of the benchmark data) are written out; only ranks >= 2
// loop.
//
// Shared-memory accesses of the backward kernel by 32-bit address.  The bases (B^T replica of the lane, count table of
// the warp) are computed once and made opaque (hold32), so that they stay in two registers; written as C++ pointers
// the compiler re-derives them from %tid and the shared window every step (~18 of 173 instructions per step).
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ unsigned hold32(unsigned x) { return __shfl_sync(0xffffffffu, x, threadIdx.x & 31); }
// read-only data (B^T): no memory clobber, free to move
__device__ __forceinline__ double2 lds128_ro(unsigned addr) {
    double2 v;
    asm("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ double2 lds128(unsigned addr) {
    double2 v;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void sts128(unsigned addr, double2 v) {
    asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(addr), "d"(v.x), "d"(v.y) : "memory");
}
// a double whose value is never used on the paths that do not assign it (no instruction, no zeroing)
__device__ __forceinline__ double undef_f64() {
    double x;
    asm("" : "=d"(x));
    return x;
}
// row = shared address of this lane's (j = 0, 1) count row; the (j = 2, 3) row sits `off23` bytes further
__device__ __forceinline__ void cnt_rmw4(unsigned row, unsigned off23, double g0, double g1, double g2, double g3) {
    double2 c01 = lds128(row), c23 = lds128(row + off23);
    c01.x += g0; c01.y += g1; c23.x += g2; c23.y += g3;
    sts128(row, c01); sts128(row + off23, c23);
}
// A __syncwarp() separates the rounds, so that a later round (or the next step's round 0) reads what an earlier round
// stored.  The rounds are straight-line predicated code behind a full-mask warp collective (the rank maximum), so the
// barriers (three instructions each, nine per step) could in principle go; without them k_bw_bwd4 measured 1.901 against
// 1.885 ms on config 3 (DESIGN.md §6), so they stay.
__device__ __forceinline__ void cnt_round_sync() { __syncwarp(); }
__device__ __forceinline__ void cnt_update4(unsigned row, unsigned off23, bool act, int rank, double g0, double g1,
                                            double g2, double g3) {
    const int myrank = act ? rank : -1;
    const int maxrank = __reduce_max_sync(0xffffffffu, myrank);
    if (myrank == 0) cnt_rmw4(row, off23, g0, g1, g2, g3);
    if (maxrank > 0) {  // warp-uniform
        cnt_round_sync();
        if (myrank == 1) cnt_rmw4(row, off23, g0, g1, g2, g3);
#pragma unroll 1
        for (int r = 2; r <= maxrank; ++r) {
            cnt_round_sync();
            if (myrank == r) cnt_rmw4(row, off23, g0, g1, g2, g3);
        }
    }
    cnt_round_sync();
}

// all four non-negative doubles strictly positive? (integer pipe: x > 0 <=> hi|lo != 0)
__device__ __forceinline__ bool all_pos4(double x0, double x1, double x2, double x3) {
    const unsigned m0 = (unsigned)__double2hiint(x0) | (unsigned)__double2loint(x0);
    const unsigned m1 = (unsigned)__double2hiint(x1) | (unsigned)__double2loint(x1);
    const unsigned m2 = (unsigned)__double2hiint(x2) | (unsigned)__double2loint(x2);
    const unsigned m3 = (unsigned)__double2hiint(x3) | (unsigned)__double2loint(x3);
    return min(min(m0, m1), min(m2, m3)) != 0u;
}
// x == 0 -> smallest denormal, else x (non-negative input; integer pipe, branch-free)
__device__ __forceinline__ double zero_to_tiny(double x) {
    const int hi = __double2hiint(x), lo = __double2loint(x);
    return __hiloint2double(hi, lo | (((hi | lo) == 0) ? 1 : 0));
}
// smallest denormal if x > 0, else +0.0 (non-negative input; integer pipe)
__device__ __forceinline__ double pos_to_tiny(double x) {
    return __hiloint2double(0, ((__double2hiint(x) | __double2loint(x)) != 0) ? 1 : 0);
}
// Asynchronous 16-byte global -> shared copy (LDGSTS): the codeword chunk of the next 8 steps lands in a per-thread
// shared-memory slot without holding registers while it is in flight.
__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gsrc));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
constexpr int BWD4_SPILL_PAD = 2;    // rows of padding in front of the alpha spill and its odd-row masks (see the step macro)
constexpr int BWD_L2_PREFETCH = 12;  // steps ahead of use for prefetch.global.L2 of the alpha spill (even)
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
// the same under a predicate instead of a branch (ptxas drains the load scoreboards at the first branch of a loop body
// that has a use of the loaded registers somewhere behind it: bwltr_kernels.cuh)
__device__ __forceinline__ void prefetch_l2_if(const void *p, bool on) {
    asm volatile("{\n\t.reg .pred pf;\n\tsetp.ne.u32 pf, %1, 0;\n\t@pf prefetch.global.L2 [%0];\n\t}" ::"l"(p), "r"((unsigned)on));
}
constexpr double LEAN_MIN = 0x1p-500;  // the lean backward step needs its three sums above this
constexpr unsigned LEAN_MIN_HI = (1023u - 500u) << 20;  // high word of LEAN_MIN = 2^-500

// Normalisation without a division per step.  sum_i alpha_t(i) beta_t(i) = P(O|lambda) at EVERY t (it is what the
// reference subtracts as logP, :389-410), and every rescale here is an exact power of two, so
//     norm_t = sum_i alpha-hat_t(i) beta-hat_t(i) = norm_{T-1} * 2^k_t   up to rounding.
// One true division per sequence gives rref = 1 / norm_{T-1}; afterwards r_t = rref * 2^-k_t comes from exponent
// arithmetic: x = norm_t * rref ~ 2^k_t (1 + d); a quarter added to x's mantissa makes the exponent field read k_t
// whether d is just above or just below zero.
__device__ __forceinline__ double recip_from_ref(double norm, double rref) {
    const double x = norm * rref;
    const int e = (__double2hiint(x) + 0x00040000) & 0x7ff00000;
    return __hiloint2double(__double2hiint(rref) - e + 0x3ff00000, __double2loint(rref));
}
// The same identity is the backward pass's precision check: |norm_t * r_t - 1| must stay at rounding level
// (~T * 1e-16).  A beta-hat that lost its bits in a denormal / clamped value and later carries the sequence
// (or any other loss in alpha-hat or beta-hat that matters for gamma) shows up here as a deviation of
// sum_i alpha_t(i) beta_t(i) from P(O); beyond NORM_TOL the sequence is handed to the exact log-space kernel.
constexpr double NORM_TOL = 1e-10;
constexpr unsigned NORM_TOL_HI = 0x3DDB7CDFu;  // high word of 1e-10
// (integer pipe: the high word of |x| orders like |x|; a NaN compares above every threshold)
__device__ __forceinline__ bool norm_consistent(double norm, double r) {
    return ((unsigned)__double2hiint(fma(norm, r, -1.0)) & 0x7fffffffu) < NORM_TOL_HI;
}

// State of one lane's backward recursion.
template <bool BIDIAG>
struct Bwd4State {
    double v0, v1, v2, v3;        // v_j = b_j(o_{t+1}) * beta-hat_{t+1}(j)
    double X[BIDIAG ? 7 : 16];    // sum_t u_i w_j (a_ij applied at the flush)
    double rref;                  // 1 / sum_i alpha-hat_{T-1}(i): reference of the normalisation (see above)
    unsigned seenX;               // (i,j) pairs for which a finite xi term existed
    bool imprecise;
    bool vpos;                    // every v_j > 0 (lets the lean path skip the structural masks)
};

// Careful version of one backward step (all clamps, structural masks, precision hand-over).
// Taken when the lean path's two group tests fail, at the first step of a sequence, and for
// words whose B holds exact zeros.  Returns gamma in g[], updates st (v, X, seenX).
template <bool BIDIAG>
__device__ __noinline__ void bwd4_step_slow(Bwd4State<BIDIAG> &st, const double *a, const double2 *__restrict__ sB01,
                                            const double2 *__restrict__ sB23,
                                            unsigned sym, bool last, double al0, double al1, double al2, double al3,
                                            double *g) {
    double v0 = st.v0, v1 = st.v1, v2 = st.v2, v3 = st.v3;
    double h0 = 1.0, h1 = 1.0, h2 = 1.0, h3 = 1.0;  // log beta_{T-1} = 0 (:363)
    double w0 = 0.0, w1 = 0.0, w2 = 0.0, w3 = 0.0;
    if (!last) {
        // un-normalised beta_t(i) = sum_j a_ij b_j(o_{t+1}) beta_{t+1}(j)  (:163-199)
        double q[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            q[i] = a_at<BIDIAG>(a, i, 0) * v0 + a_at<BIDIAG>(a, i, 1) * v1 + a_at<BIDIAG>(a, i, 2) * v2 +
                   a_at<BIDIAG>(a, i, 3) * v3;
            if (q[i] == 0.0 && ((a_at<BIDIAG>(a, i, 0) > 0.0 && v0 > 0.0) || (a_at<BIDIAG>(a, i, 1) > 0.0 && v1 > 0.0) ||
                                (a_at<BIDIAG>(a, i, 2) > 0.0 && v2 > 0.0) || (a_at<BIDIAG>(a, i, 3) > 0.0 && v3 > 0.0)))
                q[i] = tiny_pos();
        }
        const double qs = (q[0] + q[1]) + (q[2] + q[3]);
        const double sc = qs > 0.0 ? pow2_rescale_noacc(qs) : 1.0;
        h0 = q[0] * sc; h1 = q[1] * sc; h2 = q[2] * sc; h3 = q[3] * sc;
        // (sum q can reach N * 2, i.e. sc < 1: a denormal marker must not be flushed by the rescale — beta_t(i) is
        // finite in the reference, and gamma_t(i) / v_i below only stay positive if h_i does)
        if (h0 == 0.0 && q[0] > 0.0) h0 = tiny_pos();
        if (h1 == 0.0 && q[1] > 0.0) h1 = tiny_pos();
        if (h2 == 0.0 && q[2] > 0.0) h2 = tiny_pos();
        if (h3 == 0.0 && q[3] > 0.0) h3 = tiny_pos();
        w0 = v0 * sc; w1 = v1 * sc; w2 = v2 * sc; w3 = v3 * sc;
    }
    // gamma_t(i) = alpha_t(i) beta_t(i) / sum_i alpha_t(i) beta_t(i)   (:389-394)
    double g0 = al0 * h0, g1 = al1 * h1, g2 = al2 * h2, g3 = al3 * h3;
    double norm = (g0 + g1) + (g2 + g3);
    double u0 = al0, u1 = al1, u2 = al2, u3 = al3;
    double r;
    if (!(norm >= TINY_STEP)) {
        // forward and backward mass sit on (almost) disjoint states: redo the products 2^1000
        // larger so they neither underflow nor blow up 1/norm; the bits may already be gone,
        // so the sequence is also handed over to the exact kernel
        st.imprecise = true;
        const double big = 0x1p500;
        u0 = al0 * big; u1 = al1 * big; u2 = al2 * big; u3 = al3 * big;
        g0 = u0 * (h0 * big); g1 = u1 * (h1 * big); g2 = u2 * (h2 * big); g3 = u3 * (h3 * big);
        w0 *= big; w1 *= big; w2 *= big; w3 *= big;
        norm = (g0 + g1) + (g2 + g3);
        r = norm > 0.0 ? 1.0 / norm : 0.0;
    } else {
        r = 1.0 / norm;
        // sum_i alpha_t(i) beta_t(i) must still be P(O) (times a power of two): the backward precision check
        if (last) st.rref = r;
        else if (!norm_consistent(norm, recip_from_ref(norm, st.rref))) st.imprecise = true;
    }
    g0 *= r; g1 *= r; g2 *= r; g3 *= r;
    if (g0 == 0.0 && al0 > 0.0 && h0 > 0.0) g0 = tiny_pos();
    if (g1 == 0.0 && al1 > 0.0 && h1 > 0.0) g1 = tiny_pos();
    if (g2 == 0.0 && al2 > 0.0 && h2 > 0.0) g2 = tiny_pos();
    if (g3 == 0.0 && al3 > 0.0 && h3 > 0.0) g3 = tiny_pos();
    g[0] = g0; g[1] = g1; g[2] = g2; g[3] = g3;
    if (!last) {
        // xi_t(i,j) = alpha_t(i) a_ij b_j(o_{t+1}) beta_{t+1}(j) / norm   (:397-410)
        u0 *= r; u1 *= r; u2 *= r; u3 *= r;
        const double uu[4] = {u0, u1, u2, u3}, ww[4] = {w0, w1, w2, w3};
        if (BIDIAG) {
#pragma unroll
            for (int i = 0; i < 4; ++i) st.X[i] = fma(uu[i], ww[i], st.X[i]);
#pragma unroll
            for (int i = 0; i < 3; ++i) st.X[4 + i] = fma(uu[i], ww[i + 1], st.X[4 + i]);
        } else {
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) st.X[i * 4 + j] = fma(uu[i], ww[j], st.X[i * 4 + j]);
        }
        const unsigned mv = (v0 > 0.0 ? 1u : 0u) | (v1 > 0.0 ? 2u : 0u) | (v2 > 0.0 ? 4u : 0u) | (v3 > 0.0 ? 8u : 0u);
        st.seenX |= (al0 > 0.0 ? mv : 0u) | (al1 > 0.0 ? mv << 4 : 0u) | (al2 > 0.0 ? mv << 8 : 0u) |
                    (al3 > 0.0 ? mv << 12 : 0u);
    }
    // v_j = b_j(o_t) beta-hat_t(j) for step t-1
    const double2 b01 = sB01[sym], b23 = sB23[sym];
    v0 = b01.x * h0; v1 = b01.y * h1; v2 = b23.x * h2; v3 = b23.y * h3;
    const double vs = (v0 + v1) + (v2 + v3);
    if (!(vs >= TINY_STEP)) {
        // tiny emission column: exponent-split products (the scale of v is free)
        double o[4];
        int E;
        if (exact_products4(h0, h1, h2, h3, b01.x, b01.y, b23.x, b23.y, o, &E) == 2) st.imprecise = true;
        v0 = o[0]; v1 = o[1]; v2 = o[2]; v3 = o[3];
    } else {
        if (v0 == 0.0 && b01.x > 0.0 && h0 > 0.0) v0 = tiny_pos();
        if (v1 == 0.0 && b01.y > 0.0 && h1 > 0.0) v1 = tiny_pos();
        if (v2 == 0.0 && b23.x > 0.0 && h2 > 0.0) v2 = tiny_pos();
        if (v3 == 0.0 && b23.y > 0.0 && h3 > 0.0) v3 = tiny_pos();
    }
    st.v0 = v0; st.v1 = v1; st.v2 = v2; st.v3 = v3;
    st.vpos = (v0 > 0.0) & (v1 > 0.0) & (v2 > 0.0) & (v3 > 0.0);
}

// Careful version of the LAST part of a backward step only: v_j = b_j(o_t) beta-hat_t(j) when the lean step found
// that sum tiny (its gamma / xi part had passed the magnitude tests and is already committed).  Same arithmetic
// as the tail of bwd4_step_slow.  Returns true if the sequence has to be handed to the exact kernel.
__device__ __noinline__ bool bwd4_v_slow(double h0, double h1, double h2, double h3, double b0, double b1, double b2,
                                         double b3, double *v) {
    bool imprecise = false;
    double v0 = b0 * h0, v1 = b1 * h1, v2 = b2 * h2, v3 = b3 * h3;
    const double vs = (v0 + v1) + (v2 + v3);
    if (!(vs >= TINY_STEP)) {
        double o[4];
        int E;
        if (exact_products4(h0, h1, h2, h3, b0, b1, b2, b3, o, &E) == 2) imprecise = true;
        v0 = o[0]; v1 = o[1]; v2 = o[2]; v3 = o[3];
    } else {
        if (v0 == 0.0 && b0 > 0.0 && h0 > 0.0) v0 = tiny_pos();
        if (v1 == 0.0 && b1 > 0.0 && h1 > 0.0) v1 = tiny_pos();
        if (v2 == 0.0 && b2 > 0.0 && h2 > 0.0) v2 = tiny_pos();
        if (v3 == 0.0 && b3 > 0.0 && h3 > 0.0) v3 = tiny_pos();
    }
    v[0] = v0; v[1] = v1; v[2] = v2; v[3] = v3;
    return imprecise;
}

// (max, sum exp(. - max)) of log P_r over the sequences of one CTA work item, in a fixed order; the pairs of a
// word's CTAs are combined by k_bw_reduce (HMM/hmm_training.py:503).  NaN marks (sequences still waiting for the
// exact kernel) and -inf (impossible sequences) drop out.  Called by all BW_THREADS threads; out[0..1].
__device__ __forceinline__ void cta_ll_stat(const Blk *__restrict__ blks, const CtaWork &cw, const double *__restrict__ ll_seq,
                                            double (*sRed)[20], double *__restrict__ out) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nthreads = blockDim.x, nwarps = nthreads >> 5;
    const int r0 = blks[cw.blk_begin].first, r1 = blks[cw.blk_end - 1].first + blks[cw.blk_end - 1].nseq;
    // The sums are taken by the first 128 threads whatever the CTA's size, so that the pair does not depend on the
    // kernel that takes it (k_bw_bwd4's fat CTA or k_bw_llstat_fix's small one): same order, same bits.
    constexpr int NT = 128;
    double m = neg_inf();
    if (tid < NT)
        for (int r = r0 + tid; r < r1; r += NT) m = fmax(m, ll_seq[r]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) sRed[warp][0] = m;
    __syncthreads();
    m = fmax(fmax(sRed[0][0], sRed[1][0]), fmax(sRed[2][0], sRed[3][0]));
    double sum = 0.0;
    if (tid < NT && m > neg_inf())
        for (int r = r0 + tid; r < r1; r += NT) {
            const double l = ll_seq[r];
            if (l > neg_inf()) sum += exp(l - m);
        }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) sRed[warp][1] = sum;
    __syncthreads();
    if (tid == 0) {
        out[0] = m;
        out[1] = ((sRed[0][1] + sRed[1][1]) + sRed[2][1]) + sRed[3][1];
    }
    (void)nwarps;
}

// Pipelined first E-step only: there the exact kernel runs AFTER the staged backward passes, so a sequence the
// forward pass handed over still carried its NaN mark when k_bw_bwd4 took the CTA's statistic.  Once the exact
// kernel has filled in those log-likelihoods this kernel retakes every CTA's pair (it returns at once if no flag
// was ever raised), which makes the staged pass equal to forward -> exact -> backward.
__global__ void __launch_bounds__(BW_THREADS)
k_bw_llstat_fix(const CtaWork *__restrict__ work, const Blk *__restrict__ blks, const double *__restrict__ ll_seq,
                const int32_t *__restrict__ active, const uint8_t *__restrict__ flag, double *__restrict__ partials,
                int64_t pstride, int M) {
    if (!any_flag_raised(flag)) return;
    __shared__ double sRed[BW_WARPS][20];
    const CtaWork cw = work[blockIdx.x];
    if (!active[cw.word]) return;
    cta_ll_stat(blks, cw, ll_seq, sRed, partials + (size_t)blockIdx.x * pstride + 20 + (size_t)M * 4);
}

// Partial layout per CTA (and accumulator layout per word): [pi N][xi N*N][cnt M*N].
//
// alpha-hat comes from the spill at even steps; at odd steps it is rebuilt from the even row before it (fwd4_rebuild),
// except for the lanes the forward pass's mask word of that step names (rows it had to write).  The time loop runs
// four steps (two pairs) per iteration with fixed roles for the two sets of even-row registers (E0 / E1), so that
// loading the next pair's row needs no register-to-register copies.
// MT = 256 (the reference's codebook size, CodeVector/main.py) makes every shared-memory offset a literal;
// MT = 0 takes M at run time.
//
// One fat CTA per SM: blockDim.x / 32 warps (16 for the left-to-right kernel, 12 for the dense one, fewer when the
// count tables of a large alphabet need the room) share ONE copy of the word's B^T, which leaves room to store it
// REP = 8 times: lane l gathers from replica l & 7, so the eight lanes of a quarter-warp always hit eight different
// 16-byte bank slots.  ncu on the 4-warp version: 19.5 of the 69.5 shared-memory wavefronts per warp-step were this
// gather (ideal 8), and that pipe — 72 % busy — is what the kernel waits for.  The count tables stay warp-private.
// Shared memory: [M * REP] double2 (b0, b1), [M * REP] double2 (b2, b3), nwarps x [M] x 2 double2 counts,
// [nwarps][4] gamma_0 sums.
template <bool BIDIAG, int MT, int REP>
__global__ void __launch_bounds__(BIDIAG ? BWD4_MAX_WARPS * 32 : 384, 1)
k_bw_bwd4(const CtaWork *__restrict__ work, const Blk *__restrict__ blks, const uint4 *__restrict__ obs_blk,
          const int32_t *__restrict__ len_sorted, const double *__restrict__ A, const double *__restrict__ Bt, int M_rt,
          const double2 *__restrict__ spill, const double *__restrict__ ll_seq, const int32_t *__restrict__ active,
          const int32_t *__restrict__ b_has_zero, const uint8_t *__restrict__ allfull, double *__restrict__ partials,
          int64_t pstride, uint8_t *__restrict__ flag, int32_t *__restrict__ new_flags,
          const unsigned *__restrict__ oddmask, bool full_spill) {
    using S16 = Sym<uint16_t>;
    const int M = MT ? MT : M_rt;
    const int pf_lanes = full_spill ? 16 : 8;  // 128-byte lines of each pair prefetched towards L2
    const int nthreads = blockDim.x, nwarps = nthreads >> 5;
    extern __shared__ double smem[];
    double *sB = smem;                                    // B^T replicated: [M * REP] (b0,b1) then [M * REP] (b2,b3)
    double *sCnt = smem + (size_t)M * REP * 4;            // [nwarps] x { [M] double2 (j=0,1), [M] double2 (j=2,3) }
    double *sPi = sCnt + (size_t)M * 4 * nwarps;          // [nwarps][4] gamma_0 sums
    __shared__ double sRed[BWD4_MAX_WARPS][20];
    __shared__ unsigned sSeen;
    __shared__ uint4 sW[2][BWD4_MAX_WARPS * 32];  // codeword chunks in flight (cp.async), double-buffered per thread

    const CtaWork cw = work[blockIdx.x];
    double *part = partials + (size_t)blockIdx.x * pstride;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (!active[cw.word]) return;
    {
        const double2 *src = reinterpret_cast<const double2 *>(Bt + (size_t)cw.word * M * 4);
        double2 *dst01 = reinterpret_cast<double2 *>(sB), *dst23 = dst01 + (size_t)M * REP;
        for (int e = tid; e < M * REP; e += nthreads) {
            const int sym = e / REP;
            dst01[e] = __ldg(src + 2 * sym);
            dst23[e] = __ldg(src + 2 * sym + 1);
        }
        for (int e = tid; e < M * 4 * nwarps + nwarps * 4; e += nthreads) sCnt[e] = 0.0;  // counts + sPi
        if (tid == 0) sSeen = 0u;
    }
    double a[BIDIAG ? 7 : 16];
    load_A4<BIDIAG>(A + (size_t)cw.word * 16, a);
    // lean path precondition (structure only): B > 0 everywhere and no all-zero row in A, so
    // every beta_t(i) and every v_j is finite in the reference; whether every alpha_t(i) is
    // finite is read off the spilled values
    const Masks4 mk = make_masks4(A + (size_t)cw.word * 16, nullptr);
    const bool lean_ok = (b_has_zero[cw.word] == 0) && (lut4(mk.lutB, 0xFu) == 0xFu);
    const double tiny = tiny_pos();
    __syncthreads();

    double2 *cntw01 = reinterpret_cast<double2 *>(sCnt + (size_t)warp * M * 4);  // (j = 2, 3) rows M entries further
    // this lane's replica column of B^T: the row of codeword sym is at [sym * REP]
    const double2 *sB01 = reinterpret_cast<const double2 *>(sB) + (lane & (REP - 1)), *sB23 = sB01 + (size_t)M * REP;
    double *mypi = sPi + (size_t)warp * 4;
    // 32-bit shared addresses of the lane's B^T replica column and of the warp's count table, held in registers
    const unsigned bbase = hold32(smem_u32(sB01)), cbase = hold32(smem_u32(cntw01));
    const unsigned B23_OFF = (unsigned)M * REP * 16u, CNT23_OFF = (unsigned)M * 16u;
    Bwd4State<BIDIAG> st;
#pragma unroll
    for (int q = 0; q < (BIDIAG ? 7 : 16); ++q) st.X[q] = 0.0;
    st.seenX = 0u;

    for (int b = cw.blk_begin + warp; b < cw.blk_end; b += nwarps) {
        const Blk bk = blks[b];
        int T = 0;
        bool apos = false;
        if (lane < bk.nseq) {
            T = len_sorted[bk.first + lane];
            if (!(ll_seq[bk.first + lane] > neg_inf())) T = 0;  // impossible sequence: contributes nothing (:391-394)
            if (flag[bk.first + lane]) T = 0;                   // exact log-space kernel did this one
            apos = allfull[bk.first + lane] != 0;               // forward pass: every alpha-hat of this sequence > 0
        }
        st.v0 = st.v1 = st.v2 = st.v3 = 0.0;
        st.imprecise = false;
        st.vpos = false;
        st.rref = 1.0;
        const uint4 *op = obs_blk + bk.obs_base + lane;
        const double2 *sp = spill + bk.spill_base * 64 + lane;
        // the block's first row as a 32-bit index (the spill, 1 KB a row, fits in device memory): the mask words are
        // then addressed from the kernel argument, without a 64-bit pointer held through the time loop
        const int mrow = (int)bk.spill_base;
        const int nch = (bk.tmax + SPC4 - 1) / SPC4;
        // Even-step alpha-hat rows and the odd-row lane masks of their pairs (odd 2k + 1, even 2k): pair k is held in
        // set 0 if k is odd, in set 1 if k is even.  The even step of a pair loads the next pair's row into the other set.
        double2 E0_01 = make_double2(0.0, 0.0), E0_23 = E0_01, E1_01 = E0_01, E1_23 = E0_01;
        unsigned M0 = 0u, M1 = 0u;
        {
            // the rows of the block's first BWD_L2_PREFETCH steps are not covered by the prefetch inside the loop
            // (even rows only, unless every row was written)
            const int r1 = nch * SPC4, r0 = max(r1 - BWD_L2_PREFETCH, 0);
            const char *base = reinterpret_cast<const char *>(sp - lane) + (size_t)r0 * 1024;
            for (int l = lane; l < (r1 - r0) * 8; l += 32)
                if (full_spill || !((l >> 3) & 1)) prefetch_l2(base + (size_t)l * 128);
            const int ta = bk.tmax - 1;  // the first step of the block, in pair k = ta / 2
            const double2 x01 = __ldcs(sp + (size_t)(ta & ~1) * 64), x23 = __ldcs(sp + (size_t)(ta & ~1) * 64 + 32);
            const unsigned mw = (ta & 1) ? __ldg(oddmask + mrow + ta) : 0u;
            if ((ta >> 1) & 1) { E0_01 = x01; E0_23 = x23; M0 = mw; }
            else               { E1_01 = x01; E1_23 = x23; M1 = mw; }
        }
        int wbuf = 0;
        cp_async16(&sW[0][tid], op + (size_t)(nch - 1) * 32);
        cp_async_commit();

// One backward step at time T_ (ODD_ = T_ & 1 is a literal) of the pair held in set X_ (Y_ = the other set).
// PACKED_ = the step's codeword | rank << SYM_BITS.
#define HMMB_BWD_STEP(T_, ODD_, X_, Y_, SP_, PACKED_)                                                               \
    {                                                                                                               \
        const int t = (T_);                                                                                         \
        const double2 *spt = (SP_); /* = sp + t * 64: every address below is an immediate offset from it */         \
        const unsigned packed = (PACKED_);                                                                          \
        if (t < bk.tmax) { /* warp-uniform */                                                                       \
            const unsigned sym = packed & SYM_MASK;                                                                 \
            const bool act = t < T;                                                                                 \
            const unsigned brow = bbase + sym * (unsigned)(REP * 16);                                               \
            const unsigned crow = cbase + sym * 16u;                                                                \
            double2 bc01, bc23; /* b(o_t): gathered at the top of an odd step, in the lean path of an even one */   \
            double al0, al1, al2, al3;                                                                              \
            if (ODD_) {                                                                                             \
                /* alpha-hat_t of a plain forward step, rebuilt from the even row t - 1 (fwd4_rebuild); the      */ \
                /* lanes whose step was not plain wrote their row, and the pair's mask word says which (rare)   */ \
                bc01 = lds128_ro(brow); bc23 = lds128_ro(brow + B23_OFF);                                           \
                double2 x01 = E##X_##_01, x23 = E##X_##_23;                                                         \
                fwd4_rebuild<BIDIAG>(a, x01, x23, bc01, bc23, tiny);                                                \
                if (M##X_) { /* warp-uniform */                                                                     \
                    if ((M##X_ >> lane) & 1u) { x01 = __ldcs(spt); x23 = __ldcs(spt + 32); }                        \
                }                                                                                                   \
                al0 = x01.x; al1 = x01.y; al2 = x23.x; al3 = x23.y;                                                 \
            } else {                                                                                                \
                al0 = E##X_##_01.x; al1 = E##X_##_01.y; al2 = E##X_##_23.x; al3 = E##X_##_23.y;                     \
                /* the next pair's even row (t - 2) and mask word go straight into the other set (free since the */ \
                /* odd step of this pair: no copies).  One step ahead of its first use is enough because the rows */\
                /* were pulled into L2 BWD_L2_PREFETCH steps ago.  Unconditional: a row at or beyond a lane's own */\
                /* T is never used, and for t = 0 the loads land in the previous block's tail / the front padding */\
                /* of the spill and of the masks (BWD4_SPILL_PAD).                                               */ \
                E##Y_##_01 = __ldcs(spt - 128);                                                                     \
                E##Y_##_23 = __ldcs(spt - 128 + 32);                                                                \
                M##Y_ = __ldg(oddmask + (mrow + t - 1));                                                            \
            }                                                                                                       \
            const int rank = (int)(packed >> SYM_BITS);                                                             \
            double g0 = undef_f64(), g1 = undef_f64(), g2 = undef_f64(), g3 = undef_f64();                          \
            if (act) {                                                                                              \
                bool done = false;                                                                                  \
                if (lean_ok && st.vpos) { /* (vpos is false until the sequence's first step has run) */             \
                    /* lean path: beta_t(i) ~ q_i = sum_j a_ij v_j (:163-199); gamma_t(i) = al_i q_i / norm   */    \
                    /* (:389-394); xi_t(i,j) = al_i a_ij v_j / norm (:397-410); norm = sum_i al_i q_i.  The    */   \
                    /* denormal addends keep a finite-but-underflowed log value (barely) positive.            */    \
                    double q0, q1, q2, q3;                                                                          \
                    if (BIDIAG) {                                                                                   \
                        q0 = fma(a[4], st.v1, fma(a[0], st.v0, tiny));                                              \
                        q1 = fma(a[5], st.v2, fma(a[1], st.v1, tiny));                                              \
                        q2 = fma(a[6], st.v3, fma(a[2], st.v2, tiny));                                              \
                        q3 = fma(a[3], st.v3, tiny);                                                                \
                    } else {                                                                                        \
                        q0 = fma(a[3], st.v3, fma(a[2], st.v2, fma(a[1], st.v1, fma(a[0], st.v0, tiny))));          \
                        q1 = fma(a[7], st.v3, fma(a[6], st.v2, fma(a[5], st.v1, fma(a[4], st.v0, tiny))));          \
                        q2 = fma(a[11], st.v3, fma(a[10], st.v2, fma(a[9], st.v1, fma(a[8], st.v0, tiny))));        \
                        q3 = fma(a[15], st.v3, fma(a[14], st.v2, fma(a[13], st.v1, fma(a[12], st.v0, tiny))));      \
                    }                                                                                               \
                    const double qs = (q0 + q1) + (q2 + q3);                                                        \
                    const double c0 = al0 * q0, c1 = al1 * q1, c2 = al2 * q2, c3 = al3 * q3;                        \
                    const double norm = (c0 + c1) + (c2 + c3);                                                      \
                    const double r = recip_from_ref(norm, st.rref); /* 1 / norm without a division */               \
                    /* the sums are positive doubles: compare their high words on the integer pipe */               \
                    const unsigned lo2 = min((unsigned)__double2hiint(norm), (unsigned)__double2hiint(qs));         \
                    if ((lo2 >= LEAN_MIN_HI) & norm_consistent(norm, r) && (apos || all_pos4(al0, al1, al2, al3))) {\
                        /* gamma and xi are committed here; what is left of the step is v for step t - 1 */         \
                        g0 = fma(c0, r, tiny); g1 = fma(c1, r, tiny); g2 = fma(c2, r, tiny); g3 = fma(c3, r, tiny); \
                        const double u0 = al0 * r, u1 = al1 * r, u2 = al2 * r, u3 = al3 * r;                        \
                        if (BIDIAG) {                                                                               \
                            st.X[0] = fma(u0, st.v0, st.X[0]); st.X[1] = fma(u1, st.v1, st.X[1]);                   \
                            st.X[2] = fma(u2, st.v2, st.X[2]); st.X[3] = fma(u3, st.v3, st.X[3]);                   \
                            st.X[4] = fma(u0, st.v1, st.X[4]); st.X[5] = fma(u1, st.v2, st.X[5]);                   \
                            st.X[6] = fma(u2, st.v3, st.X[6]);                                                      \
                        } else {                                                                                    \
                            st.X[0] = fma(u0, st.v0, st.X[0]);   st.X[1] = fma(u0, st.v1, st.X[1]);                 \
                            st.X[2] = fma(u0, st.v2, st.X[2]);   st.X[3] = fma(u0, st.v3, st.X[3]);                 \
                            st.X[4] = fma(u1, st.v0, st.X[4]);   st.X[5] = fma(u1, st.v1, st.X[5]);                 \
                            st.X[6] = fma(u1, st.v2, st.X[6]);   st.X[7] = fma(u1, st.v3, st.X[7]);                 \
                            st.X[8] = fma(u2, st.v0, st.X[8]);   st.X[9] = fma(u2, st.v1, st.X[9]);                 \
                            st.X[10] = fma(u2, st.v2, st.X[10]); st.X[11] = fma(u2, st.v3, st.X[11]);               \
                            st.X[12] = fma(u3, st.v0, st.X[12]); st.X[13] = fma(u3, st.v1, st.X[13]);               \
                            st.X[14] = fma(u3, st.v2, st.X[14]); st.X[15] = fma(u3, st.v3, st.X[15]);               \
                        }                                                                                           \
                        st.seenX = 0xffffu; /* every alpha_i > 0 and every v_j > 0 */                               \
                        const double sc = pow2_rescale_noacc(qs);                                                   \
                        const double h0 = q0 * sc, h1 = q1 * sc, h2 = q2 * sc, h3 = q3 * sc; /* beta-hat_t */       \
                        if (!(ODD_)) { bc01 = lds128_ro(brow); bc23 = lds128_ro(brow + B23_OFF); }                  \
                        st.v0 = fma(bc01.x, h0, tiny); st.v1 = fma(bc01.y, h1, tiny);                               \
                        st.v2 = fma(bc23.x, h2, tiny); st.v3 = fma(bc23.y, h3, tiny);                               \
                        const double vs = (st.v0 + st.v1) + (st.v2 + st.v3);                                        \
                        if ((unsigned)__double2hiint(vs) < LEAN_MIN_HI) { /* tiny emission column: careful v */     \
                            double vv[4];                                                                           \
                            /* (q > 0 on this path: a beta-hat the rescale flushed is still a finite log value) */ \
                            if (bwd4_v_slow(zero_to_tiny(h0), zero_to_tiny(h1), zero_to_tiny(h2), zero_to_tiny(h3), bc01.x, bc01.y,     \
                                            bc23.x, bc23.y, vv)) st.imprecise = true; \
                            st.v0 = vv[0]; st.v1 = vv[1]; st.v2 = vv[2]; st.v3 = vv[3];                             \
                            st.vpos = all_pos4(vv[0], vv[1], vv[2], vv[3]);                                         \
                        }                                                                                           \
                        done = true;                                                                                \
                    }                                                                                               \
                }                                                                                                   \
                if (!done) {                                                                                        \
                    if (t == T - 1) {                                                                               \
                        /* first step of the sequence, inline: log beta_{T-1} = 0 (:363), so beta-hat = 1, gamma = */\
                        /* alpha-hat / sum alpha-hat, no xi term, v = b(o_{T-1}).  The one true division of the     */\
                        /* sequence; every later step derives its 1 / norm from it (recip_from_ref).               */\
                        const double n0 = (al0 + al1) + (al2 + al3); /* in [1, 2): the forward pass rescaled it */  \
                        const double r0 = 1.0 / n0;                                                                 \
                        st.rref = r0;                                                                               \
                        g0 = fma(al0, r0, pos_to_tiny(al0)); g1 = fma(al1, r0, pos_to_tiny(al1));                   \
                        g2 = fma(al2, r0, pos_to_tiny(al2)); g3 = fma(al3, r0, pos_to_tiny(al3));                   \
                        if (!(ODD_)) { bc01 = lds128_ro(brow); bc23 = lds128_ro(brow + B23_OFF); }                  \
                        st.v0 = bc01.x; st.v1 = bc01.y; st.v2 = bc23.x; st.v3 = bc23.y;                             \
                        st.vpos = all_pos4(bc01.x, bc01.y, bc23.x, bc23.y);                                         \
                    } else {                                                                                        \
                        /* the careful step works on a stack copy so that `st` itself never has its address */      \
                        /* taken and stays in registers on the lean path                                     */     \
                        Bwd4State<BIDIAG> tmp = st;                                                                 \
                        double g[4];                                                                                \
                        bwd4_step_slow<BIDIAG>(tmp, a, sB01, sB23, sym * REP, false, al0, al1, al2, al3, g);        \
                        st = tmp;                                                                                   \
                        g0 = g[0]; g1 = g[1]; g2 = g[2]; g3 = g[3];                                                 \
                    }                                                                                               \
                }                                                                                                   \
            }                                                                                                       \
            if (t == 0) { /* gamma_0 sums (:415-426): once per block, fixed-order warp tree (inactive lanes add 0) */ \
                const int am = act ? -1 : 0; /* (bit masks: g is not defined for a lane without a frame) */         \
                double p0 = __hiloint2double(__double2hiint(g0) & am, __double2loint(g0) & am);                     \
                double p1 = __hiloint2double(__double2hiint(g1) & am, __double2loint(g1) & am);                     \
                double p2 = __hiloint2double(__double2hiint(g2) & am, __double2loint(g2) & am);                     \
                double p3 = __hiloint2double(__double2hiint(g3) & am, __double2loint(g3) & am);                     \
                _Pragma("unroll") for (int o = 16; o > 0; o >>= 1) {                                                \
                    p0 += __shfl_xor_sync(0xffffffffu, p0, o); p1 += __shfl_xor_sync(0xffffffffu, p1, o);           \
                    p2 += __shfl_xor_sync(0xffffffffu, p2, o); p3 += __shfl_xor_sync(0xffffffffu, p3, o);           \
                }                                                                                                   \
                if (lane == 0) { mypi[0] += p0; mypi[1] += p1; mypi[2] += p2; mypi[3] += p3; }                      \
            }                                                                                                       \
            /* emission-count numerators (:460-500): warp-private rows, conflict-free rank order */                \
            cnt_update4(crow, CNT23_OFF, act, rank, g0, g1, g2, g3);                                                \
        }                                                                                                           \
    }

        const double2 *spp = sp + (size_t)(nch * SPC4 - 2) * 64;  // alpha-hat row of the even step of the pair
        for (int c = nch - 1; c >= 0; --c) {
            cp_async_wait_all();  // (issued eight steps ago)
            uint4 w = sW[wbuf][tid];
            wbuf ^= 1;
            if (c > 0) {  // the next 8 codewords, straight into the other slot
                cp_async16(&sW[wbuf][tid], op + (size_t)(c - 1) * 32);
                cp_async_commit();
            }
            // two pairs per iteration, so that the two register sets keep fixed roles (pair 2 qq + 1 in set 0)
#pragma unroll 1
            for (int qq = SPC4 / 4 - 1; qq >= 0; --qq) {
                // pull the even alpha-hat row that will be needed BWD_L2_PREFETCH steps from now (1 KB) towards L2:
                // lanes 0..7 take one 128-byte line each (lanes 8..15 the odd row after it, if every row was written)
                if (c * SPC4 + 4 * qq + 2 >= BWD_L2_PREFETCH && lane < pf_lanes)
                    prefetch_l2(reinterpret_cast<const char *>(spp) - BWD_L2_PREFETCH * 1024 + lane * (128 - 16));
                unsigned p = S16::pop_back(w);
                HMMB_BWD_STEP(c * SPC4 + 4 * qq + 3, 1, 0, 1, spp + 64, p)
                p = S16::pop_back(w);
                HMMB_BWD_STEP(c * SPC4 + 4 * qq + 2, 0, 0, 1, spp, p)
                spp -= 2 * 64;
                if (c * SPC4 + 4 * qq >= BWD_L2_PREFETCH && lane < pf_lanes)
                    prefetch_l2(reinterpret_cast<const char *>(spp) - BWD_L2_PREFETCH * 1024 + lane * (128 - 16));
                p = S16::pop_back(w);
                HMMB_BWD_STEP(c * SPC4 + 4 * qq + 1, 1, 1, 0, spp + 64, p)
                p = S16::pop_back(w);
                HMMB_BWD_STEP(c * SPC4 + 4 * qq, 0, 1, 0, spp, p)
                spp -= 2 * 64;
            }
        }
#undef HMMB_BWD_STEP
        if (st.imprecise) {  // sticky hand-over; the host redoes this E-step once (hmmb_bw_iterate)
            raise_flag(flag, bk.first + lane);
            atomicAdd(new_flags, 1);
        }
    }

    // ---- CTA flush: deterministic (fixed-order) reduction into this CTA's partial
    double Xf[16];
    if (BIDIAG) {
#pragma unroll
        for (int q = 0; q < 16; ++q) Xf[q] = 0.0;
        Xf[0] = st.X[0]; Xf[5] = st.X[1]; Xf[10] = st.X[2]; Xf[15] = st.X[3];
        Xf[1] = st.X[4]; Xf[6] = st.X[5]; Xf[11] = st.X[6];
    } else {
#pragma unroll
        for (int q = 0; q < 16; ++q) Xf[q] = st.X[q];
    }
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        double v = Xf[q];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) sRed[warp][4 + q] = v;
    }
    if (lane == 0) {
#pragma unroll
        for (int q = 0; q < 4; ++q) sRed[warp][q] = mypi[q];  // (already summed over the warp's lanes)
    }
    const unsigned seenW = __reduce_or_sync(0xffffffffu, st.seenX);
    if (lane == 0) atomicOr(&sSeen, seenW);
    __syncthreads();
    if (tid < 20) {
        double v = 0.0;
        for (int w = 0; w < nwarps; ++w) v += sRed[w][tid];  // fixed order
        if (tid >= 4) {
            const int q = tid - 4;
            const double aij = __ldg(A + (size_t)cw.word * 16 + q);
            double val = aij > 0.0 ? aij * v : 0.0;  // impossible transitions: ignore whatever piled up
            if (val == 0.0 && aij > 0.0 && ((sSeen >> q) & 1u)) val = tiny_pos();
            v = val;
        }
        part[tid] = v;
    }
    for (int e = tid; e < M * 4; e += nthreads) {
        const int sym = e >> 2, j = e & 3;
        const size_t o = (size_t)(j >> 1) * 2 * M + (size_t)sym * 2 + (j & 1);  // split (j=0,1) / (j=2,3) arrays
        double v = 0.0;
        for (int w = 0; w < nwarps; ++w) v += sCnt[(size_t)w * M * 4 + o];  // the warps' tables, in fixed order
        part[20 + e] = v;
    }
    // ---- this CTA's share of the convergence statistic log_sum_exp_r log P_r (:503)
    __syncthreads();  // sRed is free again
    cta_ll_stat(blks, cw, ll_seq, sRed, part + 20 + (size_t)M * 4);
}

}  // namespace hmmb

// Baum-Welch kernels (E-step forward / backward+accumulate, reduce, M-step, finalize).
//
// Replaces HMM/hmm_training.py:265-541 of the reference.  Two kernel families:
//   * N == 4: bw4_kernels.cuh (one sequence per thread).
//   * generic N <= 32: NP = 4/8/16/32 lanes per sequence (lane = state), alpha/v broadcast
//     through a per-warp shared staging buffer, accumulators via fp64 RED to L2.
#pragma once

#include "bw4_kernels.cuh"

namespace hmmb {

// resident CTAs per SM the generic E-step kernels are compiled for (1 = no register cap)
constexpr int GEN_FWD_MIN_CTAS = 1;
constexpr int GEN_BWD_MIN_CTAS = 1;

// generic path: convert to the canonical symbol width, validate range
template <typename InT, typename SymT>
__global__ void k_convert_obs(const InT *__restrict__ obs, int64_t n, SymT *__restrict__ out, int M,
                              int *__restrict__ bad) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        unsigned long long v = (unsigned long long)obs[i];
        if (v >= (unsigned long long)M) { atomicOr(bad, 1); v = 0; }
        out[i] = (SymT)v;
    }
}

// ---------------------------------------------------------------- generic-N forward
// Each group of NP lanes walks the contiguous range of sequences
// [group * per_group, (group+1) * per_group) of the word-sorted order.
template <int NP, typename SymT>
__global__ void __launch_bounds__(BW_THREADS, GEN_FWD_MIN_CTAS)
k_bw_fwdG(const SymT *__restrict__ obs, const int64_t *__restrict__ off_sorted, const int32_t *__restrict__ len_sorted,
          const int32_t *__restrict__ word_sorted, const int64_t *__restrict__ foff_sorted, int64_t R,
          int64_t per_group, int N, int M, const double *__restrict__ pi, const double *__restrict__ A,
          const double *__restrict__ Bt, double *__restrict__ spill, double *__restrict__ ll_seq,
          const int32_t *__restrict__ active, uint8_t *__restrict__ flag) {
    __shared__ __align__(16) double sStage[BW_WARPS][128];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int GPW = 32 / NP;
    const int j = lane % NP, gbase = lane - j;
    const int64_t group = ((int64_t)blockIdx.x * BW_WARPS + warp) * GPW + lane / NP;
    double acol[NP];
    double pj = 0.0;
    int curw = -1;
    for (int64_t k = 0; k < per_group; ++k) {
        const int64_t r = group * per_group + k;
        int T = 0, w = 0;
        if (r < R) {
            w = word_sorted[r];
            if (active[w] && !flag[r]) T = len_sorted[r];
        }
        const int Tw = warp_max_int(T);
        if (Tw == 0) continue;  // warp-uniform
        if (T > 0 && w != curw) {
            curw = w;
#pragma unroll
            for (int i = 0; i < NP; ++i) acol[i] = (i < N && j < N) ? __ldg(A + ((size_t)w * N + i) * N + j) : 0.0;
            pj = j < N ? __ldg(pi + (size_t)w * N + j) : 0.0;
        }
        const SymT *o = obs + (T > 0 ? off_sorted[r] : 0);
        double *sp = spill + (T > 0 ? foff_sorted[r] * N : 0);
        const double ll = fwdG_run<NP, SymT, true>(T, Tw, N, j, gbase, lane, o, Bt + (size_t)w * M * N, acol, pj, sp,
                                                   sStage[warp]);
        if (T > 0 && j == 0) {
            ll_seq[r] = ll;
            if (ll != ll) raise_flag(flag, r);  // precision guard: hand over to the exact kernel (sticky)
        }
    }
}

// ---------------------------------------------------------------- generic-N backward + accumulate
// Lane i = state i of its group's sequence; holds row i of A and row i of the xi accumulator.
// Accumulator layout per word: [pi N][xi N*N][cnt M*N] (fp64 RED into `accum`).
template <int NP, typename SymT>
__global__ void __launch_bounds__(BW_THREADS, GEN_BWD_MIN_CTAS)
k_bw_bwdG(const SymT *__restrict__ obs, const int64_t *__restrict__ off_sorted, const int32_t *__restrict__ len_sorted,
          const int32_t *__restrict__ word_sorted, const int64_t *__restrict__ foff_sorted, int64_t R,
          int64_t per_group, int N, int M, const double *__restrict__ A, const double *__restrict__ Bt,
          const double *__restrict__ spill, const double *__restrict__ ll_seq, const int32_t *__restrict__ active,
          double *__restrict__ accum, int64_t astride, uint8_t *__restrict__ flag, int32_t *__restrict__ new_flags) {
    __shared__ __align__(16) double sStage[BW_WARPS][128];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int GPW = 32 / NP;
    const int i = lane % NP, gbase = lane - i;
    const unsigned gmask = (NP == 32) ? 0xffffffffu : ((1u << NP) - 1u);
    const int64_t group = ((int64_t)blockIdx.x * BW_WARPS + warp) * GPW + lane / NP;
    double arow[NP], Xrow[NP];
    int curw = -1;
    double *stage = sStage[warp];
    for (int64_t k = 0; k < per_group; ++k) {
        const int64_t r = group * per_group + k;
        int T = 0, w = 0;
        if (r < R) {
            w = word_sorted[r];
            if (active[w] && !flag[r] && ll_seq[r] > neg_inf()) T = len_sorted[r];
        }
        const int Tw = warp_max_int(T);
        if (Tw == 0) continue;
        bool imprecise = false;
        if (T > 0 && w != curw) {
            curw = w;
#pragma unroll
            for (int jj = 0; jj < NP; ++jj) arow[jj] = (i < N && jj < N) ? __ldg(A + ((size_t)w * N + i) * N + jj) : 0.0;
        }
#pragma unroll
        for (int jj = 0; jj < NP; ++jj) Xrow[jj] = 0.0;
        unsigned seenrow = 0u;
        const SymT *o = obs + (T > 0 ? off_sorted[r] : 0);
        const double *sp = spill + (T > 0 ? foff_sorted[r] * N : 0);
        const double *Btw = Bt + (size_t)w * M * N;
        double *acc = accum + (size_t)w * astride;
        double v = 0.0;
        int par = 0;
        stage[par * 32 + lane] = 0.0;
        __syncwarp();
        const unsigned gm = gmask << gbase;
        // software pipeline of the step's loads (as in fwdG_run): alpha-hat and b(o_t) one step ahead, the codeword
        // two steps ahead — the step used to wait for all three in turn (half of the kernel's stall samples)
        unsigned sym_c = 0u, sym_n = 0u;
        double al_c = 0.0, b_c = 0.0;
        {
            const int t0 = Tw - 1;
            if (t0 < T) {
                sym_c = (unsigned)o[t0];
                if (i < N) {
                    al_c = sp[(size_t)t0 * N + i];
                    b_c = __ldg(Btw + (size_t)sym_c * N + i);
                }
            }
            if (t0 >= 1 && t0 - 1 < T) sym_n = (unsigned)o[t0 - 1];
        }
        for (int t = Tw - 1; t >= 0; --t) {
            const bool act = t < T;
            const bool last = (t == T - 1);
            double al_n = 0.0, b_n = 0.0;
            unsigned sym_nn = 0u;
            if (t >= 1 && t - 1 < T && i < N) {
                al_n = sp[(size_t)(t - 1) * N + i];
                b_n = __ldg(Btw + (size_t)sym_n * N + i);
            }
            if (t >= 2 && t - 2 < T) sym_nn = (unsigned)o[t - 2];
            const unsigned vmask = (__ballot_sync(0xffffffffu, v > 0.0) >> gbase) & gmask;
            double q = 0.0;
            if (act) {
                if (last) {
                    q = i < N ? 1.0 : 0.0;  // log beta_{T-1} = 0 (:363)
                } else {
                    const double *sv = stage + par * 32 + gbase;
                    const double2 *sv2 = reinterpret_cast<const double2 *>(sv);  // (gbase is a multiple of NP >= 4)
#pragma unroll
                    for (int jj = 0; jj < NP; jj += 2) {
                        const double2 x = sv2[jj / 2];
                        q = fma(arow[jj], x.x, q);
                        q = fma(arow[jj + 1], x.y, q);
                    }
                    if (q == 0.0 && i < N) {
                        bool reach = false;
                        for (int jj = 0; jj < NP; ++jj) reach |= (arow[jj] > 0.0 && sv[jj] > 0.0);
                        if (reach) q = tiny_pos();
                    }
                }
            }
            // sum_i q_i and sum_i alpha-hat_i q_i in one interleaved shuffle pass: the normaliser sum_i alpha-hat_i (q_i sc)
            // is the second sum times sc exactly (sc is a power of two), and the two reductions no longer wait for
            // each other (their eight dependent DADDs were 15 % of the kernel's stall samples)
            double qs = q, ns = act ? al_c * q : 0.0;
#pragma unroll
            for (int o = NP / 2; o > 0; o >>= 1) {
                qs += __shfl_xor_sync(0xffffffffu, qs, o);
                ns += __shfl_xor_sync(0xffffffffu, ns, o);
            }
            double h = 0.0, al = 0.0, g = 0.0, sc = 1.0;
            if (act) {
                if (!last && qs > 0.0) sc = pow2_rescale_noacc(qs);
                h = q * sc;  // beta-hat_t(i), group sum in [1,2)
                if (h == 0.0 && q > 0.0) h = tiny_pos();  // (sc < 1 must not flush a denormal marker: bw4_kernels.cuh)
                al = al_c;
                g = al * h;
            }
            double norm = ns * sc;
            unsigned sym = 0;
            if (act) {
                double u = al, wscale = 1.0;
                if (!(norm >= TINY_STEP)) {  // group-uniform: see the N = 4 kernel
                    imprecise = true;
                    const double big = 0x1p500;
                    u = al * big;
                    g = u * (h * big);
                    wscale = big;
                    norm = g;
#pragma unroll
                    for (int o = NP / 2; o > 0; o >>= 1) norm += __shfl_xor_sync(gm, norm, o);
                }
                const double r1 = norm > 0.0 ? 1.0 / norm : 0.0;
                g *= r1;  // gamma_t(i) (:389-394)
                if (g == 0.0 && al > 0.0 && h > 0.0) g = tiny_pos();
                sym = sym_c;
                if (!last) {
                    u *= r1;
                    // xi_t(i, j) / a_ij = u_i (v_j sc wscale): sc and wscale are powers of two, so scaling u once instead of
                    // every v_j leaves each product's exact value — and the rounded sum — as it was
                    const double uf = (u * sc) * wscale;
                    const double2 *sv2 = reinterpret_cast<const double2 *>(stage + par * 32 + gbase);
#pragma unroll
                    for (int jj = 0; jj < NP; jj += 2) {
                        const double2 x = sv2[jj / 2];
                        Xrow[jj] = fma(uf, x.x, Xrow[jj]);
                        Xrow[jj + 1] = fma(uf, x.y, Xrow[jj + 1]);
                    }
                    if (al > 0.0) seenrow |= vmask;
                }
                if (i < N && g > 0.0) {
                    atomicAdd(acc + N + N * N + (size_t)sym * N + i, g);  // (:460-500 numerators)
                    if (t == 0) atomicAdd(acc + i, g);                   // (:415-426)
                }
            }
            // v_i = b_i(o_t) beta-hat_t(i) for step t-1
            double b = 0.0;
            if (act) {
                b = b_c;
                v = b * h;
                if (v == 0.0 && b > 0.0 && h > 0.0) v = tiny_pos();
            }
            const unsigned okm = (__ballot_sync(0xffffffffu, v >= TINY_STEP) >> gbase) & gmask;
            if (act && okm == 0u) {
                // every v of the group is tiny: exponent-split products (the scale of v is free)
                double m = 0.0;
                int e = INT_MIN;
                if (b > 0.0 && h > 0.0) frexp_prod(b, h, m, e);
                int E = e;
#pragma unroll
                for (int o2 = NP / 2; o2 > 0; o2 >>= 1) E = max(E, __shfl_xor_sync(gm, E, o2));
                v = 0.0;
                if (e != INT_MIN) {
                    v = ldexp(m, max(e - E, -1200));
                    if (v == 0.0) v = tiny_pos();
                    if (e >= E - 64 && h < SUBNORMAL_LIMIT) imprecise = true;
                }
            }
            par ^= 1;
            stage[par * 32 + lane] = v;
            __syncwarp();
            al_c = al_n; b_c = b_n; sym_c = sym_n; sym_n = sym_nn;
        }
        if (T > 0 && i < N) {
#pragma unroll
            for (int jj = 0; jj < NP; ++jj) {
                if (jj < N) {
                    double val = arow[jj] * Xrow[jj];
                    if (val == 0.0 && arow[jj] > 0.0 && ((seenrow >> jj) & 1u)) val = tiny_pos();
                    if (arow[jj] > 0.0 && val > 0.0) atomicAdd(acc + N + (size_t)i * N + jj, val);
                }
            }
        }
        {
            const unsigned bal = __ballot_sync(0xffffffffu, imprecise && T > 0);
            if (((bal >> gbase) & gmask) != 0u && T > 0 && i == 0) {
                raise_flag(flag, r);
                atomicAdd(new_flags, 1);
            }
            imprecise = false;
        }
        v = 0.0;
    }
}

// ---------------------------------------------------------------- exact log-space E-step (rare)
// One warp per sequence handed over by the precision guard (flag[r] != 0): the reference's
// log-space forward / backward, contributions added to `accum` with fp64 atomics.  Runs after
// the fast forward kernel and before the reduce kernel.  base_sorted[r]: codeword offset of the
// sequence (generic: into the linear stream; N = 4 path: uint4 row of its lane in obs_blk).
template <typename SymT, bool BLOCKED>
__global__ void __launch_bounds__(BW_THREADS)
k_bw_exact(const void *__restrict__ obs, const int64_t *__restrict__ base_sorted, const int32_t *__restrict__ len_sorted,
           const int32_t *__restrict__ word_sorted, int64_t R, int N, int M, const double *__restrict__ pi,
           const double *__restrict__ A, const double *__restrict__ Bt, double *__restrict__ ll_seq,
           const int32_t *__restrict__ active, const uint8_t *__restrict__ flag, double *__restrict__ scratch,
           int64_t scratch_stride, double *__restrict__ accum, int64_t astride, int64_t *__restrict__ n_exact,
           unsigned symmask) {
    if (!any_flag_raised(flag)) return;  // nothing was ever handed over: no scan of the R flags
    const int lane = threadIdx.x & 31;
    const int64_t gw = (int64_t)blockIdx.x * BW_WARPS + (threadIdx.x >> 5);
    const int64_t nw = (int64_t)gridDim.x * BW_WARPS;
    double *sc = scratch + gw * scratch_stride;
    for (int64_t base = gw * 32; base < R; base += nw * 32) {
        const int64_t r = base + lane;
        const bool f = r < R && flag[r] && active[word_sorted[r]];
        unsigned m = __ballot_sync(0xffffffffu, f);
        while (m) {
            const int l = __ffs(m) - 1;
            m &= m - 1;
            const int64_t rr = base + l;
            const int w = word_sorted[rr], T = len_sorted[rr];
            const double *piw = pi + (size_t)w * N, *Aw = A + (size_t)w * N * N, *Btw = Bt + (size_t)w * M * N;
            double logP;
            if (BLOCKED) {
                BlkObs<SymT> o{reinterpret_cast<const uint4 *>(obs) + base_sorted[rr], symmask};
                logP = exact_forward(T, N, lane, o, piw, Aw, Btw, sc);
                __syncwarp();
                if (logP > neg_inf()) exact_backward_accumulate(T, N, lane, o, Aw, Btw, sc, logP, accum + (size_t)w * astride);
            } else {
                LinObs<SymT> o{reinterpret_cast<const SymT *>(obs) + base_sorted[rr]};
                logP = exact_forward(T, N, lane, o, piw, Aw, Btw, sc);
                __syncwarp();
                if (logP > neg_inf()) exact_backward_accumulate(T, N, lane, o, Aw, Btw, sc, logP, accum + (size_t)w * astride);
            }
            if (lane == 0) {
                ll_seq[rr] = logP;
                atomicAdd(reinterpret_cast<unsigned long long *>(n_exact), 1ULL);
            }
            __syncwarp();
        }
    }
}

// ---------------------------------------------------------------- reduce + LL statistics
// One CTA per word.  (N = 4 path) sums the word's CTA partials in fixed order into accum;
// (both) writes the word's sequence count and this rank's (max, sum exp) of the
// per-sequence log-likelihoods, the two halves of log_sum_exp (:503), into
// llstats[rank][w][2].
constexpr int RED_THREADS = 256;
// ---------------------------------------------------------------- thin-state rescue (hmm_device.cuh)
// own-rank slot region -> -inf ("no finite term yet"); the other ranks' regions keep the zeros of the accumulator memset
__global__ void k_bw_rescue_init(double *__restrict__ slots, int64_t n) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x)
        slots[e] = neg_inf();
}
// One warp per sequence of a word that has flagged states: the reference's log-space forward / backward pass, rows of
// the flagged states accumulated in log space.  Same argument conventions as k_bw_exact; every sequence of the word
// takes part (also those the fast kernels or the exact kernel have just handled: the slots replace their rows).
template <typename SymT, bool BLOCKED>
__global__ void __launch_bounds__(BW_THREADS)
k_bw_rescue(const void *__restrict__ obs, const int64_t *__restrict__ base_sorted, const int32_t *__restrict__ len_sorted,
            const int32_t *__restrict__ word_sorted, int64_t R, int N, int M, const double *__restrict__ pi,
            const double *__restrict__ A, const double *__restrict__ Bt, const int32_t *__restrict__ active,
            double *__restrict__ scratch, int64_t scratch_stride, const uint32_t *__restrict__ thinmask,
            const int32_t *__restrict__ slot_of, double *__restrict__ slots, int64_t rstride, unsigned symmask) {
    const int lane = threadIdx.x & 31;
    const int64_t gw = (int64_t)blockIdx.x * BW_WARPS + (threadIdx.x >> 5);
    const int64_t nw = (int64_t)gridDim.x * BW_WARPS;
    double *sc = scratch + gw * scratch_stride;
    for (int64_t base = gw * 32; base < R; base += nw * 32) {
        const int64_t r = base + lane;
        const bool f = r < R && active[word_sorted[r]] && thinmask[word_sorted[r]] != 0u;
        unsigned m = __ballot_sync(0xffffffffu, f);
        while (m) {
            const int l = __ffs(m) - 1;
            m &= m - 1;
            const int64_t rr = base + l;
            const int w = word_sorted[rr], T = len_sorted[rr];
            const double *piw = pi + (size_t)w * N, *Aw = A + (size_t)w * N * N, *Btw = Bt + (size_t)w * M * N;
            if (BLOCKED) {
                BlkObs<SymT> o{reinterpret_cast<const uint4 *>(obs) + base_sorted[rr], symmask};
                const double logP = exact_forward(T, N, lane, o, piw, Aw, Btw, sc);
                __syncwarp();
                if (logP > neg_inf())
                    exact_backward_rescue(T, N, M, lane, o, Aw, Btw, sc, logP, thinmask[w], slot_of + (size_t)w * N, slots, rstride);
            } else {
                LinObs<SymT> o{reinterpret_cast<const SymT *>(obs) + base_sorted[rr]};
                const double logP = exact_forward(T, N, lane, o, piw, Aw, Btw, sc);
                __syncwarp();
                if (logP > neg_inf())
                    exact_backward_rescue(T, N, M, lane, o, Aw, Btw, sc, logP, thinmask[w], slot_of + (size_t)w * N, slots, rstride);
            }
            __syncwarp();
        }
    }
}

constexpr int RED_EX = 32;  // accumulator entries per CTA of k_bw_reduce
constexpr int RED_CY = RED_THREADS / RED_EX;

// grid = (W, ceil(nacc / RED_EX)).  Thread (ex, cy) sums every RED_CY-th CTA partial of entry
// e; the RED_CY partial sums are combined in fixed order, so the result is deterministic.
__global__ void __launch_bounds__(RED_THREADS)
k_bw_reduce(const double *__restrict__ partials, int64_t pstride, const int32_t *__restrict__ cta_begin,
            const double *__restrict__ ll_seq, const int64_t *__restrict__ seq_begin, double *__restrict__ accum,
            int64_t astride, int64_t nacc, double *__restrict__ llstats, int rank, int W,
            const int32_t *__restrict__ active) {
    __shared__ double sM[RED_THREADS / 32], sS[RED_THREADS / 32];
    __shared__ double sPart[RED_CY][RED_EX];
    const int w = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (!active[w]) return;
    double *acc = accum + (size_t)w * astride;
    if (partials) {
        const int ex = tid % RED_EX, cy = tid / RED_EX;
        const int64_t e = (int64_t)blockIdx.y * RED_EX + ex;
        const int c0 = cta_begin[w], c1 = cta_begin[w + 1];
        double s = 0.0;
        if (e < nacc)
            for (int c = c0 + cy; c < c1; c += RED_CY) s += partials[(size_t)c * pstride + e];
        sPart[cy][ex] = s;
        __syncthreads();
        if (cy == 0 && e < nacc) {
            double tot = 0.0;
#pragma unroll
            for (int q = 0; q < RED_CY; ++q) tot += sPart[q][ex];
            acc[e] += tot;  // the exact log-space kernel may already have added flagged sequences
        }
    }
    if (blockIdx.y != 0) return;
    // items of the log-sum-exp: the word's sequences (log P_r, weight 1), or — N = 4 path — the
    // (max, sum) pairs its CTAs left behind their partials
    const int64_t r0 = seq_begin[w], r1 = seq_begin[w + 1];
    const int64_t i0 = partials ? cta_begin[w] : r0, i1 = partials ? cta_begin[w + 1] : r1;
    auto item_m = [&](int64_t i) { return partials ? partials[(size_t)i * pstride + nacc] : ll_seq[i]; };
    auto item_s = [&](int64_t i) { return partials ? partials[(size_t)i * pstride + nacc + 1] : 1.0; };
    double m = neg_inf();
    for (int64_t i = i0 + tid; i < i1; i += RED_THREADS) m = fmax(m, item_m(i));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) sM[warp] = m;
    __syncthreads();
    m = sM[0];
    for (int q = 1; q < RED_THREADS / 32; ++q) m = fmax(m, sM[q]);
    double s = 0.0;
    if (m > neg_inf())
        for (int64_t i = i0 + tid; i < i1; i += RED_THREADS) {
            const double l = item_m(i);
            if (l > neg_inf()) s += item_s(i) * exp(l - m);
        }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) sS[warp] = s;
    __syncthreads();
    if (tid == 0) {
        double tot = 0.0;
        for (int q = 0; q < RED_THREADS / 32; ++q) tot += sS[q];
        acc[nacc] = (double)(r1 - r0);  // sequences of this word on this rank (num_recordings, :268)
        llstats[((size_t)rank * W + w) * 2 + 0] = m;
        llstats[((size_t)rank * W + w) * 2 + 1] = tot;
    }
}

// ---------------------------------------------------------------- M-step
// One CTA per word; replaces hmm_training.py:412-514.
__global__ void __launch_bounds__(RED_THREADS)
k_bw_mstep(const double *__restrict__ accum, int64_t astride, const double *__restrict__ llstats, int world, int W,
           int N, int M, double *__restrict__ pi, double *__restrict__ A, double *__restrict__ Bt,
           const int32_t *__restrict__ active_in, int32_t *__restrict__ active, int32_t *__restrict__ iters,
           double *__restrict__ prev_ll, double *__restrict__ ll_hist, int hist_cap, double eps, int max_iter,
           int32_t *__restrict__ any_active, int32_t *__restrict__ b_has_zero, uint32_t *__restrict__ thinmask,
           int32_t *__restrict__ thin_new, int32_t *__restrict__ redo, int skip_new_thin,
           const int32_t *__restrict__ slot_of, const double *__restrict__ slots, int64_t slot_cap, int64_t rstride,
           double thin_limit) {
    __shared__ double sDen[HMMB_MAX_STATES];
    __shared__ double sPart[RED_THREADS / 32][HMMB_MAX_STATES];
    __shared__ int sSkip;
    const int w = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (!active_in[w]) return;
    const double *acc = accum + (size_t)w * astride;
    const double *xi = acc + N;
    const double *cnt = acc + N + N * N;
    const double nseq = acc[N + N * N + (size_t)M * N];

    // B denominators: sum over all t of gamma_t(j) = column sums of the counts (:462-472)
    if (RED_THREADS % N == 0) {
        // N divides the CTA size: a thread's elements tid, tid + RED_THREADS, ... all belong to state tid % N, so the
        // [M][N] table is read once, coalesced, and the per-thread sums are folded in a fixed order
        __shared__ double sThread[RED_THREADS];
        double s = 0.0;
        for (int e = tid; e < M * N; e += RED_THREADS) s += cnt[e];
        sThread[tid] = s;
        __syncthreads();
        if (tid < N) {
            double d = 0.0;
            for (int q = tid; q < RED_THREADS; q += N) d += sThread[q];
            sDen[tid] = d;
        }
    } else {
        for (int j = 0; j < N; ++j) {
            double s = 0.0;
            for (int k = tid; k < M; k += RED_THREADS) s += cnt[(size_t)k * N + j];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == 0) sPart[warp][j] = s;
        }
        __syncthreads();
        if (tid < N) {
            double s = 0.0;
            for (int q = 0; q < RED_THREADS / 32; ++q) s += sPart[q][tid];
            sDen[tid] = s;
        }
    }
    __syncthreads();
    // Thin states (hmm_device.cuh, "thin-state rescue"): a positive denominator below THIN_LIMIT means the row's sums sit
    // where the linear accumulators run out of range.  The state is flagged (sticky); with skip_new_thin the word leaves
    // this iteration untouched and is marked in `redo`, so that the host can give the state a slot and repeat the
    // iteration for the marked words — otherwise the flag takes effect from the next iteration on.
    __shared__ unsigned sThinBits;
    if (tid == 0) sThinBits = 0u;
    __syncthreads();
    if (tid < N) {
        double denA = 0.0;
        for (int j = 0; j < N; ++j) denA += xi[tid * N + j];
        if ((denA > 0.0 && denA < thin_limit) || (sDen[tid] > 0.0 && sDen[tid] < thin_limit)) atomicOr(&sThinBits, 1u << tid);
    }
    __syncthreads();
    if (tid == 0) {
        const unsigned have = thinmask[w];
        const unsigned fresh = sThinBits & ~have;
        if (fresh) {
            thinmask[w] = have | fresh;
            atomicAdd(thin_new, __popc(fresh));
        }
        sSkip = (fresh && skip_new_thin) ? 1 : 0;
        if (redo) redo[w] = sSkip;
    }
    __syncthreads();
    if (sSkip) return;
    // B (:474-497): no finite term -> 1e-20 floor; empty denominator -> row stays -inf (0)
    for (int e = tid; e < M * N; e += RED_THREADS) {
        const int j = e % N;
        const double den = sDen[j];
        const double c = cnt[e];
        double b = 0.0;
        if (den > 0.0) {
            if (c > 0.0) {
                b = c / den;
                if (b == 0.0) b = tiny_pos();
            } else {
                b = 1e-20;
            }
        }
        Bt[(size_t)w * M * N + e] = b;
    }
    // A (:429-457): a_ij = sum xi / sum_{t<T-1} gamma(i); the denominator equals the row sum of xi
    if (tid < N) {
        const int i = tid;
        double den = 0.0;
        for (int j = 0; j < N; ++j) den += xi[i * N + j];
        for (int j = 0; j < N; ++j) {
            double x = xi[i * N + j];
            double v = 0.0;
            if (den > 0.0 && x > 0.0) {
                v = x / den;
                if (v == 0.0) v = tiny_pos();
            }
            A[((size_t)w * N + i) * N + j] = v;
        }
        // pi (:415-426): sum_r gamma_0^r(i) / num_recordings
        const double p = acc[i];
        double pv = 0.0;
        if (p > 0.0) {
            pv = p / nseq;
            if (pv == 0.0) pv = tiny_pos();
        }
        pi[(size_t)w * N + i] = pv;
    }
    // Flagged states with a slot: rows of A and B from the log-space sums (the ranks' slots combined by log_sum_exp in
    // rank order), as the reference forms them (:429-457, :460-497)
    {
        const unsigned tm = thinmask[w];
        if (tm != 0u && slot_cap > 0) {
            __syncthreads();  // the plain rows above are written
            for (int i = 0; i < N; ++i) {
                if (!((tm >> i) & 1u)) continue;
                const int sl = slot_of[(size_t)w * N + i];
                if (sl < 0) continue;
                auto entry = [&](int e) {  // log sum over ranks of entry e of the state's slot
                    double mx = neg_inf();
                    for (int r = 0; r < world; ++r) mx = fmax(mx, slots[((size_t)r * slot_cap + sl) * rstride + e]);
                    if (!(mx > neg_inf())) return neg_inf();
                    double sm = 0.0;
                    for (int r = 0; r < world; ++r) {
                        const double v = slots[((size_t)r * slot_cap + sl) * rstride + e];
                        if (v > neg_inf()) sm += exp(v - mx);
                    }
                    return mx + log(sm);
                };
                // block-wide log_sum_exp of entries [e0, e0 + n)
                auto block_lse = [&](int e0, int n) {
                    double mx = neg_inf();
                    for (int e = tid; e < n; e += RED_THREADS) mx = fmax(mx, entry(e0 + e));
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
                    if (lane == 0) sPart[warp][0] = mx;
                    __syncthreads();
                    mx = sPart[0][0];
                    for (int q = 1; q < RED_THREADS / 32; ++q) mx = fmax(mx, sPart[q][0]);
                    __syncthreads();
                    double sm = 0.0;
                    if (mx > neg_inf())
                        for (int e = tid; e < n; e += RED_THREADS) {
                            const double v = entry(e0 + e);
                            if (v > neg_inf()) sm += exp(v - mx);
                        }
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) sm += __shfl_xor_sync(0xffffffffu, sm, o);
                    if (lane == 0) sPart[warp][0] = sm;
                    __syncthreads();
                    double tot = 0.0;
                    for (int q = 0; q < RED_THREADS / 32; ++q) tot += sPart[q][0];
                    __syncthreads();
                    return (mx > neg_inf()) ? mx + log(tot) : neg_inf();
                };
                const double denA = block_lse(0, N), denB = block_lse(N, M);
                if (tid < N) {
                    const double x = entry(tid);
                    double v = 0.0;
                    if (denA > neg_inf() && x > neg_inf()) {
                        v = exp(x - denA);
                        if (v == 0.0) v = tiny_pos();
                    }
                    A[((size_t)w * N + i) * N + tid] = v;
                }
                for (int k = tid; k < M; k += RED_THREADS) {
                    const double c = entry(N + k);
                    double b = 0.0;
                    if (denB > neg_inf()) {
                        if (c > neg_inf()) {
                            b = exp(c - denB);
                            if (b == 0.0) b = tiny_pos();
                        } else {
                            b = 1e-20;
                        }
                    }
                    Bt[(size_t)w * M * N + (size_t)k * N + i] = b;
                }
            }
            __syncthreads();
        }
    }
    if (tid == 0) {
        // a state that was never visited keeps an all-zero (log: -inf) emission row (:471)
        int z = 0;
        for (int j = 0; j < N; ++j) z |= (sDen[j] > 0.0) ? 0 : 1;
        b_has_zero[w] = z;
        // convergence statistic: log_sum_exp over all sequences of the word (:503-508)
        double mx = neg_inf();
        for (int r = 0; r < world; ++r) mx = fmax(mx, llstats[((size_t)r * W + w) * 2]);
        double cur = neg_inf();
        if (mx > neg_inf()) {
            double s = 0.0;
            for (int r = 0; r < world; ++r) {
                const double m = llstats[((size_t)r * W + w) * 2];
                if (m > neg_inf()) s += llstats[((size_t)r * W + w) * 2 + 1] * exp(m - mx);
            }
            cur = mx + log(s);
        }
        const double prev = prev_ll[w];
        const double diff = (prev > neg_inf()) ? fabs(cur - prev) : pos_inf();
        int it = iters[w];
        if (it < hist_cap) ll_hist[(size_t)w * hist_cap + it] = cur;
        ++it;
        iters[w] = it;
        prev_ll[w] = cur;
        const int act = (diff >= eps && it < max_iter) ? 1 : 0;  // loop condition (:346)
        active[w] = act;
        if (act) atomicOr(any_active, 1);
    }
}

// ---------------------------------------------------------------- exit normalisation (:524-539)
// finalize: safe_exp of the log parameters (:524-526) then the row normalisations.  A value
// held at the smallest denormal is our marker for "finite log value below the double range"
// (the reference's exp underflows to exactly 0.0 there), so it is flushed to 0 on exit.
__device__ __forceinline__ double exit_value(double v, int finalize) {
    return (finalize && v == tiny_pos()) ? 0.0 : v;
}

__global__ void __launch_bounds__(RED_THREADS)
k_bw_finalize(const double *__restrict__ pi, const double *__restrict__ A, const double *__restrict__ Bt, int N, int M,
              int finalize, double *__restrict__ pi_out, double *__restrict__ A_out, double *__restrict__ B_out) {
    __shared__ double sDen[HMMB_MAX_STATES];
    __shared__ double sPart[RED_THREADS / 32][HMMB_MAX_STATES];
    const int w = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const double *Bw = Bt + (size_t)w * M * N;
    for (int j = 0; j < N; ++j) {
        double s = 0.0;
        for (int k = tid; k < M; k += RED_THREADS) s += exit_value(Bw[(size_t)k * N + j], finalize);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) sPart[warp][j] = s;
    }
    __syncthreads();
    if (tid < N) {
        double s = 0.0;
        for (int q = 0; q < RED_THREADS / 32; ++q) s += sPart[q][tid];
        sDen[tid] = s;
    }
    __syncthreads();
    for (int e = tid; e < M * N; e += RED_THREADS) {
        const int k = e / N, j = e - k * N;
        double b = exit_value(Bw[e], finalize);
        if (finalize && sDen[j] > 0.0) b = b / sDen[j];
        B_out[((size_t)w * N + j) * M + k] = b;
    }
    if (tid < N) {
        const int i = tid;
        double rs = 0.0;
        for (int j = 0; j < N; ++j) rs += exit_value(A[((size_t)w * N + i) * N + j], finalize);
        for (int j = 0; j < N; ++j) {
            double v = exit_value(A[((size_t)w * N + i) * N + j], finalize);
            if (finalize && rs > 0.0) v = v / rs;
            A_out[((size_t)w * N + i) * N + j] = v;
        }
        double ps = 0.0;
        for (int j = 0; j < N; ++j) ps += exit_value(pi[(size_t)w * N + j], finalize);
        double p = exit_value(pi[(size_t)w * N + i], finalize);
        if (finalize) p = p / ps;  // no zero guard in the reference either (:529)
        pi_out[(size_t)w * N + i] = p;
    }
}

}  // namespace hmmb

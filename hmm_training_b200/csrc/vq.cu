// VQ encode and LBG (binary-split k-means) codebook kernels for sm_100a.
//
// Replaces (reference paths relative to the reference root):
//   get_observations ........ HMM/hmm_training.py:82-120
//   createCodeVector ........ CodeVector/codevector_functions.py:442-531
//   new_epsilon_centroids ... CodeVector/codevector_functions.py:383-411
//   new_adjust_centroids .... CodeVector/codevector_functions.py:414-439
//
// Arithmetic contract (bit-exact indices): the reference computes
// np.linalg.norm(x[1:] - c[1:]) = sqrt(dot(d, d)); with the image's numpy/OpenBLAS the
// 12-term dot is the sequential FMA chain acc = fma(d_i, d_i, acc), i = 1..12.  The kernel
// evaluates exactly that chain in fp64 (__dsub_rn + __fma_rn, no re-association), compares
// with strict '<' on the square root (only evaluated when the squared distance improves),
// so the lowest index wins ties exactly as at hmm_training.py:112.
//
// Roofline: 12 DADD + 12 DFMA per (frame, centroid) pair -> FP64-pipe bound
// (AI ~ 85 flop/B); HBM traffic is 104 B in + 4 B out per frame.
#include <algorithm>
#include <cstdlib>

#include "common.cuh"

namespace hmmb {

constexpr int VQ_THREADS = 256;
constexpr int VQ_MIN_CTAS = 3;  // resident CTAs per SM the assign kernel is compiled for: 80 registers, no spills; encode call 0.212 (2) / 0.199 (3) / 0.206 ms (4)
constexpr int VQ_TILE = 512;  // centroids per shared-memory tile: 512 * 12 * 8 B = 48 KB
constexpr int VQ_D = 12;      // dims 1..12 take part in the distance
constexpr int ACC_W = 14;     // per-centroid accumulator row: 13 sums + count
constexpr int VQ_PRIV_K = 32; // up to this many centroids every warp keeps a private accumulator table

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---------------------------------------------------------------- accumulate helper (LBG pass)
// Adds one frame (all 13 dims) to row `best` of the per-centroid accumulators (13 sums + count).
// priv: warp-private tables, the 32 lanes park frame and key in shared memory and lanes 0..13 (one per
// column) walk them — no atomics; otherwise fp64 atomics on the CTA's shared table or the global one.
struct AccCtx {
    double *acc;   // shared [K][14] (or the global table)
    double *wAcc;  // warp-private [K][14]
    double *wX;    // warp-private [32][13]
    int *wKey;     // warp-private [32]
    bool priv;
    int K;
};
__device__ __forceinline__ void lbg_accumulate(const AccCtx &ac, int lane, bool valid, int best, const double (&x)[13]) {
    if (ac.priv) {
#pragma unroll
        for (int d = 0; d < 13; ++d) ac.wX[lane * 13 + d] = x[d];
        ac.wKey[lane] = valid ? best : -1;
        __syncwarp();
        if (lane < ACC_W) {
            for (int l = 0; l < 32; ++l) {
                const int k = ac.wKey[l];
                if (k >= 0) ac.wAcc[k * ACC_W + lane] += (lane < 13) ? ac.wX[l * 13 + lane] : 1.0;
            }
        }
        __syncwarp();
    } else if (ac.K <= 16) {
        // few centroids: every lane hits the same handful of rows, so reduce per key across the warp with
        // shuffles and issue one atomic per (key, dim)
        unsigned remaining = __ballot_sync(0xffffffffu, valid);
        while (remaining) {
            const int leader = __ffs(remaining) - 1;
            const int key = __shfl_sync(0xffffffffu, best, leader);
            const bool mine = valid && best == key;
            const unsigned m = __ballot_sync(0xffffffffu, mine);
            remaining &= ~m;
#pragma unroll
            for (int d = 0; d < 13; ++d) {
                const double v = warp_sum(mine ? x[d] : 0.0);
                if (lane == 0) atomicAdd(ac.acc + key * ACC_W + d, v);
            }
            if (lane == 0) atomicAdd(ac.acc + key * ACC_W + 13, (double)__popc(m));
        }
    } else if (valid) {
#pragma unroll
        for (int d = 0; d < 13; ++d) atomicAdd(ac.acc + best * ACC_W + d, x[d]);
        atomicAdd(ac.acc + best * ACC_W + 13, 1.0);
    }
}

// The reference's distance of one (frame, centroid) pair, squared: the sequential FMA chain (see the header).
__device__ __forceinline__ double exact_d2(const double (&x)[13], const double *__restrict__ c) {
    double a = 0.0;
#pragma unroll
    for (int d = 0; d < VQ_D; ++d) {
        const double v = __dsub_rn(x[1 + d], c[d]);
        a = __fma_rn(v, v, a);
    }
    return a;
}

// ---------------------------------------------------------------- prefilter + exact winner
// Two-stage nearest centroid with bit-exact results (north_star (3): the ||x||^2 - 2 x.c + ||c||^2 form):
//
//  1. PREFILTER, fp32 CUDA cores: s_k = ||c_k||^2 - 2 x.c_k over dims 1..12 (||x||^2 is common to every k) as one
//     12-term FFMA chain per pair, running smallest / second smallest value and the index of the smallest.
//     With u = 2^-24: x-hat = fl32(x), c-hat = fl32(c), n-hat = fl32(||c||^2 in fp64), chain of 12 fused ops:
//         |s-hat_k - s_k| <= 14.1 u (||c_k||^2 + 2 ||x|| ||c_k||) <= 28.2 u (||x||^2 + ||c_k||^2) = 1.68e-6 (...)
//     so with tol = 2.05e-6 (||x||^2 + max_k ||c_k||^2) (+ an absolute 1e-37 for fp32 underflow) every k whose
//     true squared distance is within rounding of the smallest has s-hat_k <= m1 + 2 tol.
//  2. If the second smallest value is beyond m1 + 2 tol the argmin is unique and no other centroid can tie or win
//     under the reference's arithmetic (its fp64 chain and the sqrt move a value by < 1e-14 relative): the winner
//     is k1, and its reference distance sqrt(fma chain) is evaluated once, exactly.
//  3. Otherwise (two candidates within ~1e-6 of ||x||^2 + ||c||^2 of each other: twins, duplicates, non-finite
//     input) the frame goes to a work list and k_vq_exact_list gives it the reference's full scan: every
//     centroid in index order, strict '<' on the square root (hmm_training.py:107-114).  That kernel also
//     reports the contract's near-ties, (d2 - d1) / d1 < 1e-12.
// Indices are therefore those of the exact scan for EVERY frame; only the amount of fp64 work differs.
constexpr int VQ_FPT = 2;            // frames per thread in the prefilter (each shared-memory centroid row feeds both)
static_assert(VQ_FPT == 2, "the prefilter packs its two frames into one f32x2 chain");
__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(unsigned long long v, float &lo, float &hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long ffma2(unsigned long long a, unsigned long long b, unsigned long long c) {
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
constexpr double VQ_TOL_REL = 2.05e-6;
constexpr double VQ_TOL_ABS = 1e-37;

// MODE 0: encode only.  MODE 1: LBG pass = encode + per-centroid 13-dim sums, counts and the sum of winning
// distances, reduced in shared memory and flushed once per CTA.
// Shared memory: [tile][12] fp64 centroids, [tile][12] fp32 centroids, [tile] fp32 ||c||^2, accumulators.
template <int MODE>
__global__ void __launch_bounds__(VQ_THREADS, VQ_MIN_CTAS)
k_vq_assign(const double *__restrict__ X, int64_t F, const double *__restrict__ C, int K,
            int32_t *__restrict__ idx_out, double *__restrict__ dist_out, double *__restrict__ accum,
            int smem_accum, const int *__restrict__ skip, int32_t *__restrict__ worklist, int *__restrict__ n_work) {
    // a Lloyd pass queued speculatively after the generation has converged (k_lbg_check) is a no-op
    if (skip && *skip) return;
    extern __shared__ double smem[];
    const int TK = min(K, VQ_TILE);
    double *sC = smem;                                            // [tile][12] fp64
    float *sCf = reinterpret_cast<float *>(sC + (size_t)TK * VQ_D);  // [tile][12] fp32
    float *sNf = sCf + (size_t)((TK + 3) & ~3) * VQ_D;            // [tile] fp32 squared norms (both padded to 4 rows)
    double *sAcc = reinterpret_cast<double *>(sNf + ((TK + 3) & ~3)) ;  // [K][14] (MODE 1, if smem_accum)
    __shared__ double sRed[VQ_THREADS / 32];
    __shared__ double sCmax2;

    const int tid = threadIdx.x, lane = tid & 31;
    const bool priv = MODE == 1 && smem_accum == 2;
    AccCtx ac;
    ac.priv = priv;
    ac.K = K;
    ac.acc = smem_accum ? sAcc : accum;
    ac.wAcc = sAcc + (size_t)(tid >> 5) * K * ACC_W;                                       // [K][14] per warp
    ac.wX = sAcc + (size_t)(VQ_THREADS / 32) * K * ACC_W + (size_t)(tid >> 5) * 32 * 13;   // [32][13] per warp
    ac.wKey = reinterpret_cast<int *>(sAcc + (size_t)(VQ_THREADS / 32) * (K * ACC_W + 32 * 13)) + (tid >> 5) * 32;
    if (MODE == 1 && smem_accum) {
        const int n = priv ? (VQ_THREADS / 32) * K * ACC_W : K * ACC_W;
        for (int e = tid; e < n; e += VQ_THREADS) sAcc[e] = 0.0;
    }
    // max_k ||c_k||^2 over ALL centroids (the tolerance of every tile uses it)
    {
        double m = 0.0;
        for (int k = tid; k < K; k += VQ_THREADS) {
            double n2 = 0.0;
#pragma unroll
            for (int d = 0; d < VQ_D; ++d) { const double c = __ldg(C + (size_t)k * 13 + 1 + d); n2 = fma(c, c, n2); }
            m = fmax(m, n2);  // (NaN-free maximum: a NaN norm makes the fp32 value NaN, which lands on the work list)
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (lane == 0) sRed[tid >> 5] = m;
        __syncthreads();
        if (tid == 0) {
            double mm = 0.0;
            for (int w = 0; w < VQ_THREADS / 32; ++w) mm = fmax(mm, sRed[w]);
            sCmax2 = mm;
        }
        __syncthreads();
    }
    const double cmax2 = sCmax2;
    double dist_local = 0.0;
    const int ntiles = (K + VQ_TILE - 1) / VQ_TILE;
    constexpr int FPB = VQ_THREADS * VQ_FPT;  // frames per CTA batch
    const int64_t nbatch = (F + FPB - 1) / FPB;

    for (int64_t batch = blockIdx.x; batch < nbatch; batch += gridDim.x) {
        // ---- stage 1: fp32 prefilter, VQ_FPT frames per thread (frame u of the thread: batch * FPB + u * 256 + tid)
        float xm2[VQ_FPT][VQ_D];  // -2 x-hat
        float m1[VQ_FPT], m2[VQ_FPT];
        int k1[VQ_FPT];
        double tol2[VQ_FPT];      // 2 tol
#pragma unroll
        for (int u = 0; u < VQ_FPT; ++u) {
            const int64_t f = batch * FPB + (int64_t)u * VQ_THREADS + tid;
            double xx = 0.0;
#pragma unroll
            for (int d = 0; d < VQ_D; ++d) {
                const double xd = f < F ? __ldg(X + f * 13 + 1 + d) : 0.0;
                xx = fma(xd, xd, xx);
                xm2[u][d] = (float)(-2.0 * xd);
            }
            tol2[u] = 2.0 * (VQ_TOL_REL * (xx + cmax2) + VQ_TOL_ABS);
            m1[u] = m2[u] = __int_as_float(0x7f800000);
            k1[u] = 0;
        }
        unsigned long long x2[VQ_D];  // (-2 x-hat of frame 0, of frame 1) per dimension
#pragma unroll
        for (int d = 0; d < VQ_D; ++d) x2[d] = pack2(xm2[0][d], xm2[1][d]);
        for (int tile = 0; tile < ntiles; ++tile) {
            const int k0 = tile * VQ_TILE;
            const int kt = min(VQ_TILE, K - k0);
            if (ntiles > 1 || batch == blockIdx.x) {
                __syncthreads();
                for (int e = tid; e < ((kt + 3) & ~3) * VQ_D; e += VQ_THREADS) {
                    const int k = e / VQ_D, d = e - k * VQ_D;
                    if (k < kt) {
                        const double c = __ldg(C + (size_t)(k0 + k) * 13 + 1 + d);
                        sC[e] = c;
                        sCf[e] = (float)c;
                    } else {
                        sCf[e] = 0.f;  // padding row of the last group of four
                    }
                }
                for (int k = tid; k < ((kt + 3) & ~3); k += VQ_THREADS) {
                    double n2 = 0.0;
                    if (k < kt) {
#pragma unroll
                        for (int d = 0; d < VQ_D; ++d) { const double c = __ldg(C + (size_t)(k0 + k) * 13 + 1 + d); n2 = fma(c, c, n2); }
                    }
                    sNf[k] = k < kt ? (float)n2 : __int_as_float(0x7f800000);  // padding rows never win
                }
                __syncthreads();
            }
            const float4 *c4 = reinterpret_cast<const float4 *>(sCf);
            const float4 *n4 = reinterpret_cast<const float4 *>(sNf);
            const int kt4 = (kt + 3) & ~3;
#pragma unroll 1
            for (int k = 0; k < kt4; k += 4) {
                const float4 nn = n4[k >> 2];
                const float nv[4] = {nn.x, nn.y, nn.z, nn.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    // padding rows (k + j >= kt) are zeros starting from +inf: never the smallest or second smallest
                    const float4 ca = c4[(k + j) * 3], cb = c4[(k + j) * 3 + 1], cc = c4[(k + j) * 3 + 2];
                    // Both frames of the thread in one packed chain: FFMA2 with the centroid coordinate as the
                    // broadcast scalar operand (sm_100a: `FFMA2 Rd, Ra.F32x2, Rb.F32, Rc.F32x2`), 12 instructions
                    // instead of 24 for the pair; each half is the same IEEE fused multiply-add as fmaf.
                    const float cv[VQ_D] = {ca.x, ca.y, ca.z, ca.w, cb.x, cb.y, cb.z, cb.w, cc.x, cc.y, cc.z, cc.w};
                    unsigned long long s2 = pack2(nv[j], nv[j]);
#pragma unroll
                    for (int d = 0; d < VQ_D; ++d) s2 = ffma2(x2[d], pack2(cv[d], cv[d]), s2);
                    float sv[VQ_FPT];
                    unpack2(s2, sv[0], sv[1]);
#pragma unroll
                    for (int u = 0; u < VQ_FPT; ++u) {
                        const float s = sv[u];
                        const float hi = fmaxf(s, m1[u]);
                        k1[u] = (s < m1[u]) ? (k0 + k + j) : k1[u];
                        m1[u] = fminf(s, m1[u]);
                        m2[u] = fminf(m2[u], hi);
                    }
                }
            }
        }
        // ---- stage 2: the winner's exact distance, or the work list
#pragma unroll
        for (int u = 0; u < VQ_FPT; ++u) {
            const int64_t f = batch * FPB + (int64_t)u * VQ_THREADS + tid;
            const bool valid = f < F;
            double x[13];
#pragma unroll
            for (int d = 0; d < 13; ++d) x[d] = valid ? __ldg(X + f * 13 + d) : 0.0;
            // unique <=> second smallest beyond m1 + 2 tol (false for NaN / inf anywhere)
            const bool unique = (double)m2[u] > (double)m1[u] + tol2[u];
            bool done = valid && unique;
            int best = k1[u];
            double best_s = 0.0;
            if (done) {
                const double *c = (ntiles == 1) ? sC + (size_t)best * VQ_D : nullptr;
                double a;
                if (c) {
                    a = exact_d2(x, c);
                } else {  // several tiles: the winner's row may not be resident
                    double cr[VQ_D];
#pragma unroll
                    for (int d = 0; d < VQ_D; ++d) cr[d] = __ldg(C + (size_t)best * 13 + 1 + d);
                    a = exact_d2(x, cr);
                }
                best_s = sqrt(a);
                if (idx_out) idx_out[f] = best;
                if (dist_out) dist_out[f] = best_s;
                if (MODE == 1) dist_local += best_s;
            } else if (valid) {
                worklist[atomicAdd(n_work, 1)] = (int32_t)f;
            }
            if (MODE == 1) lbg_accumulate(ac, lane, done, best, x);
        }
    }
    if (MODE == 1) {
        double v = warp_sum(dist_local);
        if (lane == 0) sRed[tid >> 5] = v;
        __syncthreads();
        if (tid == 0) {
            double s = 0.0;
            for (int w = 0; w < VQ_THREADS / 32; ++w) s += sRed[w];
            atomicAdd(accum + (size_t)K * ACC_W, s);
        }
        if (priv) {
            __syncthreads();
            for (int e = tid; e < K * ACC_W; e += VQ_THREADS) {
                double a = 0.0;
#pragma unroll
                for (int w = 0; w < VQ_THREADS / 32; ++w) a += sAcc[(size_t)w * K * ACC_W + e];
                if (a != 0.0) atomicAdd(accum + e, a);
            }
        } else if (smem_accum) {
            for (int e = tid; e < K * ACC_W; e += VQ_THREADS) {
                double a = sAcc[e];
                if (a != 0.0) atomicAdd(accum + e, a);
            }
        }
    }
}

// The reference's full scan for the frames on the work list (one thread per listed frame): every centroid in index
// order, strict '<' on sqrt(fma chain) — hmm_training.py:107-114, codevector_functions.py:493-503.  MODE 1 adds the
// frame to the global accumulators.  near (nullable): frames whose two smallest distances differ by less than
// 1e-12 relative — the contract's "near-ties ... listed" (their index may differ on another CPU / BLAS).
constexpr double VQ_NEAR_TIE_REL = 1e-12;
template <int MODE>
__global__ void __launch_bounds__(128)
k_vq_exact_list(const double *__restrict__ X, const double *__restrict__ C, int K, const int32_t *__restrict__ worklist,
                const int *__restrict__ n_work, int32_t *__restrict__ idx_out, double *__restrict__ dist_out,
                double *__restrict__ accum, const int *__restrict__ skip, int32_t *__restrict__ near, int near_cap,
                int *__restrict__ n_near, int32_t near_base) {
    if (skip && *skip) return;
    const int n = *n_work;
    // One WARP per listed frame (a single thread's scan of K centroids is a serial chain of ~40 K dependent DP
    // instructions: with a few hundred frames on the list that latency, 0.1 ms, was a third of the whole encode call).
    // Lane l scans centroids l, l + 32, ... in index order with the reference's rule and keeps (smallest, its index,
    // second smallest); the lanes' triples are merged with "smaller distance, then lower index" — the first centroid
    // that attains the minimum in index order, and the second order statistic of all K distances, as the serial scan.
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int i = warp; i < n; i += nwarps) {
        const int64_t f = worklist[i];
        double x[13];
#pragma unroll
        for (int d = 0; d < 13; ++d) x[d] = __ldg(X + f * 13 + d);
        double best_s = pos_inf(), second_s = pos_inf();
        int best = lane;
        for (int k = lane; k < K; k += 32) {
            double c[VQ_D];
#pragma unroll
            for (int d = 0; d < VQ_D; ++d) c[d] = __ldg(C + (size_t)k * 13 + 1 + d);
            const double sk = sqrt(exact_d2(x, c));
            if (sk < best_s) {
                second_s = best_s;
                best_s = sk; best = k;
            } else if (sk < second_s) {
                second_s = sk;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ob = __shfl_xor_sync(0xffffffffu, best_s, o), o2 = __shfl_xor_sync(0xffffffffu, second_s, o);
            const int oi = __shfl_xor_sync(0xffffffffu, best, o);
            const bool other_wins = ob < best_s || (ob == best_s && oi < best);
            if (other_wins) {
                second_s = fmin(best_s, o2);
                best_s = ob; best = oi;
            } else {
                second_s = fmin(ob, second_s);
            }
        }
        if (best >= K) best = 0;  // (K < 32 and nothing comparable: the serial scan's initial index)
        if (lane == 0) {
            if (idx_out) idx_out[f] = best;
            if (dist_out) dist_out[f] = best_s;
            if (n_near && (second_s - best_s) <= VQ_NEAR_TIE_REL * best_s) {  // (also exact ties: twins, duplicates)
                const int p = atomicAdd(n_near, 1);
                if (p < near_cap) near[p] = (int32_t)f + near_base;
            }
        }
        if (MODE == 1) {
            if (lane < 13) atomicAdd(accum + best * ACC_W + lane, __ldg(X + f * 13 + lane));
            if (lane == 13) atomicAdd(accum + best * ACC_W + 13, 1.0);
            if (lane == 14) atomicAdd(accum + (size_t)K * ACC_W, best_s);
        }
    }
}

// new_adjust_centroids: mean of the assigned frames (all 13 dims), zeros(13) if empty.
// Convergence state of one LBG generation, kept on the device so that Lloyd passes can be queued
// several at a time without a host round trip per pass (codevector_functions.py:475-476, :485, :509-510).
struct LbgState {
    double prev, gd;
    int it, done;
};
__global__ void k_lbg_reset(LbgState *st) {
    st->prev = 0.0;
    st->gd = 0.0;
    st->it = 0;
    st->done = 0;
}
// after the centroid update of a pass: count it, compare the summed distance with the previous pass
__global__ void k_lbg_check(const double *__restrict__ gdp, LbgState *st, double eps, double *__restrict__ hist, int hist_n) {
    if (st->done) return;
    const double gd = *gdp;
    const double diff = fabs(st->prev - gd);
    if (hist && st->it < hist_n) hist[st->it] = gd;
    st->it += 1;
    st->prev = gd;
    st->gd = gd;
    if (!(diff > eps)) st->done = 1;  // loop condition `while diff > eps` (:485)
}

__global__ void k_lbg_update(const double *__restrict__ accum, int K, double *__restrict__ C,
                             const LbgState *__restrict__ st) {
    if (st && st->done) return;  // (the flag only changes in k_lbg_check, a separate launch)
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= K * 13) return;
    int k = e / 13, d = e - k * 13;
    double n = accum[k * ACC_W + 13];
    C[e] = n > 0.0 ? accum[k * ACC_W + d] / n : 0.0;
}

// new_epsilon_centroids: centroid i -> 2i = c * 1.001, 2i+1 = c * 0.999 (all 13 dims).
__global__ void k_lbg_split(const double *__restrict__ C, int K, double *__restrict__ C2) {
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= K * 13) return;
    int k = e / 13, d = e - k * 13;
    double v = C[e];
    C2[(size_t)(2 * k) * 13 + d] = v * 1.001;
    C2[(size_t)(2 * k + 1) * 13 + d] = v * 0.999;
}

// smem_accum: 0 = accumulate straight into global memory, 1 = one shared [K][14] table per CTA,
// 2 = one private table per warp (K <= VQ_PRIV_K)
static size_t vq_smem_bytes(int K, int mode, int *smem_accum) {
    const size_t tk = (size_t)std::min(K, VQ_TILE), tk4 = (tk + 3) & ~size_t(3);
    size_t tile = tk * VQ_D * sizeof(double) + tk4 * VQ_D * sizeof(float) + tk4 * sizeof(float);
    size_t acc = (size_t)K * ACC_W * sizeof(double);
    *smem_accum = 0;
    if (mode == 1 && K <= VQ_PRIV_K) {
        *smem_accum = 2;
        const size_t warps = VQ_THREADS / 32;
        return tile + warps * (acc + 32 * 13 * sizeof(double)) + warps * 32 * sizeof(int);
    }
    if (mode == 1 && tile + acc <= 200 * 1024) {
        *smem_accum = 1;
        return tile + acc;
    }
    return tile;
}

// Device scratch of the two-stage search: the work list of ambiguous frames (capacity F) and its counter, and
// optionally the near-tie list.  n_work must be zero before the launch.
struct VqScratch {
    int32_t *worklist = nullptr;
    int *n_work = nullptr;
    int32_t *near = nullptr;
    int near_cap = 0;
    int *n_near = nullptr;
    int32_t near_base = 0;  // added to the frame ids written to `near` (chunked encode)
};

static int vq_launch(int mode, const double *dX, int64_t F, const double *dC, int K, int32_t *d_idx,
                     double *d_dist, double *d_accum, const VqScratch &sc, const int *d_skip = nullptr) {
    Ctx &c = ctx();
    int smem_accum = 0;
    size_t smem = vq_smem_bytes(K, mode, &smem_accum);
    constexpr int FPB = VQ_THREADS * VQ_FPT;
    int64_t nbatch = (F + FPB - 1) / FPB;
    if (nbatch == 0) return HMMB_OK;
    // persistent-style grid: a multiple of the SM count, each CTA strides over frame batches
    int per_sm = smem > 100 * 1024 ? 1 : (smem * VQ_MIN_CTAS <= 200 * 1024 ? VQ_MIN_CTAS : 2);
    int64_t grid = (int64_t)c.sm_count * per_sm * (mode == 1 ? 1 : 2);
    if (grid > nbatch) grid = nbatch;
    const unsigned egrid = (unsigned)std::min<int64_t>((int64_t)c.sm_count * 4, (F + 127) / 128);
    if (mode == 0) {
        HMMB_CUDA(cudaFuncSetAttribute(k_vq_assign<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        HMMB_LAUNCH("vq_encode", k_vq_assign<0>, (unsigned)grid, VQ_THREADS, smem, dX, F, dC, K, d_idx, d_dist,
                    d_accum, smem_accum, d_skip, sc.worklist, sc.n_work);
        HMMB_LAUNCH("vq_exact", k_vq_exact_list<0>, egrid, 128, 0, dX, dC, K, sc.worklist, sc.n_work, d_idx, d_dist, d_accum,
                    d_skip, sc.near, sc.near_cap, sc.n_near, sc.near_base);
    } else {
        HMMB_CUDA(cudaFuncSetAttribute(k_vq_assign<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        HMMB_LAUNCH("lbg_assign", k_vq_assign<1>, (unsigned)grid, VQ_THREADS, smem, dX, F, dC, K, d_idx, d_dist,
                    d_accum, smem_accum, d_skip, sc.worklist, sc.n_work);
        HMMB_LAUNCH("lbg_exact", k_vq_exact_list<1>, egrid, 128, 0, dX, dC, K, sc.worklist, sc.n_work, d_idx, d_dist, d_accum,
                    d_skip, sc.near, sc.near_cap, sc.n_near, sc.near_base);
    }
    return HMMB_OK;
}

struct DevBuf {
    void *p = nullptr;
    ~DevBuf() { dev_free(p); }
    template <typename T> T *as() { return reinterpret_cast<T *>(p); }
};

}  // namespace hmmb

using namespace hmmb;

extern "C" {

// Scratch of one encode call: work list (capacity F frames), its counter and the near-tie counter in one block.
struct EncodeScratch {
    DevBuf list, cnt, near;
    VqScratch sc;
    int init(int64_t F, int64_t near_cap) {
        Ctx &c = ctx();
        HMMB_TRY(dev_alloc(&list.p, (size_t)std::max<int64_t>(F, 1) * sizeof(int32_t)));
        HMMB_TRY(dev_alloc(&cnt.p, 2 * sizeof(int)));
        HMMB_CUDA(cudaMemsetAsync(cnt.p, 0, 2 * sizeof(int), c.stream));
        sc.worklist = list.as<int32_t>();
        sc.n_work = cnt.as<int>();
        sc.n_near = cnt.as<int>() + 1;
        if (near_cap > 0) {
            HMMB_TRY(dev_alloc(&near.p, (size_t)near_cap * sizeof(int32_t)));
            sc.near = near.as<int32_t>();
            sc.near_cap = (int)near_cap;
        }
        return HMMB_OK;
    }
};

static int check_frame_count(const char *who, int64_t F) {
    if (F > (int64_t)INT32_MAX) {  // frame ids on the work list are 32-bit (2^31 frames = 223 GB of fp64 MFCCs)
        set_error("%s: F=%lld exceeds 2^31-1 frames per call; encode in slices", who, (long long)F);
        return HMMB_ERR_ARG;
    }
    return HMMB_OK;
}

int hmmb_vq_encode_dev(const double *dX, int64_t F, const double *dC, int K, int32_t *d_idx, double *d_dist) {
    HMMB_TRY(require_init());
    if (F < 0 || K <= 0 || !dC || (F > 0 && (!dX || !d_idx))) {
        set_error("hmmb_vq_encode_dev: bad arguments (F=%lld, K=%d)", (long long)F, K);
        return HMMB_ERR_ARG;
    }
    HMMB_TRY(check_frame_count("hmmb_vq_encode_dev", F));
    if (F == 0) return HMMB_OK;
    EncodeScratch es;
    HMMB_TRY(es.init(F, 0));
    return vq_launch(0, dX, F, dC, K, d_idx, d_dist, nullptr, es.sc);  // (scratch blocks: stream-ordered reuse)
}

int hmmb_vq_encode(const double *X, int64_t F, const double *C, int K, int32_t *idx_out) {
    return hmmb_vq_encode_ex(X, F, C, K, idx_out, nullptr, 0, nullptr);
}

int hmmb_vq_encode_ex(const double *X, int64_t F, const double *C, int K, int32_t *idx_out, int32_t *near_out,
                      int64_t near_cap, int64_t *n_near_out) {
    HMMB_TRY(require_init());
    if (F < 0 || K <= 0 || !C || (F > 0 && (!X || !idx_out)) || near_cap < 0 || (near_cap > 0 && !near_out)) {
        set_error("hmmb_vq_encode: bad arguments (F=%lld, K=%d)", (long long)F, K);
        return HMMB_ERR_ARG;
    }
    HMMB_TRY(check_frame_count("hmmb_vq_encode", F));
    if (n_near_out) *n_near_out = 0;
    if (F == 0) return HMMB_OK;
    Ctx &c = ctx();
    const bool want_near = n_near_out != nullptr;
    near_cap = std::min<int64_t>(near_cap, F);
    DevBuf dX, dC, dI;
    HMMB_TRY(dev_alloc(&dX.p, (size_t)F * 13 * sizeof(double)));
    HMMB_TRY(dev_alloc(&dC.p, (size_t)K * 13 * sizeof(double)));
    HMMB_TRY(dev_alloc(&dI.p, (size_t)F * sizeof(int32_t)));
    EncodeScratch es;
    HMMB_TRY(es.init(F, want_near ? std::max<int64_t>(near_cap, 1) : 0));
    if (want_near && near_cap == 0) es.sc.near_cap = 0;  // count only
    HMMB_CUDA(cudaMemcpyAsync(dC.p, C, (size_t)K * 13 * sizeof(double), cudaMemcpyHostToDevice, c.stream));
    // Frames in pinned host memory go up in chunks on the copy stream and every chunk is encoded as soon
    // as it has landed: the kernel hides behind the PCIe transfer (0.5 G frames/s).
    cudaPointerAttributes attr;
    const bool pinned = cudaPointerGetAttributes(&attr, X) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    (void)cudaGetLastError();
    const int64_t chunk = 1 << 17;  // 131 072 frames = 13.6 MB
    if (pinned && F >= 2 * chunk) {
        cudaEvent_t fence = event_get();  // recycled device blocks may still be in use on the compute stream
        HMMB_CUDA(cudaEventRecord(fence, c.stream));
        HMMB_CUDA(cudaStreamWaitEvent(c.copy_stream, fence, 0));
        event_put(fence);
        for (int64_t f0 = 0; f0 < F; f0 += chunk) {
            const int64_t n = std::min<int64_t>(chunk, F - f0);
            HMMB_CUDA(cudaMemcpyAsync(dX.as<double>() + f0 * 13, X + f0 * 13, (size_t)n * 13 * sizeof(double),
                                      cudaMemcpyHostToDevice, c.copy_stream));
            cudaEvent_t landed = event_get();
            HMMB_CUDA(cudaEventRecord(landed, c.copy_stream));
            HMMB_CUDA(cudaStreamWaitEvent(c.stream, landed, 0));
            event_put(landed);
            if (f0 > 0) HMMB_CUDA(cudaMemsetAsync(es.sc.n_work, 0, sizeof(int), c.stream));  // the list is per chunk
            es.sc.near_base = (int32_t)f0;
            HMMB_TRY(vq_launch(0, dX.as<double>() + f0 * 13, n, dC.as<double>(), K, dI.as<int32_t>() + f0, nullptr, nullptr, es.sc));
        }
    } else {
        HMMB_TRY(h2d_big(dX.p, X, (size_t)F * 13 * sizeof(double), c.stream));  // pageable frames: pinned bounce buffers
        HMMB_TRY(vq_launch(0, dX.as<double>(), F, dC.as<double>(), K, dI.as<int32_t>(), nullptr, nullptr, es.sc));
    }
    HMMB_TRY(d2h_big(idx_out, dI.p, (size_t)F * sizeof(int32_t), c.stream));
    if (want_near) {
        int n_near = 0;
        HMMB_CUDA(cudaMemcpyAsync(&n_near, es.sc.n_near, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
        HMMB_CUDA(cudaStreamSynchronize(c.stream));
        *n_near_out = n_near;
        const int64_t ncopy = std::min<int64_t>(n_near, near_cap);
        if (ncopy > 0) {
            HMMB_CUDA(cudaMemcpy(near_out, es.sc.near, (size_t)ncopy * sizeof(int32_t), cudaMemcpyDeviceToHost));
            std::sort(near_out, near_out + ncopy);
        }
    }
    return HMMB_OK;
}

int hmmb_lbg_fit(const double *X, int64_t F, int x_on_device, int K, int max_iter, double eps, double *C_out,
                 double *gens_out, int32_t *assign_out, int32_t *iters_per_gen, double *gdist_out,
                 hmmb_allreduce_fn allreduce, void *user) {
    return hmmb_lbg_fit_ex(X, F, x_on_device, K, max_iter, eps, C_out, gens_out, assign_out, iters_per_gen, gdist_out,
                           nullptr, allreduce, user);
}

int hmmb_lbg_fit_ex(const double *X, int64_t F, int x_on_device, int K, int max_iter, double eps, double *C_out,
                    double *gens_out, int32_t *assign_out, int32_t *iters_per_gen, double *gdist_out,
                    double *gdist_hist, hmmb_allreduce_fn allreduce, void *user) {
    HMMB_TRY(require_init());
    HMMB_TRY(check_frame_count("hmmb_lbg_fit", F));
    if (F <= 0 && !allreduce) {
        set_error("No raw data provided");  // codevector_functions.py:445-446
        return HMMB_ERR_EMPTY;
    }
    if (K <= 0 || !C_out || !gens_out || (F > 0 && !X) || F < 0) {
        set_error("hmmb_lbg_fit: bad arguments (F=%lld, K=%d)", (long long)F, K);
        return HMMB_ERR_ARG;
    }
    Ctx &c = ctx();
    int n_gen = 0;
    while ((2 << n_gen) <= K) ++n_gen;  // floor(log2 K)
    const int Kmax = 1 << (n_gen > 0 ? n_gen : 1);
    DevBuf dXb, dCa, dCb, dI, dAcc;
    const double *dX = X;
    if (!x_on_device && F > 0) {
        HMMB_TRY(dev_alloc(&dXb.p, (size_t)F * 13 * sizeof(double)));
        HMMB_TRY(h2d_big(dXb.p, X, (size_t)F * 13 * sizeof(double), c.stream));
        dX = dXb.as<double>();
    }
    HMMB_TRY(dev_alloc(&dCa.p, (size_t)Kmax * 13 * sizeof(double)));
    HMMB_TRY(dev_alloc(&dCb.p, (size_t)Kmax * 13 * sizeof(double)));
    HMMB_TRY(dev_alloc(&dI.p, (size_t)(F > 0 ? F : 1) * sizeof(int32_t)));
    // accumulators of one pass: [K][14] sums and counts, the summed distance, and (in the last slot, so that one
    // memset clears everything) the counter of the ambiguous-frame work list
    const size_t acc_n = (size_t)Kmax * ACC_W + 2;
    HMMB_TRY(dev_alloc(&dAcc.p, acc_n * sizeof(double)));
    DevBuf dList, dHist;
    HMMB_TRY(dev_alloc(&dList.p, (size_t)(F > 0 ? F : 1) * sizeof(int32_t)));
    const int hist_n = std::max(max_iter, 1);
    HMMB_TRY(dev_alloc(&dHist.p, (size_t)hist_n * sizeof(double)));
    VqScratch sc;
    sc.worklist = dList.as<int32_t>();
    double *cur = dCa.as<double>(), *nxt = dCb.as<double>();
    double *acc = dAcc.as<double>();
    int32_t *d_idx = dI.as<int32_t>();
    std::vector<double> hC((size_t)Kmax * 13);

    // C0 = mean of all frames (:458-459): one accumulate pass against a single zero centroid
    HMMB_CUDA(cudaMemsetAsync(cur, 0, 13 * sizeof(double), c.stream));
    HMMB_CUDA(cudaMemsetAsync(acc, 0, acc_n * sizeof(double), c.stream));
    sc.n_work = reinterpret_cast<int *>(acc + ACC_W + 1);
    HMMB_TRY(vq_launch(1, dX, F, cur, 1, d_idx, nullptr, acc, sc));
    if (allreduce) {
        int rc = allreduce(acc, ACC_W + 1, user);
        if (rc != 0) { set_error("allreduce hook failed (%d)", rc); return HMMB_ERR_CUDA; }
    }
    HMMB_LAUNCH("lbg_update", k_lbg_update, 1, 32, 0, acc, 1, cur, (const LbgState *)nullptr);
    size_t gpos = 0;
    HMMB_CUDA(cudaMemcpyAsync(gens_out, cur, 13 * sizeof(double), cudaMemcpyDeviceToHost, c.stream));
    gpos += 13;
    HMMB_LAUNCH("lbg_split", k_lbg_split, 1, 32, 0, cur, 1, nxt);  // :469
    { double *t = cur; cur = nxt; nxt = t; }
    int Kg = 2;
    HMMB_CUDA(cudaMemsetAsync(d_idx, 0, (size_t)(F > 0 ? F : 1) * sizeof(int32_t), c.stream));

    DevBuf dState;
    HMMB_TRY(dev_alloc(&dState.p, sizeof(LbgState)));
    LbgState *st = dState.as<LbgState>();
    constexpr int LBG_QUEUE = 8;  // Lloyd passes queued per host round trip
    for (int g = 1; g <= n_gen; ++g) {
        // Lloyd loop of the generation (:475-514).  The convergence test runs on the device (k_lbg_check); passes
        // are queued LBG_QUEUE at a time and the ones behind the converged pass return at once, so the host
        // synchronises once per LBG_QUEUE passes instead of once per pass.
        HMMB_LAUNCH("lbg_update", k_lbg_reset, 1, 1, 0, st);
        double *buf[2] = {cur, nxt};
        LbgState hs{0.0, 0.0, 0, 0};
        int enq = 0;
        while (!hs.done && enq < max_iter) {
            const int n = std::min(LBG_QUEUE, max_iter - enq);
            for (int i = 0; i < n; ++i) {
                const int p = enq + i;
                HMMB_CUDA(cudaMemsetAsync(acc, 0, ((size_t)Kg * ACC_W + 2) * sizeof(double), c.stream));
                sc.n_work = reinterpret_cast<int *>(acc + (size_t)Kg * ACC_W + 1);
                HMMB_TRY(vq_launch(1, dX, F, buf[p & 1], Kg, d_idx, nullptr, acc, sc, &st->done));
                if (allreduce) {
                    int rc = allreduce(acc, (int64_t)Kg * ACC_W + 1, user);
                    if (rc != 0) { set_error("allreduce hook failed (%d)", rc); return HMMB_ERR_CUDA; }
                }
                HMMB_LAUNCH("lbg_update", k_lbg_update, (Kg * 13 + 127) / 128, 128, 0, acc, Kg, buf[(p + 1) & 1], st);
                HMMB_LAUNCH("lbg_update", k_lbg_check, 1, 1, 0, acc + (size_t)Kg * ACC_W, st, eps, dHist.as<double>(), hist_n);
            }
            enq += n;
            HMMB_CUDA(cudaMemcpyAsync(&hs, st, sizeof(LbgState), cudaMemcpyDeviceToHost, c.stream));
            HMMB_CUDA(cudaStreamSynchronize(c.stream));
        }
        const int it = hs.it;
        const double gd = hs.gd;
        cur = buf[it & 1];  // written by the last pass that ran
        nxt = buf[(it + 1) & 1];
        if (iters_per_gen) iters_per_gen[g - 1] = it;
        if (gdist_out) gdist_out[g - 1] = gd;
        if (gdist_hist)  // summed distance of every pass of this generation (the reference prints dist / diff from it, :512-516)
            HMMB_CUDA(cudaMemcpyAsync(gdist_hist + (size_t)(g - 1) * hist_n, dHist.p, (size_t)std::min(it, hist_n) * sizeof(double),
                                      cudaMemcpyDeviceToHost, c.stream));
        HMMB_CUDA(cudaMemcpyAsync(gens_out + gpos, cur, (size_t)Kg * 13 * sizeof(double), cudaMemcpyDeviceToHost, c.stream));
        gpos += (size_t)Kg * 13;
        if (g < n_gen) {  // :520-521
            HMMB_LAUNCH("lbg_split", k_lbg_split, (Kg * 13 + 127) / 128, 128, 0, cur, Kg, nxt);
            { double *t = cur; cur = nxt; nxt = t; }
            Kg *= 2;
        }
    }
    HMMB_CUDA(cudaMemcpyAsync(C_out, cur, (size_t)Kg * 13 * sizeof(double), cudaMemcpyDeviceToHost, c.stream));
    if (assign_out && F > 0)
        HMMB_CUDA(cudaMemcpyAsync(assign_out, d_idx, (size_t)F * sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
    HMMB_CUDA(cudaStreamSynchronize(c.stream));
    return Kg;
}

}  // extern "C"

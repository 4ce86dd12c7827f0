/* hmmb200 — C ABI of the B200-native HMM hot path (libhmmb200.so).
 *
 * The reference (DemianMArin/HMM_Training) is pure Python and has no FFI of its own; its
 * hot path sits behind plain Python functions.  Each entry point below names the reference
 * function (file:line, relative to the reference root) whose arithmetic it replaces; the
 * Python shims in hmm_training_b200/ keep the reference's signatures and call these through
 * ctypes (INTEGRATION.md shows the stub a reference maintainer would add).
 *
 * Conventions
 *   - plain pointers and sizes only; host buffers are caller-owned unless a parameter is
 *     documented as a device pointer; matrices are C-contiguous fp64.
 *   - every function returns HMMB_OK (0) or a negative HMMB_ERR_* code;
 *     hmmb_last_error() returns a thread-local message for the last failure.
 *   - one context per process per GPU (hmmb_init); the library is NOT thread-safe.
 *   - all kernels are launched on one stream (hmmb_set_stream / hmmb_get_stream).
 *   - there is no CPU fallback: without a CUDA device every compute call fails with
 *     HMMB_ERR_CUDA.
 */
#ifndef HMMB200_H
#define HMMB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HMMB_OK 0
#define HMMB_ERR_CUDA (-1)        /* CUDA runtime failure / no device                        */
#define HMMB_ERR_ARG (-2)         /* invalid argument                                        */
#define HMMB_ERR_OOM (-3)         /* device or host allocation failed                        */
#define HMMB_ERR_EMPTY (-4)       /* empty input: T == 0 sequence (reference: IndexError,    */
                                  /* hmm_training.py:376) or no frames (ValueError,          */
                                  /* codevector_functions.py:445)                            */
#define HMMB_ERR_RANGE (-5)       /* codeword >= M (reference: IndexError on log_b_matrix)   */
#define HMMB_ERR_UNSUPPORTED (-6) /* outside documented limits (N > 32, M > 65536, ...)      */

#define HMMB_DIM 13               /* MFCC vector length (codevector_classes.py:211)          */
#define HMMB_MAX_STATES 32

/* ------------------------------------------------------------------ context */
int hmmb_init(int device);                 /* select device, create stream + workspace      */
int hmmb_shutdown(void);                   /* free workspace, destroy stream                */
const char *hmmb_last_error(void);
const char *hmmb_version(void);
int hmmb_device_info(int *sm_count, int *cc_major, int *cc_minor, int64_t *global_mem_bytes);
/* NULL restores the library's own stream.  The stream is used from the next call on and starts behind the work
 * queued on the previous one; the library's own stream is non-blocking (not ordered with the legacy default
 * stream), so without hmmb_set_stream a caller synchronises around calls that take device pointers. */
int hmmb_set_stream(void *cuda_stream);
void *hmmb_get_stream(void);
int hmmb_synchronize(void);
/* pinned host memory for callers that want async H2D/D2H */
void *hmmb_host_alloc(int64_t bytes);
int hmmb_host_free(void *p);
/* kernels launched by this library since hmmb_init (the "gpu_launches" claim in bench.py) */
int64_t hmmb_launch_count(void);
/* elapsed ms of the last call's named phase, measured with CUDA events on the stream:
 * "vq_encode", "lbg_assign", "bw_forward", "bw_backward", "bw_reduce", "bw_mstep", "score";
 * negative if the phase has not run.  Accumulated over launches; *launches gets the count. */
double hmmb_phase_ms(const char *phase, int64_t *launches);
int hmmb_phase_reset(void);
int hmmb_set_profiling(int enabled);       /* event timing around every kernel (default off) */
/* Measured FMA throughput of this GPU in TFLOP/s (what = 0: fp64 DFMA, 1: fp32 FFMA; ~1 ms of dependent-chain-free
 * FMAs, best of three): the denominator bench.py uses for the compute-bound kernels' roofline fractions.      */
int hmmb_peak_probe(int what, double *tflops);

/* Sum-allreduce hook for the multi-GPU path: called between the E-step and the M-step
 * (and once per Lloyd pass) with a DEVICE buffer of n doubles that must be summed in place
 * across ranks, ordered after all work already queued on hmmb_get_stream().  The Python
 * shim implements it with torch.distributed.all_reduce over NCCL.  NULL = single GPU. */
typedef int (*hmmb_allreduce_fn)(void *dev_buf, int64_t n_doubles, void *user);

/* Built-in NCCL communicator for callers without their own collective (SURVEY.md section 8b).  libnccl.so.2 is
 * opened with dlopen at the first call (inside a PyTorch process that is the copy torch has already mapped).
 * Rank 0 obtains the 128-byte id with hmmb_comm_unique_id and distributes it out of band; every rank then calls
 * hmmb_comm_init (collective, after hmmb_init on its GPU).  hmmb_comm_allreduce is an hmmb_allreduce_fn: pass it
 * to hmmb_bw_set_dist / hmmb_lbg_fit (hmmb_bw_set_dist also falls back to it when its hook argument is NULL). */
int hmmb_comm_unique_id(void *id_out, int id_bytes /* >= 128 */);
int hmmb_comm_init(int rank, int world, const void *nccl_id);
int hmmb_comm_allreduce(void *dev_buf, int64_t n_doubles, void *user);
int hmmb_comm_rank(int *rank, int *world);   /* world = 1 while no communicator exists */
int hmmb_comm_destroy(void);

/* ------------------------------------------------------------------ VQ encode
 * Replaces get_observations, HMM/hmm_training.py:82-120: per frame argmin_k of
 * sqrt(sum_{d=1..12} (x_d - c_kd)^2), strict '<' (lowest index wins ties); dimension 0
 * (energy) is ignored (:100,:107).  X [F,13], C [K,13] fp64 -> idx_out [F] int32.        */
int hmmb_vq_encode(const double *X, int64_t F, const double *C, int K, int32_t *idx_out);
/* same on device-resident buffers; d_dist (nullable) receives the winning distance.  dX / dC are read and
 * d_idx / d_dist written on hmmb_get_stream(): the inputs must be complete on that stream when the call runs, and
 * the call returns WITHOUT waiting — the outputs are ready for work queued on that stream afterwards, or after
 * hmmb_synchronize().                                                                     */
int hmmb_vq_encode_dev(const double *dX, int64_t F, const double *dC, int K, int32_t *d_idx,
                       double *d_dist);
/* hmmb_vq_encode + the near-tie report of the parity contract (BASELINE.json north_star: "codeword indices
 * bit-exact (near-ties within a stated epsilon documented)"): near_out [near_cap] (nullable if near_cap == 0)
 * receives, in ascending order, the frames whose two smallest distances differ by less than 1e-12 relative
 * ((d2 - d1) / d1 < 1e-12, exact ties included) — the frames whose index, decided by hmm_training.py:112's
 * strict '<', could differ under another BLAS's summation order; *n_near_out = how many there are (it may
 * exceed near_cap).  At most 2^31-1 frames per call.                                                        */
int hmmb_vq_encode_ex(const double *X, int64_t F, const double *C, int K, int32_t *idx_out, int32_t *near_out,
                      int64_t near_cap, int64_t *n_near_out);

/* ------------------------------------------------------------------ LBG codebook
 * Replaces createCodeVector, CodeVector/codevector_functions.py:442-531 (with
 * new_epsilon_centroids :383-411 and new_adjust_centroids :414-439).  K =
 * centroids_quantity; n_gen = floor(log2 K); the call returns Kout = 2^max(n_gen,1), the
 * number of rows written to C_out, or a negative error.
 *   C_out [Kout,13]; gens_out [(1 + 2 + ... + 2^n_gen), 13] = [C0] + converged centroids of
 *   each generation (:466,:517); assign_out [F] = frame.parent_centroid_id (:502);
 *   iters_per_gen [n_gen]; gdist_out [n_gen] (nullable) last sum of min distances (:503).
 * x_on_device != 0: X is a device pointer (frames already resident in HBM), read on hmmb_get_stream() (it must be
 * complete on that stream); the call returns with every output written to the host and X no longer in use.
 * Multi-GPU: every rank passes its shard of frames and the same hook; sums/counts/distance
 * are all-reduced once per Lloyd pass (SURVEY.md §8e).                                      */
int hmmb_lbg_fit(const double *X, int64_t F, int x_on_device, int K, int max_iter, double eps,
                 double *C_out, double *gens_out, int32_t *assign_out, int32_t *iters_per_gen,
                 double *gdist_out, hmmb_allreduce_fn allreduce, void *user);
/* same + gdist_hist [n_gen, max(max_iter, 1)] (nullable): the summed distance after EVERY Lloyd pass of every
 * generation (row g holds iters_per_gen[g] values) — what the reference prints as dist / diff every tenth pass
 * and as the final diff of a generation (codevector_functions.py:509-516).                                   */
int hmmb_lbg_fit_ex(const double *X, int64_t F, int x_on_device, int K, int max_iter, double eps,
                    double *C_out, double *gens_out, int32_t *assign_out, int32_t *iters_per_gen,
                    double *gdist_out, double *gdist_hist, hmmb_allreduce_fn allreduce, void *user);

/* ------------------------------------------------------------------ Baum-Welch
 * Replaces hmm_training, HMM/hmm_training.py:265-541, batched over W word models:
 * E-step (calculate_log_alpha :122-160, calculate_log_beta :163-199, gamma/xi :380-410),
 * M-step (:412-500, 1e-20 floor :497), convergence statistic (:503-508), exit
 * normalisation (:524-539).  The reference trains words one at a time; here every word
 * keeps its own iteration counter and stops exactly where the reference would.
 *
 * Sequences are ragged: obs holds all codewords back to back (idx_bytes = 1, 2, 4 or 8 per
 * codeword, unsigned), sequence r is obs[offsets[r] .. offsets[r+1]) and belongs to word
 * word_of_seq[r] in [0, W).  Limits: 1 <= N <= 32, 1 <= M <= 65536, T >= 1.            */
typedef struct hmmb_bw hmmb_bw_t;

/* obs_on_device != 0: obs is a device pointer (offsets and word_of_seq stay on the host) and sequence r starts at
 * codeword offsets[r] of it; it is read on hmmb_get_stream() (it must be complete on that stream) and no longer in
 * use when the create returns: the trainer keeps its own copies.  A codeword >= M fails the create
 * (HMMB_ERR_RANGE).                                                                      */
int hmmb_bw_create(hmmb_bw_t **out, const void *obs, int idx_bytes, int obs_on_device,
                   const int64_t *offsets, const int32_t *word_of_seq, int64_t R, int W, int N,
                   int M);
/* flags for hmmb_bw_create_ex.  HMMB_BW_PIPELINE_UPLOAD: when the codewords come from PINNED host
 * memory in (word, length-descending) order and either N = 4, or N = 8 / 16 with initial parameters
 * whose A are all upper-bidiagonal (left-to-right kernels), the call returns while they are still
 * being uploaded (copy stream, a few chunks) and the first hmmb_bw_iterate runs its E-step stage
 * by stage behind the upload (repack -> forward -> backward of the blocks that have landed).
 * The caller must keep `obs` — and pi0 / A0 / B0 where they are pinned too: those then go up
 * straight from the caller's memory — valid and unchanged until that first hmmb_bw_iterate has
 * returned; a codeword >= M is then reported by that call (HMMB_ERR_RANGE) instead of by the create.
 * Results are those of the unpipelined path (the CTA partition is finer, so sums may differ in
 * the last bits).                                                                            */
#define HMMB_BW_PIPELINE_UPLOAD 1
/* pi0 / A0 / B0 (all three or none): initial parameters as for hmmb_bw_set_params, uploaded by the
 * create itself ahead of the bulk of the codewords (a later hmmb_bw_set_params is still allowed). */
int hmmb_bw_create_ex(hmmb_bw_t **out, const void *obs, int idx_bytes, int obs_on_device,
                      const int64_t *offsets, const int32_t *word_of_seq, int64_t R, int W, int N,
                      int M, int flags, const double *pi0, const double *A0, const double *B0);
int hmmb_bw_destroy(hmmb_bw_t *h);
/* pi0 [W,N], A0 [W,N,N], B0 [W,N,M] linear-space initial parameters; resets iteration state */
int hmmb_bw_set_params(hmmb_bw_t *h, const double *pi0, const double *A0, const double *B0);
int hmmb_bw_set_dist(hmmb_bw_t *h, int rank, int world, hmmb_allreduce_fn allreduce, void *user);
/* Communication / compute overlap for the left-to-right kernels (N = 8 / 16), whose accumulator buffer is large
 * (133 MB at 1000 words x 16 states x 1024 codewords).  groups > 1: the backward pass runs word group by word
 * group and the hook is called once per group with that group's slice of the buffer, then once for the
 * log-likelihood statistics, then once as hook(NULL, 0, user) = "join".  A hook that runs each collective on a
 * side stream (ordered behind the work queued on hmmb_get_stream() at the time of the call) and makes
 * hmmb_get_stream() wait for that side stream in the join call overlaps the transfer of group g with the
 * backward pass of group g+1; a plain synchronous hook must simply ignore the n == 0 call.  With groups > 1 a
 * backward-pass hand-over takes effect from the next iteration (as with sync_each == 0).  Default 1.      */
int hmmb_bw_set_overlap(hmmb_bw_t *h, int groups);
/* run up to n_iter EM iterations (stops early when every word has converged: diff < eps or
 * max_iter reached, :346).  sync_each != 0 checks the device-side "any word active" flag
 * after each iteration; 0 queues all n_iter iterations without a host sync.             */
int hmmb_bw_iterate(hmmb_bw_t *h, int n_iter, double eps, int max_iter, int sync_each);
/* finalize != 0 applies the exit normalisation (:529-539).  Outputs: pi [W,N], A [W,N,N],
 * B [W,N,M]; ll_hist [W,max_iter_cap] per-iteration convergence statistic (NaN-padded),
 * iters [W]; any output pointer may be NULL.                                              */
int hmmb_bw_get_params(hmmb_bw_t *h, int finalize, double *pi, double *A, double *B);
int hmmb_bw_get_history(hmmb_bw_t *h, double *ll_hist, int hist_cap, int32_t *iters);
/* per-sequence log P(O|lambda) of the last E-step, in input order [R] (:376-377)         */
int hmmb_bw_get_seq_ll(hmmb_bw_t *h, double *ll_seq);
int64_t hmmb_bw_total_frames(hmmb_bw_t *h);
/* which E-step kernels the parameters set by hmmb_bw_set_params select: "n4_left_to_right" /
 * "n4_dense" (one sequence per thread, N = 4), "left_to_right" (one sequence per thread,
 * N = 8 / 16 with upper-bidiagonal A) or "generic" (lanes per state, N <= 32)            */
const char *hmmb_bw_kernel_family(hmmb_bw_t *h);
/* precision-guard counters since hmmb_bw_set_params: sequence passes recomputed by the exact
 * log-space kernel, and sequences handed over by the backward pass (each costs one E-step
 * redo when hmmb_bw_iterate runs with sync_each != 0; with sync_each == 0 they are only
 * counted and take effect from the next iteration).                                        */
int hmmb_bw_diagnostics(hmmb_bw_t *h, int64_t *exact_sequence_passes, int64_t *backward_handovers);
/* Number of (word, state) pairs whose A / B rows are currently formed from log-space sums because their posterior
 * mass fell below 2^-200 ("thin states": the linear accumulators cannot hold sums below ~1e-308, the reference's
 * log sums can — HMM/hmm_training.py:429-497).  With sync_each the iteration that finds such a state is repeated
 * for its word; without, the state is rescued from the next hmmb_bw_iterate call on.                             */
int hmmb_bw_thin_states(hmmb_bw_t *h, int64_t *n_states);

/* one-shot convenience: create + set_params + iterate + get + destroy (host buffers)      */
int hmmb_bw_fit(const void *obs, int idx_bytes, const int64_t *offsets, const int32_t *word_of_seq,
                int64_t R, int W, int N, int M, const double *pi0, const double *A0,
                const double *B0, double eps, int max_iter, double *pi, double *A, double *B,
                double *ll_hist, int32_t *iters);

/* ------------------------------------------------------------------ recognition
 * Replaces calculate_log_likelihood, HMM/hmm_testing.py:49-104, and the argmax loop of
 * test_hmm, :139-161: ll_out [U,W] = log P(O_u | model_w) from LINEAR pi/A/B (zeros are
 * structural -inf, :67-69); argmax_out [U] = first model with the strictly largest score,
 * -1 ("unknown", :161) if every score is -inf.  ll_out / argmax_out may be NULL.
 * obs_on_device != 0: obs is a device pointer; offsets stay on the host.  It is read on hmmb_get_stream() (it must
 * be complete on that stream); the call returns with ll_out / argmax_out written and obs no longer in use.     */
int hmmb_score(const void *obs, int idx_bytes, int obs_on_device, const int64_t *offsets, int64_t U,
               int W, int N, int M, const double *pi, const double *A, const double *B,
               double *ll_out, int32_t *argmax_out);

/* ------------------------------------------------------------------ Viterbi decoding
 * An extension: the reference has no Viterbi.  The most likely state path of every utterance under its own model
 * (utterance u against model model_of_utt[u], host array, values in [0, W)) and that path's log-probability, from
 * LINEAR pi [W,N], A [W,N,N], B [W,N,M] (entries <= 0 or NaN are structural zeros, log = -inf):
 *     delta_0(j) = log pi_j + log b_j(o_0)
 *     delta_t(j) = (max_i (delta_t-1(i) + log a_ij)) + log b_j(o_t)
 *     psi_t(j)   = the smallest i that reaches the max;  the last state is the smallest j that reaches
 *                  max_j delta_T-1(j), and score_out[u] is that max.
 * An utterance that is impossible under its model (score -inf) gets -1 for every frame.
 * path_out [offsets[U] - offsets[0]] int8, input frame order: frame t of utterance u is at
 * path_out[offsets[u] - offsets[0] + t].  path_out == NULL decodes the scores only (no backpointers are stored);
 * score_out is then bit-identical to the call with a path.  score_out may be NULL.
 * obs / idx_bytes / obs_on_device / offsets as for hmmb_score.  1 <= N <= 32, 1 <= M <= 65536, W <= 65535.
 * Errors: HMMB_ERR_RANGE (codeword >= M), HMMB_ERR_EMPTY (empty utterance), HMMB_ERR_ARG (model index outside
 * [0, W)), HMMB_ERR_UNSUPPORTED (N or M out of range), HMMB_ERR_OOM (the backpointers do not fit: 1 byte per frame
 * at N = 4 and left-to-right N = 8, 2 at left-to-right N = 16, N bytes otherwise).                                */
int hmmb_viterbi(const void *obs, int idx_bytes, int obs_on_device, const int64_t *offsets, int64_t U,
                 const int32_t *model_of_utt, int W, int N, int M, const double *pi, const double *A,
                 const double *B, double *score_out, int8_t *path_out);

/* ------------------------------------------------------------------ MFCC front-end
 * Replaces RawDataMFCC.calculate_mfcc, CodeVector/codevector_classes.py:226-250, batched: F frames
 * of L samples each (Y [F,L] fp64, host or device) -> mfcc_out [F,13] (host), the coefficients of
 * librosa.feature.mfcc(y=frame, sr, n_mfcc=13, n_fft=L, hop_length=None, center=False, n_mels=26).
 * 2 <= L <= 1024 (the reference's frames have 320 samples, the tail frame of a recording 13..319).
 * librosa is not available where this was built: the kernel follows its published algorithm as
 * restated in oracle/mfcc_oracle.py; parity with librosa itself is unpinned (DESIGN.md).
 * y_on_device != 0: Y is read on hmmb_get_stream() (it must be complete on that stream); the call returns with
 * mfcc_out written and Y no longer in use.                                                       */
int hmmb_mfcc_frames(const double *Y, int64_t F, int L, int y_on_device, double sr, double *mfcc_out);

/* ------------------------------------------------------------------ frame-file loader (host only)
 * Replaces the json.load + RawDataMFCC.from_dict loop of DataStorage.load_raw_data_mfcc,
 * CodeVector/codevector_classes.py:478-495, for the one field the hot path reads: scans the
 * text of a frame file (a JSON list of RawDataMFCC.to_dict() objects, :252-264) and writes
 * every "mfcc_vector" (13 fp64, bit-identical to Python's float parsing) to mfcc_out
 * [cap_frames,13] in file order.  Returns the number of frames found (frames beyond
 * cap_frames are counted but not stored; mfcc_out may be NULL to count only) or a negative
 * error (HMMB_ERR_RANGE: a vector that does not have 13 entries — the reference raises
 * ValueError("Vectors must be of size 13."), codevector_functions.py:83-84).  No CUDA needed.
 * text[len] must be readable and not part of a number (a NUL terminator, as in a C string or a
 * Python bytes object): numbers are parsed with strtod.                                      */
int64_t hmmb_frames_json_scan(const char *text, int64_t len, double *mfcc_out, int64_t cap_frames);

#ifdef __cplusplus
}
#endif
#endif /* HMMB200_H */

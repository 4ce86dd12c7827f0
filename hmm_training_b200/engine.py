"""Array-level Python API over the C ABI (packed codewords / flat matrices in, numpy out).

The reference-shaped drop-in modules (hmm_training.py, hmm_testing.py,
codevector_functions.py) are thin adapters from lists of dataclass objects to these calls.
Everything here runs on the GPU through libhmmb200.so; nothing falls back to the CPU.
"""
from __future__ import annotations

import ctypes
from typing import Callable, Optional, Tuple

import numpy as np

from . import _lib
from ._lib import check, c_f64, ptr


def default_init(N: int, M: int) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """(pi, A, B) defaults.  N == 4: the reference's literals (HMM/hmm_training.py:301,
    307-312, 318).  N != 4: the reference has no defaults (it raises IndexError); the
    generalisation (0.6/0.4 upper-bidiagonal A with absorbing last state,
    pi = [.97, .03/(N-1), ...]) is our documented extension."""
    if N == 4:
        pi = np.array([0.97, 0.02, 0.005, 0.005])
    else:
        pi = np.full(N, 0.03 / max(N - 1, 1))
        pi[0] = 0.97 if N > 1 else 1.0
    A = np.zeros((N, N))
    for i in range(N - 1):
        A[i, i] = 0.6
        A[i, i + 1] = 0.4
    A[N - 1, N - 1] = 1.0
    B = np.full((N, M), 1.0 / M)
    return pi, A, B


# ------------------------------------------------------------------------------- VQ / LBG
def vq_encode(X: np.ndarray, C: np.ndarray, near_ties: bool = False, near_cap: int = 1 << 20):
    """Nearest-centroid indices (int32 [F]) of frames X [F,13] against codebook C [K,13];
    dims 1..12 only, lowest index wins ties (HMM/hmm_training.py:95-118).

    near_ties=True also returns the parity contract's near-tie report: (idx, near, n_near) with ``near`` the
    ascending frame numbers (at most near_cap of them) whose two smallest distances differ by less than 1e-12
    relative — exact ties between duplicate centroids included — and n_near their total count.  Those are the
    frames whose index could differ under another BLAS's summation order in the reference's np.linalg.norm."""
    X = c_f64(X)
    C = c_f64(C)
    if X.ndim != 2 or X.shape[1] != 13 or C.ndim != 2 or C.shape[1] != 13:
        raise ValueError("Vectors must be of size 13.")  # codevector_functions.py:84
    idx = np.empty(X.shape[0], dtype=np.int32)
    if not near_ties:
        check(_lib.load().hmmb_vq_encode(ptr(X), X.shape[0], ptr(C), C.shape[0], ptr(idx)))
        return idx
    near = np.empty(max(min(int(near_cap), X.shape[0]), 1), dtype=np.int32)
    n_near = ctypes.c_int64(0)
    check(_lib.load().hmmb_vq_encode_ex(ptr(X), X.shape[0], ptr(C), C.shape[0], ptr(idx), ptr(near), len(near),
                                        ctypes.byref(n_near)))
    return idx, near[:min(n_near.value, len(near))].copy(), int(n_near.value)


def mfcc_frames(Y: np.ndarray, sr: float = 16000.0) -> np.ndarray:
    """[F, 13] MFCCs of F equal-length frames Y [F, L] — what RawDataMFCC.calculate_mfcc computes per frame
    with librosa (CodeVector/codevector_classes.py:226-250), batched on the GPU (hmmb_mfcc_frames)."""
    Y = c_f64(Y)
    if Y.ndim != 2:
        raise ValueError("frames must be [F, L]")
    out = np.empty((Y.shape[0], 13))
    if Y.shape[0]:
        check(_lib.load().hmmb_mfcc_frames(ptr(Y), Y.shape[0], Y.shape[1], 0, float(sr), ptr(out)))
    return out


def _wrap_allreduce(fn: Optional[Callable[[int, int], None]]):
    """fn(dev_ptr, n_doubles) -> None, wrapped as the C hook; returns (cfunc, keepalive)."""
    if fn is None:
        return None, None
    if isinstance(fn, str):
        if fn != "native":
            raise ValueError("allreduce must be a callable, None or 'native'")
        return _lib.load().hmmb_comm_allreduce, None  # the library's own NCCL communicator (dist.native_comm_init)

    def hook(dev_ptr, n, _user):
        try:
            fn(dev_ptr or 0, n)  # (NULL, 0) = "join" of an overlapping hook (hmmb_bw_set_overlap)
            return 0
        except Exception as exc:  # pragma: no cover - surfaced through the C error path
            import traceback
            traceback.print_exc()
            return 1

    cfn = _lib.ALLREDUCE_FN(hook)
    return cfn, hook


def lbg_fit(X, K: int = 256, max_iterations: int = 100, epsilon: float = 0.001,
            allreduce: Optional[Callable[[int, int], None]] = None, x_dev_ptr: Optional[int] = None,
            F: Optional[int] = None, history: bool = False):
    """LBG codebook (CodeVector/codevector_functions.py:442-531) on frames X [F,13].

    Returns (centroids [Kout,13], generations list of arrays, assign int32 [F],
    iters_per_generation int32 [n_gen], last global distance per generation); with history=True a sixth item:
    the list (one array per generation) of the summed distance after every Lloyd pass (:503, printed at :512-516)."""
    lib = _lib.load()
    if x_dev_ptr is None:
        X = c_f64(X)
        if X.ndim != 2 or (X.shape[0] and X.shape[1] != 13):
            raise ValueError("frames must be [F, 13]")
        F = X.shape[0]
        xp, on_dev = ptr(X), 0
    else:
        xp, on_dev = ctypes.c_void_p(x_dev_ptr), 1
    if K < 1:
        raise ValueError("centroids_quantity must be >= 1")
    n_gen = int(np.log2(K))
    kout = 1 << max(n_gen, 1)
    n_rows = 1 + sum(1 << g for g in range(1, n_gen + 1))
    C = np.zeros((kout, 13))
    gens = np.zeros((n_rows, 13))
    assign = np.zeros(max(F, 1), dtype=np.int32)
    iters = np.zeros(max(n_gen, 1), dtype=np.int32)
    gdist = np.zeros(max(n_gen, 1))
    hist = np.full((max(n_gen, 1), max(int(max_iterations), 1)), np.nan) if history else None
    cfn, keep = _wrap_allreduce(allreduce)
    rc = check(lib.hmmb_lbg_fit_ex(xp, F, on_dev, K, int(max_iterations), float(epsilon), ptr(C), ptr(gens),
                                   ptr(assign), ptr(iters), ptr(gdist), ptr(hist),
                                   ctypes.cast(cfn, ctypes.c_void_p) if cfn else None, None))
    del keep
    out, pos = [gens[0:1].copy()], 1
    for g in range(1, n_gen + 1):
        out.append(gens[pos:pos + (1 << g)].copy())
        pos += 1 << g
    res = (C[:rc].copy(), out, assign[:F], iters[:n_gen], gdist[:n_gen])
    if history:
        res += ([hist[g, :iters[g]].copy() for g in range(n_gen)],)
    return res


# ------------------------------------------------------------------------------- Baum-Welch
class BaumWelch:
    """Device-resident batched Baum-Welch trainer (wraps hmmb_bw_*).

    obs: packed unsigned codewords (uint8/uint16/uint32/int64 accepted), offsets int64 [R+1],
    word_of_seq int32 [R] in [0, W).  ``obs_dev_ptr`` passes codewords already in HBM."""

    def __init__(self, obs, offsets, word_of_seq, W: int, N: int, M: int, obs_dev_ptr: Optional[int] = None,
                 idx_bytes: Optional[int] = None, pipeline_upload: bool = False, init=None):
        lib = _lib.load()
        self._lib = lib
        self.W, self.N, self.M = int(W), int(N), int(M)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        word_of_seq = np.ascontiguousarray(word_of_seq, dtype=np.int32)
        self.R = len(offsets) - 1
        if obs_dev_ptr is None:
            obs = np.ascontiguousarray(obs)
            if obs.dtype.kind not in "iu":
                raise TypeError("codewords must be integers")
            if obs.dtype.kind == "i":
                if obs.size and int(obs.min()) < 0:
                    raise IndexError("negative codeword index")
                obs = obs.view({1: np.uint8, 2: np.uint16, 4: np.uint32, 8: np.uint64}[obs.dtype.itemsize])
            op, on_dev, ib = ptr(obs), 0, obs.dtype.itemsize
        else:
            op, on_dev, ib = ctypes.c_void_p(obs_dev_ptr), 1, int(idx_bytes)
        h = ctypes.c_void_p()
        # pipeline_upload: hmmb_bw_create_ex may return while pinned codewords are still crossing PCIe;
        # the first iterate() runs behind the upload, so the buffer is kept alive until close()
        # init = (pi0, A0, B0): uploaded by the create ahead of the bulk of the codewords (= set_params)
        p0 = a0 = b0 = None
        if init is not None:
            p0, a0, b0 = (c_f64(x) for x in init)
            if p0.shape != (self.W, self.N) or a0.shape != (self.W, self.N, self.N) or b0.shape != (self.W, self.N, self.M):
                raise ValueError(f"parameter shapes must be ({W},{N}), ({W},{N},{N}), ({W},{N},{M})")
        check(lib.hmmb_bw_create_ex(ctypes.byref(h), op, ib, on_dev, ptr(offsets), ptr(word_of_seq), self.R, self.W,
                                    self.N, self.M, 1 if pipeline_upload else 0, ptr(p0), ptr(a0), ptr(b0)))
        self._h = h
        self._keep = None
        self._obs_keepalive = (obs, p0, a0, b0) if pipeline_upload else None  # (pinned parameters go up asynchronously too)
        self.frames = int(lib.hmmb_bw_total_frames(h))

    def set_params(self, pi0, A0, B0) -> None:
        pi0, A0, B0 = c_f64(pi0), c_f64(A0), c_f64(B0)
        W, N, M = self.W, self.N, self.M
        if pi0.shape != (W, N) or A0.shape != (W, N, N) or B0.shape != (W, N, M):
            raise ValueError(f"parameter shapes must be ({W},{N}), ({W},{N},{N}), ({W},{N},{M})")
        check(self._lib.hmmb_bw_set_params(self._h, ptr(pi0), ptr(A0), ptr(B0)))

    def set_dist(self, rank: int, world: int, allreduce: Optional[Callable[[int, int], None]]) -> None:
        cfn, keep = _wrap_allreduce(allreduce)
        self._keep = (cfn, keep)
        check(self._lib.hmmb_bw_set_dist(self._h, rank, world, ctypes.cast(cfn, ctypes.c_void_p) if cfn else None,
                                         None))

    def set_overlap(self, groups: int) -> None:
        """Left-to-right kernels only: run the backward pass in `groups` word groups and hand each group's
        accumulators to the all-reduce hook as soon as its kernels are queued (use dist.make_allreduce(overlap=True))."""
        check(self._lib.hmmb_bw_set_overlap(self._h, int(groups)))

    def iterate(self, n_iter: int, epsilon: float = 1e-6, max_iterations: int = 100, sync_each: bool = True) -> None:
        check(self._lib.hmmb_bw_iterate(self._h, int(n_iter), float(epsilon), int(max_iterations), int(sync_each)))

    def params(self, finalize: bool = True, out=None):
        """(pi, A, B).  out = (pi, A, B) caller-provided C-contiguous float64 arrays of the right shapes (e.g. in
        pinned host memory: the device-to-host copy is then one direct DMA instead of going through bounce buffers)."""
        W, N, M = self.W, self.N, self.M
        if out is None:
            pi, A, B = np.empty((W, N)), np.empty((W, N, N)), np.empty((W, N, M))
        else:
            pi, A, B = out
            for x, shp in ((pi, (W, N)), (A, (W, N, N)), (B, (W, N, M))):
                if x.shape != shp or x.dtype != np.float64 or not x.flags.c_contiguous:
                    raise ValueError(f"out arrays must be C-contiguous float64 of shapes ({W},{N}), ({W},{N},{N}), ({W},{N},{M})")
        check(self._lib.hmmb_bw_get_params(self._h, int(finalize), ptr(pi), ptr(A), ptr(B)))
        return pi, A, B

    def history(self, cap: int):
        hist = np.full((self.W, max(cap, 1)), np.nan)
        iters = np.zeros(self.W, dtype=np.int32)
        check(self._lib.hmmb_bw_get_history(self._h, ptr(hist), hist.shape[1], ptr(iters)))
        return hist, iters

    def kernel_family(self) -> str:
        """E-step kernel family selected by the current parameters (see hmmb_bw_kernel_family)."""
        return self._lib.hmmb_bw_kernel_family(self._h).decode()

    def diagnostics(self):
        """(sequence passes recomputed by the exact log-space kernel, backward hand-overs)."""
        a, b = ctypes.c_int64(0), ctypes.c_int64(0)
        check(self._lib.hmmb_bw_diagnostics(self._h, ctypes.byref(a), ctypes.byref(b)))
        return a.value, b.value

    def thin_states(self) -> int:
        """(word, state) pairs whose A / B rows come from log-space sums (posterior mass below 2^-200)."""
        n = ctypes.c_int64(0)
        check(self._lib.hmmb_bw_thin_states(self._h, ctypes.byref(n)))
        return n.value

    def seq_ll(self) -> np.ndarray:
        out = np.empty(max(self.R, 1))
        check(self._lib.hmmb_bw_get_seq_ll(self._h, ptr(out)))
        return out[: self.R]

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.hmmb_bw_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def bw_fit(obs, offsets, word_of_seq, W: int, N: int, M: int, pi0, A0, B0, epsilon: float = 1e-6,
           max_iterations: int = 100, allreduce=None, rank: int = 0, world: int = 1, out=None):
    """Batched hmm_training (HMM/hmm_training.py:265-541) for W words at once.
    Returns (pi [W,N], A [W,N,N], B [W,N,M], ll_hist [W,max_iterations], iters [W]).  out: see BaumWelch.params."""
    with BaumWelch(obs, offsets, word_of_seq, W, N, M, pipeline_upload=True, init=(pi0, A0, B0)) as bw:
        if world > 1:
            bw.set_dist(rank, world, allreduce)
        bw.iterate(max_iterations, epsilon, max_iterations, sync_each=True)
        pi, A, B = bw.params(finalize=True, out=out)
        hist, iters = bw.history(max_iterations)
    return pi, A, B, hist, iters


# ------------------------------------------------------------------------------- recognition
def score(obs, offsets, N: int, M: int, pi, A, B, obs_dev_ptr: Optional[int] = None, idx_bytes: Optional[int] = None,
          want_ll: bool = True, out_ll: Optional[np.ndarray] = None):
    """log P(O_u | model_w) for every utterance x model ([U,W]) and test_hmm's argmax
    (HMM/hmm_testing.py:49-104, 139-161).  pi [W,N], A [W,N,N], B [W,N,M] linear space."""
    lib = _lib.load()
    pi, A, B = c_f64(pi), c_f64(A), c_f64(B)
    W = pi.shape[0]
    if pi.shape != (W, N) or A.shape != (W, N, N) or B.shape != (W, N, M):
        raise ValueError("model parameter shapes do not match (W, N, M)")
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    U = len(offsets) - 1
    if obs_dev_ptr is None:
        obs = np.ascontiguousarray(obs)
        if obs.dtype.kind == "i":
            if obs.size and int(obs.min()) < 0:
                raise IndexError("negative codeword index")
            obs = obs.view({1: np.uint8, 2: np.uint16, 4: np.uint32, 8: np.uint64}[obs.dtype.itemsize])
        op, on_dev, ib = ptr(obs), 0, obs.dtype.itemsize
    else:
        op, on_dev, ib = ctypes.c_void_p(obs_dev_ptr), 1, int(idx_bytes)
    if out_ll is not None:  # caller-provided [U, W] fp64 buffer (e.g. pinned memory: the D2H copy is then direct)
        if out_ll.shape != (U, W) or out_ll.dtype != np.float64 or not out_ll.flags.c_contiguous:
            raise ValueError(f"out_ll must be a C-contiguous float64 array of shape ({U}, {W})")
        ll = out_ll
    else:
        ll = np.empty((U, W)) if want_ll else None
    arg = np.empty(max(U, 1), dtype=np.int32)
    check(lib.hmmb_score(op, ib, on_dev, ptr(offsets), U, W, N, M, ptr(pi), ptr(A), ptr(B), ptr(ll), ptr(arg)))
    return ll, arg[:U]


def viterbi(obs, offsets, model_of_utt, N: int, M: int, pi, A, B, want_path: bool = True,
            obs_dev_ptr: Optional[int] = None, idx_bytes: Optional[int] = None):
    """Most likely state path of every utterance under its own model (hmmb_viterbi; an extension, the reference
    has no Viterbi).  Utterance u is decoded against model model_of_utt[u]; pi [W,N], A [W,N,N], B [W,N,M] linear.

    Returns (score float64 [U], path int8 [frames] or None): score[u] is the log-probability of the best path
    (-inf if the utterance is impossible under its model), and frame t of utterance u is path[offsets[u] -
    offsets[0] + t] (-1 on every frame of an impossible utterance).  want_path=False decodes the scores only."""
    lib = _lib.load()
    pi, A, B = c_f64(pi), c_f64(A), c_f64(B)
    W = pi.shape[0]
    if pi.shape != (W, N) or A.shape != (W, N, N) or B.shape != (W, N, M):
        raise ValueError("model parameter shapes do not match (W, N, M)")
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    U = len(offsets) - 1
    model_of_utt = np.ascontiguousarray(model_of_utt, dtype=np.int32)
    if model_of_utt.shape != (U,):
        raise ValueError(f"model_of_utt must hold one model index per utterance ({U})")
    if obs_dev_ptr is None:
        obs = np.ascontiguousarray(obs)
        if obs.dtype.kind == "i":
            if obs.size and int(obs.min()) < 0:
                raise IndexError("negative codeword index")
            obs = obs.view({1: np.uint8, 2: np.uint16, 4: np.uint32, 8: np.uint64}[obs.dtype.itemsize])
        op, on_dev, ib = ptr(obs), 0, obs.dtype.itemsize
    else:
        op, on_dev, ib = ctypes.c_void_p(obs_dev_ptr), 1, int(idx_bytes)
    frames = int(offsets[-1] - offsets[0]) if U > 0 else 0
    score = np.empty(max(U, 1))
    path = np.empty(max(frames, 1), dtype=np.int8) if want_path else None
    check(lib.hmmb_viterbi(op, ib, on_dev, ptr(offsets), U, ptr(model_of_utt), W, N, M, ptr(pi), ptr(A), ptr(B),
                           ptr(score), ptr(path)))
    return score[:U], (path[:frames] if want_path else None)

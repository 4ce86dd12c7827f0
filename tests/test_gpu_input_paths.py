"""The entry points and branches the benchmark times that the rest of the suite never reaches, against the oracle:
inputs that already live on the device (hmmb_vq_encode_dev, lbg_fit(x_dev_ptr=...), BaumWelch / score(obs_dev_ptr=...),
hmmb_mfcc_frames(y_on_device=1)), the chunked encode of frames in pinned host memory, and the argmax-only scorer
(want_ll=False, ll_out == NULL) — including how device-resident inputs are ordered with work a caller queued on torch's
stream.  Device buffers come from torch, as in bench.py.

Tolerances are those of tests/helpers.py: indices bit-exact, pi / A / B and log-likelihoods to 1e-9 relative, zero
patterns and the floored set of B exactly equal.
"""
import ctypes

import numpy as np
import pytest
import torch

from helpers import assert_close, assert_same_support, floored_set, load_golden
from hmm_training_b200 import _lib, dist, engine, synthetic
from oracle import hmm_oracle as O
from oracle import vq_oracle

pytestmark = pytest.mark.gpu

VQ_TILE = 512            # centroids per shared-memory tile of k_vq_assign (csrc/vq.cu)
VQ_CHUNK = 1 << 17       # frames per upload chunk of the pinned encode (hmmb_vq_encode_ex)


@pytest.fixture
def dev():
    """dev(a) -> a uint8 CUDA tensor holding the bytes of numpy array `a`, complete before it is returned.  At teardown
    the device is drained and the library gets its own stream back, so that a stream bound by a test (and torch's
    current stream) does not leak into other tests."""
    keep = []
    prev = torch.cuda.current_stream()

    def copy(a):
        a = np.ascontiguousarray(a)
        t = torch.from_numpy(a.reshape(-1).view(np.uint8).copy()).to("cuda")
        torch.cuda.synchronize()
        keep.append(t)
        return t

    yield copy
    torch.cuda.synchronize()
    _lib.check(_lib.load().hmmb_set_stream(None))
    torch.cuda.set_stream(prev)


def _pinned_copy(a):
    """numpy view of pinned host memory (hmmb_host_alloc) holding a copy of `a`, and its handle."""
    p = _lib.load().hmmb_host_alloc(a.nbytes)
    assert p
    buf = np.ctypeslib.as_array((ctypes.c_uint8 * a.nbytes).from_address(p)).view(a.dtype).reshape(a.shape)
    buf[...] = a
    return buf, p


def _host_free(p):
    _lib.load().hmmb_host_free(p)


# ---------------------------------------------------------------------------------------------- 1. VQ encode on device
def _encode_dev(dev, X, C, with_dist=True):
    """hmmb_vq_encode_dev on device copies of X / C; the outputs start as sentinels, so an unwritten entry shows."""
    lib = _lib.load()
    F = len(X)
    dX, dC = dev(np.asarray(X, np.float64)), dev(np.asarray(C, np.float64))
    d_idx = torch.full((F,), -7, dtype=torch.int32, device="cuda")
    d_dist = torch.full((F,), -1.0, dtype=torch.float64, device="cuda") if with_dist else None
    _lib.check(lib.hmmb_vq_encode_dev(dX.data_ptr(), F, dC.data_ptr(), len(C), d_idx.data_ptr(),
                                      d_dist.data_ptr() if with_dist else None))
    _lib.check(lib.hmmb_synchronize())  # the call returns while its kernels may still run
    return d_idx.cpu().numpy(), (d_dist.cpu().numpy() if with_dist else None)


def _check_encode_dev(dev, X, C, what):
    ref, ref_d = vq_oracle.encode(X, C, return_dist=True)
    idx, d = _encode_dev(dev, X, C)
    assert np.array_equal(idx, ref), f"{what}: {int((idx != ref).sum())} of {len(X)} indices differ"
    # both sides take sqrt of the same fma chain (DESIGN.md §5): the winning distance is bit-exact, +inf included
    assert np.array_equal(d, ref_d, equal_nan=True), f"{what}: {int((d != ref_d).sum())} distances differ"
    idx0, _ = _encode_dev(dev, X, C, with_dist=False)
    assert np.array_equal(idx0, ref), f"{what}: indices with d_dist = NULL"


@pytest.mark.parametrize("F,K", [(1, 1), (33, 7), (5000, 256), (3000, 700), (257, 1024)])
def test_vq_encode_dev_matches_oracle(F, K, dev):
    """Indices and winning distances of the device-pointer encode.  A twin centroid sends the frames nearest to it to
    the exact work list; the others are decided by the prefilter.  K > VQ_TILE: the winner's row is re-read from
    global memory."""
    X = synthetic.mfcc_mixture(F + K, F, K=min(K, 64))
    C = synthetic.random_codebook(K, K)
    if K > 3:
        C[K - 1] = C[1]
        X[: F // 4] = C[1] + 0.01 * X[: F // 4]  # a quarter of the frames lands on the twin: the work list
    _check_encode_dev(dev, X, C, f"F{F} K{K}")


@pytest.mark.parametrize("case", ["nan_inf_frames", "nan_inf_centroids", "all_centroids_nan", "one_centroid", "huge",
                                  "fp32_overflow", "tiny", "fp32_underflow", "twins", "twins_above_tile"])
def test_vq_encode_dev_edge_values_match_oracle(case, dev):
    """The edge values of test_vq_encode_edge_values_match_oracle through the device-pointer entry point, distances
    included (the all-NaN codebook keeps index 0 at distance +inf), and exact twins on both sides of VQ_TILE."""
    X = synthetic.mfcc_mixture(0, 4000, K=8); C = synthetic.random_codebook(1, 256)
    if case == "nan_inf_frames":
        X = X.copy(); X[2, 5] = np.nan; X[3, 0] = np.nan; X[4, 1] = np.inf; X[5, 2] = -np.inf; X[100:200, 7] = np.nan
    elif case == "nan_inf_centroids":
        C = C.copy(); C[0, 3] = np.nan; C[7] = np.inf; C[2, 0] = np.nan
    elif case == "all_centroids_nan": C = np.full((4, 13), np.nan)
    elif case == "one_centroid": C = C[:1]
    elif case == "huge": X, C = X * 1e200, C * 1e200
    elif case == "fp32_overflow": X, C = X * 1e30, C * 1e30
    elif case == "tiny": X, C = X * 1e-200, C * 1e-200
    elif case == "fp32_underflow": X, C = X * 1e-30, C * 1e-30
    elif case in ("twins", "twins_above_tile"):
        if case == "twins_above_tile":
            C = synthetic.random_codebook(2, VQ_TILE + 300)
        C[9] = C[2]; C[-1] = C[5]
        X = X.copy(); X[::3] = C[2] + 0.02 * X[::3]; X[1::3] = C[5] + 0.02 * X[1::3]
    _check_encode_dev(dev, X, C, case)


# ---------------------------------------------------------------------------------------------- 2. stream ordering
def test_device_inputs_are_read_in_stream_order(dev):
    """With the library bound to torch's stream, a torch write queued just before the call (and held back by a spin on
    the stream, so the host is well ahead) is what the call reads, and a torch read queued after it sees its output;
    no host synchronisation in between.  The same for a trainer created on device codewords."""
    lib = _lib.load()
    s = dist.bind_torch_stream()
    assert lib.hmmb_get_stream() == s.cuda_stream
    F, K = 200_000, 256
    X = synthetic.mfcc_mixture(21, F, K=64)
    C = synthetic.random_codebook(22, K)
    C[K - 1] = C[3]
    ref = vq_oracle.encode(X, C)
    hX = torch.from_numpy(X).pin_memory()
    dX = torch.full((F, 13), float("nan"), dtype=torch.float64, device="cuda")
    dC = torch.from_numpy(C).cuda()
    d_idx = torch.full((F,), -7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    torch.cuda._sleep(20_000_000)
    dX.copy_(hX, non_blocking=True)
    _lib.check(lib.hmmb_vq_encode_dev(dX.data_ptr(), F, dC.data_ptr(), K, d_idx.data_ptr(), None))
    got = d_idx.cpu().numpy()
    assert np.array_equal(got, ref), f"{int((got != ref).sum())} of {F} indices differ"

    # Baum-Welch: the codeword buffer holds 0xffff (>= M) until the torch copy lands
    g = load_golden("bw_clustered_s2_it1")
    N, M, W = 4, 256, 3
    obs16 = g["obs"].astype(np.uint16)
    pi0, A0, B0 = engine.default_init(N, M)
    pi0, A0, B0 = np.tile(pi0, (W, 1)), np.tile(A0, (W, 1, 1)), np.tile(B0, (W, 1, 1))
    d_obs = torch.full((obs16.size,), -1, dtype=torch.int16, device="cuda")
    h_obs = torch.from_numpy(obs16.view(np.int16)).pin_memory()
    torch.cuda.synchronize()
    torch.cuda._sleep(20_000_000)
    d_obs.copy_(h_obs, non_blocking=True)
    with engine.BaumWelch(None, g["offsets"], g["word_of_seq"], W, N, M, obs_dev_ptr=d_obs.data_ptr(), idx_bytes=2) as bw:
        bw.set_params(pi0, A0, B0)
        bw.iterate(3, 1e-6, 3)
        a = bw.params() + bw.history(3)
    with engine.BaumWelch(obs16, g["offsets"], g["word_of_seq"], W, N, M) as bw:
        bw.set_params(pi0, A0, B0)
        bw.iterate(3, 1e-6, 3)
        b = bw.params() + bw.history(3)
    for x, y in zip(a, b):
        assert np.array_equal(x, y, equal_nan=True)


def test_device_inputs_on_the_library_stream(dev):
    """Without binding, the library runs on its own non-blocking stream: the documented pattern is
    torch.cuda.synchronize() before the call and hmmb_synchronize() before the output is read."""
    lib = _lib.load()
    _lib.check(lib.hmmb_set_stream(None))
    F, K = 100_000, 256
    X = synthetic.mfcc_mixture(23, F, K=64)
    C = synthetic.random_codebook(24, K)
    ref, ref_d = vq_oracle.encode(X, C, return_dist=True)
    dX = torch.full((F, 13), float("nan"), dtype=torch.float64, device="cuda")
    dX.copy_(torch.from_numpy(X).pin_memory(), non_blocking=True)
    dC = torch.from_numpy(C).cuda()
    d_idx = torch.full((F,), -7, dtype=torch.int32, device="cuda")
    d_dist = torch.full((F,), -1.0, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    _lib.check(lib.hmmb_vq_encode_dev(dX.data_ptr(), F, dC.data_ptr(), K, d_idx.data_ptr(), d_dist.data_ptr()))
    _lib.check(lib.hmmb_synchronize())
    assert np.array_equal(d_idx.cpu().numpy(), ref)
    assert np.array_equal(d_dist.cpu().numpy(), ref_d)


def test_stream_switch_orders_the_new_stream_behind_the_old(dev):
    """hmmb_vq_encode_dev returns with its kernels queued and its scratch blocks (work list and its counter) back in
    the library's allocator.  hmmb_set_stream must therefore start the new stream behind the work queued on the old
    one, or the next call could reuse those blocks while the first call still runs: work queued on the library's own
    stream after the switch completes only after the first call (held back by a spin on torch's stream), and both
    encodes give the oracle's indices."""
    lib = _lib.load()
    F, K = 400_000, 256
    X1 = synthetic.mfcc_mixture(25, F, K=64); X2 = synthetic.mfcc_mixture(26, F, K=64)
    C = synthetic.random_codebook(27, K)
    C[K - 1] = C[3]; C[K - 2] = C[7]  # many frames on the work list
    X1[::2] = C[3] + 0.01 * X1[::2]; X2[::2] = C[7] + 0.01 * X2[::2]
    ref1, ref2 = vq_oracle.encode(X1, C), vq_oracle.encode(X2, C)
    dX1, dX2, dC = dev(X1), dev(X2), dev(C)
    i1 = torch.full((F,), -7, dtype=torch.int32, device="cuda")
    i2 = torch.full((F,), -7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    s = dist.bind_torch_stream()
    torch.cuda._sleep(50_000_000)
    _lib.check(lib.hmmb_vq_encode_dev(dX1.data_ptr(), F, dC.data_ptr(), K, i1.data_ptr(), None))
    first_done = torch.cuda.Event()
    first_done.record(s)
    _lib.check(lib.hmmb_set_stream(None))
    _lib.check(lib.hmmb_vq_encode_dev(dX2.data_ptr(), F, dC.data_ptr(), K, i2.data_ptr(), None))
    second_done = torch.cuda.Event()
    second_done.record(torch.cuda.ExternalStream(lib.hmmb_get_stream()))
    second_done.synchronize()
    assert first_done.query(), "the library's own stream ran ahead of the work queued on the stream bound before"
    s.synchronize()
    assert np.array_equal(i1.cpu().numpy(), ref1)
    assert np.array_equal(i2.cpu().numpy(), ref2)


# ---------------------------------------------------------------------------------------------- 3. pinned chunked encode
def test_vq_encode_pinned_chunks_match_oracle_and_pageable_report():
    """Frames in pinned host memory are uploaded and encoded chunk by chunk (the last chunk partial); every chunk resets
    the work list and reports its near-ties with the chunk's first frame added (near_base).  Indices equal the oracle's,
    the near-tie report equals the pageable call's, a report capped below its count keeps the full count."""
    F = 3 * VQ_CHUNK + 12_345
    X = synthetic.mfcc_mixture(31, F, K=64)
    C = synthetic.random_codebook(32, 256)
    C[9] = C[2]; C[200] = C[17]  # exact twins: every frame nearest to 2 or 17 is a near-tie
    X[::5] = C[2] + 0.02 * X[::5]
    ref = vq_oracle.encode(X, C)
    idx_h, near_h, n_h = engine.vq_encode(X, C, near_ties=True)
    assert np.array_equal(idx_h, ref)
    assert n_h == len(near_h) > 0 and (near_h >= 2 * VQ_CHUNK).any() and (near_h >= 3 * VQ_CHUNK).any()
    pinned, h = _pinned_copy(X)
    try:
        assert np.array_equal(engine.vq_encode(pinned, C), ref)
        idx_p, near_p, n_p = engine.vq_encode(pinned, C, near_ties=True)
        assert np.array_equal(idx_p, ref)
        assert n_p == n_h and np.array_equal(near_p, near_h)
        cap = 1000
        assert n_h > cap
        _, near_c, n_c = engine.vq_encode(pinned, C, near_ties=True, near_cap=cap)
        assert n_c == n_h and len(near_c) == cap and set(near_c.tolist()) <= set(near_h.tolist())
    finally:
        _host_free(h)


# ---------------------------------------------------------------------------------------------- 4. LBG from device frames
def test_lbg_50k_frames_from_device_matches_oracle(dev):
    """hmmb_lbg_fit_ex(x_on_device = 1), the path bench.py times, against vq_oracle.lbg: iteration counts, assignments,
    centroids of every generation; the per-pass distances equal those of the host-frame call."""
    F, K, it = 50_000, 256, 20
    X = synthetic.mfcc_mixture(41, F, K)
    dX = dev(X)
    C, gens, assign, iters, gd, hist = engine.lbg_fit(None, K, it, 1e-3, x_dev_ptr=dX.data_ptr(), F=F, history=True)
    Co, genso, assigno, iterso, gdo = vq_oracle.lbg(X, K, it, 1e-3)
    assert np.array_equal(iters, iterso)
    assert_close(gd, gdo, "summed distances", rtol=1e-12, atol=0)
    assert_close(C, Co, "centroids", rtol=1e-9, atol=1e-12)
    assert_close(np.concatenate(gens), np.concatenate(genso), "generations", rtol=1e-9, atol=1e-12)
    assert np.array_equal(assign, assigno), f"{int((assign != assigno).sum())} assignments differ"
    Ch, _, _, iters_h, gd_h, hist_h = engine.lbg_fit(X, K, it, 1e-3, history=True)
    assert np.array_equal(iters_h, iters)
    for g in range(len(iters)):
        assert len(hist[g]) == iters[g] and hist[g][-1] == gd[g]
        assert_close(hist[g], hist_h[g], f"generation {g}: distance after every pass", rtol=1e-12, atol=0)


# ---------------------------------------------------------------------------------------------- 5. Baum-Welch, device codewords
WIDTH_DTYPE = {1: np.uint8, 2: np.uint16, 4: np.uint32, 8: np.uint64}

BW_FAMILIES = {  # id: (N, M, transitions, expected kernel family)
    "n4_ltr": (4, 256, "bidiag", "n4_left_to_right"),
    "n4_dense": (4, 256, "dense", "n4_dense"),
    "ltr_n8": (8, 64, "bidiag", "left_to_right"),
    "ltr_n16": (16, 300, "bidiag", "left_to_right"),
    "generic_n5": (5, 40, "dense", "generic"),
    "generic_n4_m513": (4, 513, "bidiag", "generic"),
}


def _ragged_corpus(seed, W, N, M, S=30):
    """W words of S ragged recordings (T = 1 .. 40, two of them T = 1), packed in shuffled order."""
    rng = np.random.default_rng(seed)
    corpus = []
    for w in range(W):
        seqs = synthetic.clustered_sequences(rng, S + 3 * w, N=N, M=M, tmin=2, tmax=40, shift=5 * w,
                                             spread=max(2, M // (2 * N)))
        seqs[0] = seqs[0][:1]; seqs[5] = seqs[5][:1]
        corpus.append(seqs)
    flat = [(w, s) for w, word in enumerate(corpus) for s in word]
    perm = rng.permutation(len(flat))
    obs = np.concatenate([flat[i][1] for i in perm])
    offsets = np.concatenate([[0], np.cumsum([len(flat[i][1]) for i in perm])]).astype(np.int64)
    wos = np.array([flat[i][0] for i in perm], dtype=np.int32)
    return corpus, [flat[i][1] for i in perm], obs, offsets, wos


def _init(rng, W, N, M, kind):
    pi0 = np.zeros((W, N)); A0 = np.zeros((W, N, N)); B0 = rng.dirichlet(np.ones(M), size=(W, N))
    for w in range(W):
        if kind == "bidiag":
            pi0[w], A0[w], _ = engine.default_init(N, M)
        else:
            pi0[w] = rng.dirichlet(np.ones(N)); A0[w] = rng.dirichlet(np.ones(N), size=N)
    return pi0, A0, B0


def _bw_run(obs, offsets, wos, W, N, M, init, family, **kw):
    """1 iteration, the per-sequence LL of its E-step (under `init`), 2 more iterations."""
    with engine.BaumWelch(obs, offsets, wos, W, N, M, **kw) as bw:
        bw.set_params(*init)
        assert bw.kernel_family() == family
        bw.iterate(1, 1e-6, 3)
        ll = bw.seq_ll().copy()
        bw.iterate(2, 1e-6, 3)
        return bw.params() + bw.history(3) + (ll,)


def _check_bw_oracle(res, corpus, seqs, wos, init, N, M, what):
    pi, A, B, hist, iters, ll = res
    pi0, A0, B0 = init
    W = len(corpus)
    ref_ll = O.score_batch(seqs, [(A0[w], B0[w], pi0[w]) for w in range(W)])[np.arange(len(seqs)), wos]
    assert_close(ll, ref_ll, f"{what}: per-sequence LL of the first E-step")
    for w in range(W):
        Ao, Bo, pio, h, it = O.hmm_training(corpus[w], N=N, M=M, max_iterations=3, init=(pi0[w], A0[w], B0[w]),
                                            return_history=True)
        assert it == iters[w]
        assert_close(hist[w, :it], h, f"{what} w{w} ll")
        assert_close(A[w], Ao, f"{what} w{w} A"); assert_close(B[w], Bo, f"{what} w{w} B")
        assert_close(pi[w], pio, f"{what} w{w} pi")
        assert_same_support(A[w], Ao); assert_same_support(pi[w], pio)
        assert np.array_equal(floored_set(B[w], M), floored_set(Bo, M))


@pytest.mark.parametrize("fam,width", [(f, b) for f in BW_FAMILIES for b in (1, 2, 4, 8)
                                       if b > 1 or BW_FAMILIES[f][1] <= 256])  # (one byte holds M <= 256)
def test_baum_welch_device_codewords_match_oracle(fam, width, dev):
    """BaumWelch(obs_dev_ptr=..., idx_bytes=width) in every kernel family, ragged (T = 1 included) and shuffled: the
    first E-step's per-sequence LL and three iterations against the oracle.  The two N = 4 families (n4_*) have no
    atomics, so they must also equal the host-pointer call bit for bit."""
    N, M, kind, family = BW_FAMILIES[fam]
    W = 3
    corpus, seqs, obs, offsets, wos = _ragged_corpus(N * 31 + M, W, N, M)
    init = _init(np.random.default_rng(M + N), W, N, M, kind)
    raw = obs.astype(WIDTH_DTYPE[width])
    d = dev(raw)
    res = _bw_run(None, offsets, wos, W, N, M, init, family, obs_dev_ptr=d.data_ptr(), idx_bytes=width)
    _check_bw_oracle(res, corpus, seqs, wos, init, N, M, f"{fam} device u{8 * width}")
    if family.startswith("n4_"):
        host = _bw_run(raw, offsets, wos, W, N, M, init, family)
        for x, y in zip(res, host):
            assert np.array_equal(x, y, equal_nan=True)


@pytest.mark.parametrize("N", [4, 5, 8])
def test_device_codewords_from_a_slice_of_a_larger_buffer(N, dev):
    """offsets[0] > 0: the sequences start inside a larger device buffer whose head and tail hold codewords >= M.
    Training and scoring must read from obs + offsets[0], never from the head (which would raise IndexError)."""
    M, W, P = 200, 3, 37
    corpus, seqs, obs, offsets, wos = _ragged_corpus(50 + N, W, N, M)
    family = {4: "n4_left_to_right", 5: "generic", 8: "left_to_right"}[N]
    init = _init(np.random.default_rng(N), W, N, M, "bidiag")
    buf = np.concatenate([np.full(P, M + 3), obs, np.full(19, 65535)]).astype(np.uint16)
    d = dev(buf)
    res = _bw_run(None, offsets + P, wos, W, N, M, init, family, obs_dev_ptr=d.data_ptr(), idx_bytes=2)
    _check_bw_oracle(res, corpus, seqs, wos, init, N, M, f"slice N{N}")
    pi, A, B = init
    ll, arg = engine.score(None, offsets + P, N, M, pi, A, B, obs_dev_ptr=d.data_ptr(), idx_bytes=2)
    ll_h, arg_h = engine.score(obs.astype(np.uint16), offsets, N, M, pi, A, B)
    assert np.array_equal(ll, ll_h) and np.array_equal(arg, arg_h)


@pytest.mark.parametrize("width", [1, 2, 4, 8])
def test_device_codeword_out_of_range_raises(width, dev):
    """A codeword >= M inside the device buffer is reported through the device flag as IndexError by the create and by
    the scorer, for every layout (N = 4 blocked, N = 5 generic, N = 8 both) — also when only high bits are set."""
    M, W = 200, 2
    bad = {1: 250, 2: M + 1, 4: (1 << 16) + 1, 8: (1 << 40) + 1}[width]
    for N in (4, 5, 8):
        _, _, obs, offsets, wos = _ragged_corpus(60 + N, W, N, M, S=12)
        raw = obs.astype(WIDTH_DTYPE[width])
        raw[len(raw) // 2 + 3] = bad
        d = dev(raw)
        with pytest.raises(IndexError):
            engine.BaumWelch(None, offsets, wos, W, N, M, obs_dev_ptr=d.data_ptr(), idx_bytes=width)
        pi, A, B = _init(np.random.default_rng(1), W, N, M, "bidiag")
        with pytest.raises(IndexError):
            engine.score(None, offsets, N, M, pi, A, B, obs_dev_ptr=d.data_ptr(), idx_bytes=width)


def test_left_to_right_device_create_then_dense_transitions(dev):
    """N = 8 from device codewords builds both layouts at create time; set_params with a dense A after a bidiagonal one
    switches to the generic kernels, whose layout came from the same device buffer."""
    N, M, W = 8, 64, 3
    corpus, seqs, obs, offsets, wos = _ragged_corpus(70, W, N, M)
    rng = np.random.default_rng(71)
    ltr, dense = _init(rng, W, N, M, "bidiag"), _init(rng, W, N, M, "dense")
    d = dev(obs.astype(np.uint32))
    with engine.BaumWelch(None, offsets, wos, W, N, M, obs_dev_ptr=d.data_ptr(), idx_bytes=4) as bw:
        bw.set_params(*ltr)
        assert bw.kernel_family() == "left_to_right"
        bw.iterate(2, 1e-6, 2)
        bw.set_params(*dense)
        assert bw.kernel_family() == "generic"
        bw.iterate(1, 1e-6, 3)
        ll = bw.seq_ll().copy()
        bw.iterate(2, 1e-6, 3)
        res = bw.params() + bw.history(3) + (ll,)
    _check_bw_oracle(res, corpus, seqs, wos, dense, N, M, "N8 dense after bidiagonal")


# ---------------------------------------------------------------------------------------------- 6. recognition, device codewords
def _score_models(rng, W, N, M, kind):
    """W models with structural zeros: a sparse pi, a model that cannot emit the lower half of the codebook, a state
    that emits nothing; codeword M - 1 is emitted by no model ("unknown" utterances)."""
    pi, A, B = _init(rng, W, N, M, kind)
    pi[1] = 0.0; pi[1, 0] = 1.0
    B[2, :, : M // 2] = 0.0
    B[3, N - 1, :] = 0.0
    B[:, :, M - 1] = 0.0
    return pi, A, B


@pytest.mark.parametrize("N,M,kind", [(4, 256, "bidiag"), (4, 256, "dense"), (8, 200, "bidiag"), (16, 200, "bidiag"),
                                      (5, 200, "dense")])
def test_scoring_device_codewords_match_oracle(N, M, kind, dev):
    """engine.score(obs_dev_ptr=..., idx_bytes=width) in every scorer family against the oracle: structural -inf,
    unknown utterances (-1) and the first-maximum argmax; and equal to the host-pointer call."""
    rng = np.random.default_rng(N * 13 + M + len(kind))
    W, U = 5, 120
    pi, A, B = _score_models(rng, W, N, M, kind)
    seqs = [rng.integers(0, M - 1, size=int(rng.integers(1, 50))) for _ in range(U)]
    seqs[4] = rng.integers(M // 2, M - 1, size=20)           # possible under model 2
    seqs[7] = np.full(5, M - 1); seqs[8] = np.array([M - 1])  # possible under no model
    obs = np.concatenate(seqs)
    offsets = np.concatenate([[0], np.cumsum([len(s) for s in seqs])]).astype(np.int64)
    ref = O.score_batch(seqs, [(A[w], B[w], pi[w]) for w in range(W)])
    ll_h, arg_h = engine.score(obs.astype(np.int64), offsets, N, M, pi, A, B)
    for width in (1, 2, 4, 8):
        if M > 256 and width == 1:
            continue
        d = dev(obs.astype(WIDTH_DTYPE[width]))
        ll, arg = engine.score(None, offsets, N, M, pi, A, B, obs_dev_ptr=d.data_ptr(), idx_bytes=width)
        assert np.array_equal(np.isneginf(ll), np.isneginf(ref))
        assert_close(ll, ref, f"N{N} {kind} u{8 * width}")
        assert np.array_equal(arg, O.argmax_first(ref))
        assert arg[7] == arg[8] == -1 and np.isneginf(ll[:, 2]).sum() > U // 2 and np.isfinite(ll[4, 2])
        assert np.array_equal(ll, ll_h) and np.array_equal(arg, arg_h)


# ---------------------------------------------------------------------------------------------- 7. argmax-only recognition
def _check_argmax_only(obs, offsets, N, M, pi, A, B, what, other_B=None, sample_n=300):
    """Argmax-only call (want_ll=False) against the full call and the oracle on a sample.  A call with other emission
    matrices runs first, so that the device blocks the argmax-only call recycles hold a different [U, W] matrix: an
    argmax taken before every stage has been scored cannot come out right by accident."""
    if other_B is not None:
        engine.score(obs, offsets, N, M, pi, A, other_B)
    _, arg_only = engine.score(obs, offsets, N, M, pi, A, B, want_ll=False)
    ll, arg = engine.score(obs, offsets, N, M, pi, A, B)
    assert not np.isnan(ll).any()
    assert np.array_equal(arg, O.argmax_first(ll)), f"{what}: argmax of the full call"
    assert np.array_equal(arg_only, arg), f"{what}: {int((arg_only != arg).sum())} argmax-only results differ"
    U = len(offsets) - 1
    rng = np.random.default_rng(U)
    sample = np.unique(np.concatenate([np.arange(40), np.arange(U - 40, U), rng.choice(U, sample_n, replace=False)]))
    ref = O.score_batch([np.asarray(obs[offsets[u]:offsets[u + 1]], np.int64) for u in sample],
                        [(A[w], B[w], pi[w]) for w in range(len(pi))])
    assert_close(ll[sample], ref, f"{what}: sampled log-likelihoods")
    assert np.array_equal(arg[sample], O.argmax_first(ref))
    return ll


@pytest.mark.parametrize("tiny", [False, True])
def test_argmax_only_pipelined_scorer(tiny, monkeypatch):
    """Pinned codewords in length order, N = 4, 69 MB: the pipelined scorer runs its argmax-only stages (4) with no
    log-likelihood copies, and on models with denormal emissions the exact recomputation with ll_out == NULL."""
    from test_gpu_parity import _tiny_models
    monkeypatch.delenv("HMMB_SCORE_NO_PIPELINE", raising=False)
    rng = np.random.default_rng(81)
    N, W, U, T = 4, 6, 800_000, 86
    if tiny:
        M = 16
        pi, A, B = _tiny_models(rng, W, N, M)
        obs = rng.integers(0, M, size=U * T).astype(np.uint8)
    else:
        M = 256
        pi0, A0, _ = engine.default_init(N, M)
        pi, A = np.tile(pi0, (W, 1)), np.tile(A0, (W, 1, 1))
        B = rng.dirichlet(np.ones(M) * 0.3, size=(W, N))
        obs, _, _ = synthetic.fixed_length_codewords(8, 4, U // 4, T, N, M)
    assert obs.nbytes >= 4 << 24  # four upload chunks: the four argmax-only stages
    offsets = np.arange(U + 1, dtype=np.int64) * T
    pinned, h = _pinned_copy(obs)
    try:
        ll = _check_argmax_only(pinned, offsets, N, M, pi, A, B, "pipelined", other_B=B[::-1].copy())
    finally:
        _host_free(h)
    if tiny:
        fin = np.isfinite(ll)
        assert fin.any() and (ll[fin] < -700).any()  # the denormal / exact paths were exercised


def test_argmax_only_left_to_right_stress_shape():
    """BASELINE config 5's stress shape reduced in U: N = 16, M = 1024, uint16 pinned codewords, left-to-right models
    (k_scoreL), argmax only."""
    rng = np.random.default_rng(82)
    N, M, W, U, T = 16, 1024, 10, 20_000, 100
    obs, offsets, _ = synthetic.fixed_length_codewords(9, W, U // W, T, N, M)
    pi0, A0, _ = engine.default_init(N, M)
    pi, A = np.tile(pi0, (W, 1)), np.tile(A0, (W, 1, 1))
    B = rng.dirichlet(np.ones(M) * 0.3, size=(W, N))
    pinned, h = _pinned_copy(obs)
    try:
        _check_argmax_only(pinned, offsets, N, M, pi, A, B, "k_scoreL", other_B=B[::-1].copy(), sample_n=150)
    finally:
        _host_free(h)


@pytest.mark.parametrize("tiny", [False, True])
def test_argmax_only_unpipelined_scorer(tiny, monkeypatch):
    """Pageable codewords with HMMB_SCORE_NO_PIPELINE=1: the plain scorer's argmax-only call, exact recomputation
    included."""
    from test_gpu_parity import _tiny_models
    monkeypatch.setenv("HMMB_SCORE_NO_PIPELINE", "1")
    rng = np.random.default_rng(83)
    N, W, U = 4, 6, 60_000
    M = 16 if tiny else 256
    if tiny:
        pi, A, B = _tiny_models(rng, W, N, M)
    else:
        pi, A, B = _init(rng, W, N, M, "dense")
    lens = rng.integers(1, 120, size=U)
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    obs = rng.integers(0, M, size=int(offsets[-1])).astype(np.uint8)
    _check_argmax_only(obs, offsets, N, M, pi, A, B, "plain", other_B=B[::-1].copy())


# ---------------------------------------------------------------------------------------------- 8. MFCC from device samples
@pytest.mark.parametrize("L", [320, 1024, 13])
def test_mfcc_device_samples_equal_host_call(L, dev):
    """hmmb_mfcc_frames(y_on_device=1) gives the host call's bits (L = 320: MFCC_BPL_SMALL, L = 1024:
    MFCC_BPL_LARGE, L = 13: the shortest tail frame of a recording)."""
    rng = np.random.default_rng(L)
    F = 3001
    Y = rng.normal(size=(F, L)) * 2000.0
    Y[5] = 0.0
    host = engine.mfcc_frames(Y, 16000)
    d = dev(Y)
    out = np.empty((F, 13))
    _lib.check(_lib.load().hmmb_mfcc_frames(d.data_ptr(), F, L, 1, 16000.0, out.ctypes.data_as(ctypes.c_void_p)))
    assert np.array_equal(out, host)

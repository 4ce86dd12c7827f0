"""Connected-word decoding on the GPU (hmmb_decode_words, engine.decode_words, hmm_testing.recognize_connected) against
the numpy oracle oracle/words_oracle.py (itself checked against brute force in tests/test_words_oracle.py).

Scores must agree to 1e-9 relative with the same -inf pattern.  Segments must equal the oracle's wherever its
smallest decision margin exceeds 1e-9; below that, a log() differing in the last bit may pick another segmentation of
(within tolerance) the same score, so there the GPU's segments must only be a valid segmentation whose recomputed
score meets the oracle's at 1e-9."""
import numpy as np
import pytest
import torch

from helpers import RTOL, assert_close
from hmm_training_b200 import _lib, engine, hmm_testing, synthetic
from hmm_training_b200.hmm_classes import HMMTrained
from oracle.hmm_oracle import safe_log
from oracle.words_oracle import decode_words_batch

pytestmark = pytest.mark.gpu

MARGIN = 1e-9


@pytest.fixture(params=["native", "generic"])
def family(request, monkeypatch):
    """Every case once with the kernels the shape selects and once with the generic kernels forced."""
    if request.param == "generic":
        monkeypatch.setenv("HMMB_FORCE_GENERIC", "1")
    else:
        monkeypatch.delenv("HMMB_FORCE_GENERIC", raising=False)
    return request.param


def make_models(rng, W, N, M, ltr, zeros=False):
    pi = rng.random((W, N)) + 0.05
    if ltr:
        A = np.zeros((W, N, N))
        for i in range(N - 1):
            stay = rng.uniform(0.3, 0.95, size=W)
            A[:, i, i] = stay
            A[:, i, i + 1] = 1 - stay
        A[:, N - 1, N - 1] = 1.0
    else:
        A = rng.random((W, N, N)) ** 3 + 1e-3
    B = rng.random((W, N, M)) ** 4 + 1e-6
    if zeros:
        pi[rng.random((W, N)) < 0.25] = 0.0
        if not ltr:
            A[rng.random((W, N, N)) < 0.25] = 0.0
        B[rng.random((W, N, M)) < 0.25] = 0.0
    pi /= np.maximum(pi.sum(1, keepdims=True), 1e-300)
    A /= np.maximum(A.sum(2, keepdims=True), 1e-300)
    B /= np.maximum(B.sum(2, keepdims=True), 1e-300)
    return pi, A, B


def make_corpus(rng, U, M, tmax=60, long_T=None):
    lens = rng.integers(1, tmax + 1, size=U)
    lens[0] = 1
    if long_T:
        lens[1] = long_T
    return [rng.integers(0, M, size=int(T)) for T in lens]


def pack(seqs, dtype=None):
    offsets = np.zeros(len(seqs) + 1, np.int64)
    offsets[1:] = np.cumsum([len(s) for s in seqs])
    flat = np.concatenate(seqs) if seqs else np.zeros(0, np.int64)
    if dtype is None:
        dtype = np.uint8 if flat.max(initial=0) < 256 else np.uint16
    return np.ascontiguousarray(flat.astype(dtype)), offsets


def segmentation_logp(o, segs, pi, A, B, pen):
    """Sum of the best in-word paths of the segments (each entered anywhere, left from the last state) + K * pen."""
    lA, lB, lpi = safe_log(A), safe_log(B), safe_log(pi)
    N = lpi.shape[1]
    total = 0.0
    for k, (w, a) in enumerate(segs):
        b = segs[k + 1][1] - 1 if k + 1 < len(segs) else len(o) - 1
        d = lpi[w] + lB[w][:, o[a]]
        for t in range(a + 1, b + 1):
            d = np.max(d[:, None] + lA[w], axis=0) + lB[w][:, o[t]]
        total += d[N - 1]
    return total + len(segs) * pen


def check_against_oracle(seqs, pi, A, B, pen, res, what="", sample=None):
    score, seg_off, seg_word, seg_start = res
    us = np.arange(len(seqs)) if sample is None else np.asarray(sample)
    models = [(A[w], B[w], pi[w]) for w in range(pi.shape[0])]
    osc, ooff, oword, ostart, omarg = decode_words_batch([seqs[u] for u in us], models, pen)
    sc = score[us]
    assert np.array_equal(np.isneginf(sc), np.isneginf(osc)), f"{what}: -inf pattern differs"
    assert_close(sc, osc, what + " score")
    assert seg_off[0] == 0 and np.all(np.diff(seg_off) >= 0) and len(seg_word) == len(seg_start) == seg_off[-1]
    n_near = 0
    for k, u in enumerate(us):
        got = list(zip(seg_word[seg_off[u]:seg_off[u + 1]].tolist(), seg_start[seg_off[u]:seg_off[u + 1]].tolist()))
        want = list(zip(oword[ooff[k]:ooff[k + 1]].tolist(), ostart[ooff[k]:ooff[k + 1]].tolist()))
        if np.isneginf(osc[k]):
            assert got == [], f"{what}: utterance {u} is impossible but has segments"
        elif omarg[k] > MARGIN:
            assert got == want, f"{what}: utterance {u} (T={len(seqs[u])}, margin {omarg[k]:.3g}) segments differ"
        else:
            n_near += 1
            W = pi.shape[0]
            assert got and got[0][1] == 0 and all(a < b for (_, a), (_, b) in zip(got, got[1:])), f"{what}: {u} invalid"
            assert all(0 <= w < W for w, _ in got) and got[-1][1] < len(seqs[u])
            lp = segmentation_logp(seqs[u], got, pi, A, B, pen)
            assert abs(lp - osc[k]) <= RTOL * abs(osc[k]) + 1e-300, f"{what}: utterance {u} near-tie scores {lp} vs {osc[k]}"
    return n_near


def run(seqs, N, M, pi, A, B, pen=0.0, **kw):
    obs, offsets = pack(seqs)
    return engine.decode_words(obs, offsets, N, M, pi, A, B, log_penalty=pen, **kw)


@pytest.mark.parametrize("N", [3, 4, 5, 8, 16, 32])
@pytest.mark.parametrize("ltr", [True, False])
def test_states_against_oracle(N, ltr, family):
    rng = np.random.default_rng(100 * N + ltr)
    W, M = (10 if N <= 16 else 4), 32
    pi, A, B = make_models(rng, W, N, M, ltr)
    seqs = make_corpus(rng, 120, M, long_T=3000 if N in (4, 16) else None)
    check_against_oracle(seqs, pi, A, B, -2.0, run(seqs, N, M, pi, A, B, -2.0), f"N={N} ltr={ltr}")


@pytest.mark.parametrize("W", [1, 2, 10, 31, 32, 33, 100])
def test_word_counts_against_oracle(W, family):
    rng = np.random.default_rng(W)
    N, M = 4, 64
    pi, A, B = make_models(rng, W, N, M, True)
    seqs = make_corpus(rng, 80 if W < 100 else 30, M)
    check_against_oracle(seqs, pi, A, B, -1.0, run(seqs, N, M, pi, A, B, -1.0), f"W={W}")


@pytest.mark.parametrize("M", [16, 256, 300, 1024])
def test_codebook_sizes_against_oracle(M, family):
    rng = np.random.default_rng(M)
    W, N = 10, 4
    pi, A, B = make_models(rng, W, N, M, True)
    seqs = make_corpus(rng, 100, M)
    check_against_oracle(seqs, pi, A, B, 0.0, run(seqs, N, M, pi, A, B), f"M={M}")


@pytest.mark.parametrize("W,N,M", [(32, 4, 512), (20, 16, 1024), (32, 8, 600)])
def test_log_emission_table_beyond_shared_memory(W, N, M, family):
    """Left-to-right models whose [M][W][N] log-emission table is larger than a CTA's shared memory: the lane-per-word
    kernel reads it from global memory instead of staging it."""
    rng = np.random.default_rng(W * N + M)
    pi, A, B = make_models(rng, W, N, M, True)
    seqs = make_corpus(rng, 150, M, long_T=1000)
    check_against_oracle(seqs, pi, A, B, -3.0, run(seqs, N, M, pi, A, B, -3.0), f"W={W} N={N} M={M}")


@pytest.mark.parametrize("pen", [0.0, -20.0, 5.0])
@pytest.mark.parametrize("ltr", [True, False])
def test_penalties_and_structural_zeros(pen, ltr, family):
    rng = np.random.default_rng(int(abs(pen)) + 7 * ltr)
    W, N, M = 6, 5, 24
    pi, A, B = make_models(rng, W, N, M, ltr, zeros=True)
    seqs = make_corpus(rng, 150, M)
    res = run(seqs, N, M, pi, A, B, pen)
    check_against_oracle(seqs, pi, A, B, pen, res, f"pen={pen} ltr={ltr}")


def test_impossible_utterances(family):
    rng = np.random.default_rng(3)
    W, N, M = 3, 4, 8
    pi, A, B = make_models(rng, W, N, M, True)
    B[:, :, 5] = 0.0  # codeword 5 cannot be emitted by any word
    B[:, N - 1, 6] = 0.0  # no word can end on codeword 6
    seqs = make_corpus(rng, 60, M)
    seqs[3] = np.array([1, 5, 2])
    seqs[4] = np.array([0, 1, 6])
    seqs[5] = np.array([6])
    score, seg_off, _, _ = res = run(seqs, N, M, pi, A, B, -1.0)
    assert np.isneginf(score[[3, 4, 5]]).all() and (np.diff(seg_off)[[3, 4, 5]] == 0).all()
    check_against_oracle(seqs, pi, A, B, -1.0, res, "impossible")


@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.uint32, np.uint64])
def test_codeword_widths(dtype, family):
    rng = np.random.default_rng(np.dtype(dtype).itemsize)
    W, N, M = 5, 4, 200
    pi, A, B = make_models(rng, W, N, M, True)
    seqs = make_corpus(rng, 90, M)
    obs, offsets = pack(seqs, dtype)
    res = engine.decode_words(obs, offsets, N, M, pi, A, B, log_penalty=-3.0)
    check_against_oracle(seqs, pi, A, B, -3.0, res, f"{np.dtype(dtype).name}")


def test_device_codewords_and_slice(family):
    rng = np.random.default_rng(11)
    W, N, M = 7, 4, 64
    pi, A, B = make_models(rng, W, N, M, True)
    seqs = make_corpus(rng, 120, M)
    obs, offsets = pack(seqs, np.int32)
    d = torch.from_numpy(obs.astype(np.int32)).cuda()
    torch.cuda.synchronize()
    full = engine.decode_words(None, offsets, N, M, pi, A, B, -2.0, obs_dev_ptr=d.data_ptr(), idx_bytes=4)
    check_against_oracle(seqs, pi, A, B, -2.0, full, "device")
    lo = 40  # utterances [40, 120): offsets[0] > 0, the pointer still names the whole buffer
    part = engine.decode_words(None, offsets[lo:], N, M, pi, A, B, -2.0, obs_dev_ptr=d.data_ptr(), idx_bytes=4)
    check_against_oracle(seqs[lo:], pi, A, B, -2.0, part, "device slice")
    assert np.array_equal(part[0], full[0][lo:])


def test_score_only_is_bit_identical(family):
    rng = np.random.default_rng(13)
    for N, ltr in ((4, True), (6, False), (16, True)):
        W, M = 9, 40
        pi, A, B = make_models(rng, W, N, M, ltr, zeros=True)
        seqs = make_corpus(rng, 200, M, long_T=500)
        full = run(seqs, N, M, pi, A, B, -4.0)
        only = run(seqs, N, M, pi, A, B, -4.0, want_segments=False)
        assert only[1] is None and only[2] is None and only[3] is None
        assert np.array_equal(full[0], only[0]), (N, ltr)


def test_error_codes():
    W, N, M = 2, 4, 16
    rng = np.random.default_rng(0)
    pi, A, B = make_models(rng, W, N, M, True)
    obs, offsets = pack([np.array([1, 2, 16]), np.array([3])], np.uint8)
    with pytest.raises(IndexError):  # HMMB_ERR_RANGE
        engine.decode_words(obs, offsets, N, M, pi, A, B)
    obs, offsets = pack([np.array([1, 2]), np.array([], np.int64), np.array([3])], np.uint8)
    with pytest.raises(IndexError):  # HMMB_ERR_EMPTY
        engine.decode_words(obs, offsets, N, M, pi, A, B)
    lib = _lib.load()
    obs, offsets = pack([np.array([1, 2, 3])], np.uint8)
    score = np.empty(1)
    seg_off = np.empty(2, np.int64)
    seg = np.empty(3, np.int32)
    P = _lib.ptr

    def call(W_=W, N_=N, M_=M, pen=0.0, pi_=pi, word=seg, start=seg):
        return lib.hmmb_decode_words(P(obs), 1, 0, P(offsets), 1, W_, N_, M_, P(pi_), P(A), P(B), pen, P(score),
                                     P(seg_off), P(word), P(start))

    assert call() == 0
    for pen in (float("inf"), float("-inf"), float("nan")):
        assert call(pen=pen) == _lib.ERR_ARG
    assert call(W_=0) == _lib.ERR_ARG and call(W_=65536) == _lib.ERR_ARG
    assert call(pi_=None) == _lib.ERR_ARG
    assert call(start=None) == _lib.ERR_ARG
    assert call(N_=33) == _lib.ERR_UNSUPPORTED and call(M_=65537) == _lib.ERR_UNSUPPORTED


def test_generic_bound(family):
    """W * N = 8192 states decode; one word more is HMMB_ERR_UNSUPPORTED."""
    rng = np.random.default_rng(17)
    N, M = 16, 32
    W = 8192 // N
    pi, A, B = make_models(rng, W, N, M, True)
    seqs = make_corpus(rng, 6, M, tmax=25)
    check_against_oracle(seqs, pi, A, B, -1.0, run(seqs, N, M, pi, A, B, -1.0), "W*N=8192")
    pi2, A2, B2 = make_models(rng, W + 1, N, M, True)
    with pytest.raises(_lib.HmmbError) as ei:
        run(seqs, N, M, pi2, A2, B2)
    assert ei.value.code == _lib.ERR_UNSUPPORTED


def test_force_dense_a_on_bidiagonal_models(monkeypatch):
    rng = np.random.default_rng(19)
    W, N, M = 10, 4, 256
    pi, A, B = make_models(rng, W, N, M, True)
    seqs = make_corpus(rng, 300, M, tmax=400)
    base = run(seqs, N, M, pi, A, B, -5.0)
    monkeypatch.setenv("HMMB_FORCE_DENSE_A", "1")
    dense = run(seqs, N, M, pi, A, B, -5.0)
    assert_close(dense[0], base[0], "dense-A score")
    for x, y in zip(base[1:], dense[1:]):
        assert np.array_equal(x, y)


def word_strings(rng, corpus, n, kmax=6):
    strings, truth = [], []
    W = len(corpus)
    for _ in range(n):
        ws = rng.integers(0, W, size=int(rng.integers(1, kmax + 1)))
        strings.append(np.concatenate([corpus[w][int(rng.integers(0, len(corpus[w])))] for w in ws]))
        truth.append(ws.tolist())
    return strings, truth


def test_scale_100k_utterances(family):
    """100 000 strings of 1-6 words of ~100 frames each against 10 word models; 2 000 utterances (the first, the last
    and random ones) are checked against the oracle."""
    rng = np.random.default_rng(23)
    W, N, M = 10, 4, 256
    pi, A, B = make_models(rng, W, N, M, True)
    pool = [synthetic.clustered_sequences(rng, 50, N, M, 80, 120, shift=7 * w) for w in range(W)]
    seqs, _ = word_strings(rng, pool, 100_000)
    res = run(seqs, N, M, pi, A, B, -10.0)
    sample = np.unique(np.concatenate([[0, len(seqs) - 1], rng.choice(len(seqs), 1998, replace=False)]))
    check_against_oracle(seqs, pi, A, B, -10.0, res, "scale", sample=sample)


# The oracle's own trainer (oracle.hmm_oracle.hmm_training, 20 iterations) and decoder (oracle.words_oracle), computed
# once on the CPU, get every one of these 300 strings right at log_penalty -50 (0.85 at 0, 0.93 at -20)
E2E_FLOOR = 0.97


def test_end_to_end_digit_strings():
    W, N, M = 10, 4, 256
    train = synthetic.word_corpus(21, W, 40)
    held = synthetic.word_corpus(22, W, 20)
    obs, offsets, wos = synthetic.pack_corpus(train, M)
    p0, A0, B0 = engine.default_init(N, M)
    pi, A, B, _, _ = engine.bw_fit(obs, offsets, wos, W, N, M, np.tile(p0, (W, 1)), np.tile(A0, (W, 1, 1)),
                                   np.tile(B0, (W, 1, 1)), max_iterations=20)
    names = [f"digit{w}" for w in range(W)]
    hmms = [HMMTrained(states=N, symbols=M, A=A[w], B=B[w], Pi=pi[w], word=names[w]) for w in range(W)]
    strings, truth = word_strings(np.random.default_rng(23), held, 300)
    scores, words = hmm_testing.recognize_connected(strings, hmms, log_penalty=-50.0)
    osc, ooff, oword, ostart, omarg = decode_words_batch(strings, [(A[w], B[w], pi[w]) for w in range(W)], -50.0)
    assert_close(scores, osc, "end-to-end score")
    got = [[w for w, _, _ in ws] for ws in words]
    want = [[names[w] for w in oword[ooff[u]:ooff[u + 1]]] for u in range(len(strings))]
    assert got == want
    for u, ws in enumerate(words):  # the segments tile the utterance
        assert ws[0][1] == 0 and ws[-1][2] == len(strings[u]) - 1
        assert all(a[2] + 1 == b[1] for a, b in zip(ws, ws[1:]))
    acc = np.mean([g == [names[w] for w in t] for g, t in zip(got, truth)])
    assert acc >= E2E_FLOOR, acc

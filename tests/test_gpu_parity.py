"""Parity of the CUDA path (through the C ABI) with the reference's golden vectors and with
the CPU oracle on seeded inputs.  Needs a GPU: run with ``-m gpu`` on the B200 box.

Tolerances (BASELINE.md §4): indices bit-exact; A/B/pi and per-iteration LL within
|x - ref| <= 1e-9*|ref| + 1e-30; zero pattern of A/pi and the set of floored B entries equal.
"""

import numpy as np
import pytest

from helpers import assert_close, assert_same_support, floored_set, load_golden, split_corpus
from hmm_training_b200 import engine, synthetic
from oracle import hmm_oracle as O
from oracle import vq_oracle

pytestmark = pytest.mark.gpu

BW_CASES = ["bw_c1_clustered_s0_it10", "bw_uniform_s1_it3", "bw_clustered_s2_it1", "bw_converge_eps",
            "bw_warm_n6_m32", "bw_structural_zeros", "bw_ltr_n16_m64", "bw_ltr_n8_m24", "bw_word_without_sequences"]


@pytest.fixture(params=["special", "generic"])
def kernel_family(request, monkeypatch):
    """N=4 goes through the one-sequence-per-thread kernels by default; HMMB_FORCE_GENERIC
    routes the same inputs through the lanes-per-sequence kernels."""
    if request.param == "generic":
        monkeypatch.setenv("HMMB_FORCE_GENERIC", "1")
    else:
        monkeypatch.delenv("HMMB_FORCE_GENERIC", raising=False)
    return request.param


def _init_for(g, W, N, M):
    if "pi0" in g:
        return g["pi0"], g["A0"], g["B0"]
    pi, A, B = engine.default_init(N, M)
    return np.tile(pi, (W, 1)), np.tile(A, (W, 1, 1)), np.tile(B, (W, 1, 1))


def _check_bw(name, g, pi, A, B, hist, iters, N, M):
    W = A.shape[0]
    assert np.array_equal(iters, g["iters"]), f"{name}: iteration counts {iters} vs {g['iters']}"
    for w in range(W):
        it = int(iters[w])
        assert_close(hist[w, :it], g["ll_hist"][w, :it], f"{name} w{w} ll")
        assert_close(A[w], g["A"][w], f"{name} w{w} A")
        assert_close(pi[w], g["pi"][w], f"{name} w{w} pi")
        assert_close(B[w], g["B"][w], f"{name} w{w} B")
        assert_same_support(A[w], g["A"][w], f"{name} w{w} A")
        assert_same_support(pi[w], g["pi"][w], f"{name} w{w} pi")
        assert np.array_equal(floored_set(B[w], M), floored_set(g["B"][w], M)), f"{name} w{w}: floored B set"


@pytest.mark.parametrize("name", BW_CASES)
def test_baum_welch_matches_reference_golden(name, kernel_family):
    g = load_golden(name)
    N, M = int(g["N"]), int(g["M"])
    W = g["A"].shape[0]
    pi0, A0, B0 = _init_for(g, W, N, M)
    pi, A, B, hist, iters = engine.bw_fit(g["obs"], g["offsets"], g["word_of_seq"], W, N, M, pi0, A0, B0,
                                          epsilon=float(g["epsilon"]), max_iterations=int(g["max_iterations"]))
    _check_bw(name, g, pi, A, B, hist, iters, N, M)


@pytest.mark.parametrize("name", ["bw_ltr_n16_m64", "bw_ltr_n8_m24"])
def test_left_to_right_kernels_match_reference_golden(name, monkeypatch):
    """The two goldens the reference produced for bidiagonal models with 16 / 8 states (oracle/make_golden.py,
    case_bw_ltr) run on the one-sequence-per-thread left-to-right kernels — asserted, not assumed."""
    monkeypatch.delenv("HMMB_NO_LTR", raising=False); monkeypatch.delenv("HMMB_FORCE_GENERIC", raising=False)
    g = load_golden(name)
    N, M = int(g["N"]), int(g["M"])
    W = g["A"].shape[0]
    iters_max = int(g["max_iterations"])
    with engine.BaumWelch(g["obs"], g["offsets"], g["word_of_seq"], W, N, M) as bw:
        bw.set_params(g["pi0"], g["A0"], g["B0"])
        assert bw.kernel_family() == "left_to_right"
        bw.iterate(iters_max, float(g["epsilon"]), iters_max)
        pi, A, B = bw.params()
        hist, iters = bw.history(iters_max)
    _check_bw(name, g, pi, A, B, hist, iters, N, M)


def test_baum_welch_shuffled_sequence_order(kernel_family):
    """The library sorts sequences by (word, length); interleaved / shuffled input must give
    the same models (sum order changes only at the 1e-16 level), whatever the width of the codewords."""
    g = load_golden("bw_uniform_s1_it3")
    N, M = int(g["N"]), int(g["M"])
    corpus = split_corpus(g)
    rng = np.random.default_rng(0)
    seqs = [(w, s) for w, word in enumerate(corpus) for s in word]
    perm = rng.permutation(len(seqs))
    lens = np.array([len(seqs[i][1]) for i in perm])
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    wos = np.array([seqs[i][0] for i in perm], dtype=np.int32)
    W = len(corpus)
    pi0, A0, B0 = _init_for(g, W, N, M)
    for dt in (np.int64, np.uint32):  # 8- and 4-byte codewords
        obs = np.concatenate([seqs[i][1] for i in perm]).astype(dt)
        pi, A, B, hist, iters = engine.bw_fit(obs, offsets, wos, W, N, M, pi0, A0, B0, max_iterations=3)
        _check_bw(f"shuffled {np.dtype(dt).name}", g, pi, A, B, hist, iters, N, M)


@pytest.mark.parametrize("N,M,T", [(4, 256, 200), (4, 300, 37), (3, 20, 15), (8, 64, 40), (16, 1024, 50), (32, 128, 12)])
def test_baum_welch_matches_oracle_seeded(N, M, T):
    """Seeded synthetic data, random dense + default init, against the numpy oracle."""
    rng = np.random.default_rng(N * 1000 + M)
    W, S = 3, 40
    corpus = [synthetic.clustered_sequences(rng, S, N=N, M=M, tmin=max(1, T - 5), tmax=T + 5, shift=7 * w,
                                            spread=max(2, M // (2 * N))) for w in range(W)]
    obs, offsets, wos = synthetic.pack_corpus(corpus, M)
    pi0 = np.zeros((W, N)); A0 = np.zeros((W, N, N)); B0 = np.zeros((W, N, M))
    for w in range(W):
        if w == 0:
            pi0[w], A0[w], B0[w] = engine.default_init(N, M)
        else:
            pi0[w] = rng.dirichlet(np.ones(N)); A0[w] = rng.dirichlet(np.ones(N), size=N)
            B0[w] = rng.dirichlet(np.ones(M), size=N)
    iters_max = 4
    pi, A, B, hist, iters = engine.bw_fit(obs, offsets, wos, W, N, M, pi0, A0, B0, max_iterations=iters_max)
    for w in range(W):
        Ao, Bo, pio, h, it = O.hmm_training(corpus[w], N=N, M=M, max_iterations=iters_max,
                                            init=(pi0[w], A0[w], B0[w]), return_history=True)
        assert it == iters[w]
        assert_close(hist[w, :it], h, f"N{N} M{M} w{w} ll")
        assert_close(A[w], Ao, f"N{N} M{M} w{w} A")
        assert_close(B[w], Bo, f"N{N} M{M} w{w} B")
        assert_close(pi[w], pio, f"N{N} M{M} w{w} pi")
        assert_same_support(A[w], Ao)
        assert np.array_equal(floored_set(B[w], M), floored_set(Bo, M))


@pytest.mark.parametrize("N,M,T,S,family", [
    (4, 256, 6000, 3, "n4_left_to_right"),   # long horizons: thousands of rescales, per-state error bound
    (16, 1024, 6000, 3, "left_to_right"),    # the same horizon on the N = 16 kernels (config 4's shape): the scalar error
    (8, 512, 6000, 3, "left_to_right"),      # bound is seeded only where a denormal is born, so nothing is handed over
    (4, 512, 40, 40, "n4_left_to_right"),    # the largest alphabet the warp-private count tables hold
    (4, 513, 40, 40, "generic"),             # one more codeword: lanes-per-state kernels, u16 symbols
    (5, 4096, 60, 20, "generic"),            # wide alphabet, odd state count
    (16, 1400, 30, 40, "left_to_right"),     # B^T of 175 KB: the largest the left-to-right kernels keep in shared memory
    (16, 1700, 30, 40, "generic"),           # beyond it
])
def test_baum_welch_size_limits_match_oracle(N, M, T, S, family):
    """Maximum sizes of each kernel family (and the first size past each limit) against the numpy oracle,
    default left-to-right init, 3 iterations."""
    rng = np.random.default_rng(N * 100003 + M * 17 + T)
    W = 2
    corpus = [synthetic.clustered_sequences(rng, S, N=N, M=M, tmin=max(1, T - T // 8), tmax=T, shift=7 * w,
                                            spread=max(2, M // (2 * N))) for w in range(W)]
    obs, offsets, wos = synthetic.pack_corpus(corpus, M)
    pi0, A0, B0 = engine.default_init(N, M)
    init = (np.tile(pi0, (W, 1)), np.tile(A0, (W, 1, 1)), np.tile(B0, (W, 1, 1)))
    with engine.BaumWelch(obs, offsets, wos, W, N, M) as bw:
        bw.set_params(*init)
        assert bw.kernel_family() == family
        bw.iterate(3, 1e-6, 3)
        pi, A, B = bw.params()
        hist, iters = bw.history(3)
        exact_passes, handovers = bw.diagnostics()
    assert (exact_passes, handovers) == (0, 0)  # the per-state error bound keeps even T = 6000 on the fast path
    # At T = 6000 the ORACLE's log-space arithmetic (like the reference's) carries ~1e-9 of rounding noise: log alpha
    # ~ -2e4 is held to 2e-12 absolute per operation and the recursion is 6000 steps deep, so the small entries of B
    # of two correct evaluations differ by several 1e-9 (the exact log-space kernel differs from the oracle by as much).
    rtol = 1e-9 if T < 1000 else 1e-7
    for w in range(W):
        Ao, Bo, pio, h, it = O.hmm_training(corpus[w], N=N, M=M, max_iterations=3, init=(pi0, A0, B0), return_history=True)
        assert it == iters[w]
        assert_close(hist[w, :it], h, f"N{N} M{M} T{T} w{w} ll", rtol=rtol)
        assert_close(A[w], Ao, f"N{N} M{M} T{T} w{w} A", rtol=rtol)
        assert_close(B[w], Bo, f"N{N} M{M} T{T} w{w} B", rtol=rtol)
        assert_close(pi[w], pio, f"N{N} M{M} T{T} w{w} pi", rtol=rtol)
        assert_same_support(A[w], Ao)
        assert np.array_equal(floored_set(B[w], M), floored_set(Bo, M))


def _ltr_init(rng, W, N, M, kind):
    """Left-to-right (upper-bidiagonal A) initial models: 'default' = the generalised reference
    defaults, 'random' = random self/next probabilities and random dense B, 'zeros' = B with
    exact zeros and pi concentrated on state 0 (forces the careful / masked steps)."""
    pi0 = np.zeros((W, N)); A0 = np.zeros((W, N, N)); B0 = np.zeros((W, N, M))
    for w in range(W):
        if kind == "default":
            pi0[w], A0[w], B0[w] = engine.default_init(N, M)
            continue
        stay = rng.uniform(0.3, 0.9, size=N)
        for i in range(N - 1):
            A0[w, i, i] = stay[i]; A0[w, i, i + 1] = 1 - stay[i]
        A0[w, N - 1, N - 1] = 1.0
        B0[w] = rng.dirichlet(np.ones(M), size=N)
        if kind == "zeros":
            pi0[w, 0] = 1.0
            B0[w][rng.random((N, M)) < 0.15] = 0.0
            B0[w, :, 0] = 1e-3  # keep at least one symbol every state can emit
        else:
            pi0[w] = rng.dirichlet(np.ones(N))
    return pi0, A0, B0


@pytest.mark.parametrize("N,M,kind", [(16, 1024, "default"), (16, 1024, "random"), (16, 300, "zeros"),
                                      (8, 64, "default"), (8, 2048, "random"), (8, 40, "zeros")])
def test_baum_welch_left_to_right_kernels(N, M, kind, monkeypatch):
    """N = 8 / 16 with upper-bidiagonal A goes through the one-sequence-per-thread left-to-right
    kernels (bwltr_kernels.cuh: TMA bulk-reduce count accumulation); checked against the numpy
    oracle and against the generic lanes-per-state kernels on ragged input (T from 1 up)."""
    rng = np.random.default_rng(N * 7 + M)
    W = 3
    corpus = []
    for w in range(W):
        seqs = synthetic.clustered_sequences(rng, 41 + 3 * w, N=N, M=M, tmin=3, tmax=70, shift=5 * w,
                                             spread=max(2, M // (2 * N)))
        seqs[0] = seqs[0][:1]   # T == 1
        seqs[1] = seqs[1][:2]
        if kind == "zeros":
            seqs[2] = np.zeros(9, np.int64)  # only symbol 0: possible under every state
        corpus.append(seqs)
    obs, offsets, wos = synthetic.pack_corpus(corpus, M)
    pi0, A0, B0 = _ltr_init(rng, W, N, M, kind)
    iters_max = 4
    monkeypatch.delenv("HMMB_NO_LTR", raising=False)
    with engine.BaumWelch(obs, offsets, wos, W, N, M) as bw:
        bw.set_params(pi0, A0, B0)
        assert bw.kernel_family() == "left_to_right"
        bw.iterate(iters_max, 1e-6, iters_max)
        pi, A, B = bw.params()
        hist, iters = bw.history(iters_max)
        ll_seq = bw.seq_ll()
    for w in range(W):
        Ao, Bo, pio, h, it = O.hmm_training(corpus[w], N=N, M=M, max_iterations=iters_max,
                                            init=(pi0[w], A0[w], B0[w]), return_history=True)
        assert it == iters[w]
        assert_close(hist[w, :it], h, f"N{N} M{M} w{w} ll")
        assert_close(A[w], Ao, f"N{N} M{M} w{w} A")
        assert_close(B[w], Bo, f"N{N} M{M} w{w} B")
        assert_close(pi[w], pio, f"N{N} M{M} w{w} pi")
        assert_same_support(A[w], Ao); assert_same_support(pi[w], pio)
        assert np.array_equal(floored_set(B[w], M), floored_set(Bo, M))
    monkeypatch.setenv("HMMB_NO_LTR", "1")
    with engine.BaumWelch(obs, offsets, wos, W, N, M) as bw:
        bw.set_params(pi0, A0, B0)
        assert bw.kernel_family() == "generic"
        bw.iterate(iters_max, 1e-6, iters_max)
        pig, Ag, Bg = bw.params()
        llg = bw.seq_ll()
    assert_close(A, Ag, "ltr vs generic A"); assert_close(B, Bg, "ltr vs generic B"); assert_close(pi, pig, "ltr vs generic pi")
    assert_close(ll_seq, llg, "ltr vs generic per-sequence LL")


def test_left_to_right_kernels_at_config4_shape(monkeypatch):
    """BASELINE config 4's shape at a size the generic kernels still finish quickly (12 words x 300
    sequences x T = 200, N = 16, M = 1024, 6 iterations — trained B rows then hold values down to the
    1e-20 floor and far below): the left-to-right kernels must agree with the lanes-per-state kernels
    to 1e-9, keep rows stochastic, and not decrease the convergence statistic."""
    N, M, W, S, T = 16, 1024, 12, 300, 200
    obs, offsets, wos = synthetic.fixed_length_codewords(11, W, S, T, N, M)
    pi0, A0, B0 = engine.default_init(N, M)
    init = (np.tile(pi0, (W, 1)), np.tile(A0, (W, 1, 1)), np.tile(B0, (W, 1, 1)))
    res = {}
    for fam, env in (("left_to_right", None), ("generic", "1")):
        if env:
            monkeypatch.setenv("HMMB_NO_LTR", env)
        else:
            monkeypatch.delenv("HMMB_NO_LTR", raising=False)
        with engine.BaumWelch(obs, offsets, wos, W, N, M) as bw:
            bw.set_params(*init)
            assert bw.kernel_family() == fam
            bw.iterate(6, -1.0, 6)
            res[fam] = bw.params() + bw.history(6) + (bw.seq_ll(), bw.diagnostics())
    a, b = res["left_to_right"], res["generic"]
    for x, y, what in zip(a[:4], b[:4], ("pi", "A", "B", "ll history")):
        assert_close(x, y, f"left_to_right vs generic {what}")
    assert_close(a[5], b[5], "per-sequence LL of the last E-step")
    assert np.array_equal(a[4], b[4]) and np.all(a[4] == 6)
    pi, A, B, hist = a[:4]
    assert np.allclose(pi.sum(axis=1), 1) and np.allclose(A.sum(axis=2), 1) and np.allclose(B.sum(axis=2), 1)
    assert np.all(np.diff(hist, axis=1) > -1e-6)
    assert np.array_equal(A == 0, np.tile(A0 == 0, (W, 1, 1)))  # the left-to-right support is preserved
    assert a[6] == b[6] == (0, 0)  # neither family needed the exact log-space path on this data


@pytest.mark.parametrize("N", [4, 6, 8])
def test_training_from_degenerate_initial_models(N):
    """Warm start from what the reference saves for a word without sequences (pi = NaN, A = 0, B = 0), from a model with
    one NaN and from one with negative emission entries: safe_log (hmm_training.py:29-39) turns everything that is not > 0
    into -inf, so the reference trains on (checked against it on the CPU: the oracle agrees to 1e-14 on exactly these
    initial models); so must the kernels — no NaN may leak into the other words or the statistics."""
    rng = np.random.default_rng(70 + N)
    M, W = 12, 3
    word = [rng.integers(0, M, size=int(rng.integers(2, 15))) for _ in range(6)]
    corpus = [word, word, word]
    obs, offsets, wos = synthetic.pack_corpus(corpus, M)
    pi0 = rng.dirichlet(np.ones(N), size=W); A0 = rng.dirichlet(np.ones(N), size=(W, N)); B0 = rng.dirichlet(np.ones(M), size=(W, N))
    pi0[0] = np.nan; A0[0] = 0.0; B0[0] = 0.0
    pi0[1, 0] = np.nan
    B0[2, 0] = -B0[2, 0]
    pi, A, B, hist, iters = engine.bw_fit(obs, offsets, wos, W, N, M, pi0, A0, B0, epsilon=-1.0, max_iterations=3)
    for w in range(W):
        Ao, Bo, pio, h, it = O.hmm_training(word, N=N, M=M, epsilon=-1.0, max_iterations=3, init=(pi0[w], A0[w], B0[w]),
                                            return_history=True)
        assert it == iters[w]
        assert_close(hist[w, :it], h, f"N{N} w{w} ll"); assert_close(A[w], Ao, f"N{N} w{w} A")
        assert_close(B[w], Bo, f"N{N} w{w} B"); assert_close(pi[w], pio, f"N{N} w{w} pi")
    assert np.isneginf(hist[0, :3]).all() and np.isfinite(hist[1:, :3]).all()


def test_baum_welch_is_deterministic():
    g = load_golden("bw_clustered_s2_it1")
    N, M, W = 4, 256, 3
    pi0, A0, B0 = _init_for(g, W, N, M)
    a = engine.bw_fit(g["obs"], g["offsets"], g["word_of_seq"], W, N, M, pi0, A0, B0, max_iterations=3)
    b = engine.bw_fit(g["obs"], g["offsets"], g["word_of_seq"], W, N, M, pi0, A0, B0, max_iterations=3)
    for x, y in zip(a, b):
        assert np.array_equal(x, y, equal_nan=True)  # N=4 path has no atomics: bitwise reproducible


def test_baum_welch_errors():
    pi0, A0, B0 = (x[None] for x in engine.default_init(4, 256))
    with pytest.raises(IndexError):  # T == 0 (reference: IndexError at hmm_training.py:376)
        engine.bw_fit(np.array([1, 2, 3], np.uint8), np.array([0, 3, 3]), np.array([0, 0], np.int32), 1, 4, 256,
                      pi0, A0, B0, max_iterations=1)
    with pytest.raises(IndexError):  # codeword >= M
        pi1, A1, B1 = (x[None] for x in engine.default_init(4, 16))
        engine.bw_fit(np.array([1, 200, 3], np.uint8), np.array([0, 3]), np.array([0], np.int32), 1, 4, 16,
                      pi1, A1, B1, max_iterations=1)


def test_scoring_matches_reference_golden(kernel_family):
    g = load_golden("score_c1")
    ll, arg = engine.score(g["obs"], g["offsets"], 4, 256, g["pi"], g["A"], g["B"])
    assert_close(ll, g["ll"], "score ll")
    assert np.array_equal(arg, O.argmax_first(g["ll"]))


@pytest.mark.parametrize("name", ["score_ltr_n16_m64", "score_ltr_n8_m24"])
def test_scoring_left_to_right_matches_reference_golden(name, kernel_family):
    """Recognition with bidiagonal 16- / 8-state models against the reference's own numbers (k_scoreL by default, the
    generic scorer under HMMB_FORCE_GENERIC), -inf pattern included."""
    g = load_golden(name)
    ll, arg = engine.score(g["obs"], g["offsets"], int(g["N"]), int(g["M"]), g["pi"], g["A"], g["B"])
    assert np.array_equal(np.isneginf(ll), np.isneginf(g["ll"]))
    assert_close(ll, g["ll"], "score ll")
    assert np.array_equal(arg, O.argmax_first(g["ll"]))


@pytest.mark.parametrize("N", [4, 6, 8, 16])
def test_scoring_against_degenerate_models(N):
    """What training returns for a word without sequences (pi = NaN, A = 0, B = 0: tests/golden/
    bw_word_without_sequences.npz), a model with negative emission entries and one with a single NaN: the reference's
    safe_log (hmm_testing.py:66-68) maps everything that is not > 0 to -inf, NaN included, so such a model scores -inf and
    is never recognised; every scorer family must say the same and must not let a NaN through."""
    rng = np.random.default_rng(40 + N)
    M, W = 16, 4
    U = [rng.integers(0, M, size=int(rng.integers(1, 12))) for _ in range(9)]
    obs = np.concatenate(U)
    off = np.concatenate([[0], np.cumsum([len(u) for u in U])]).astype(np.int64)
    pi = rng.dirichlet(np.ones(N), size=W); A = rng.dirichlet(np.ones(N), size=(W, N)); B = rng.dirichlet(np.ones(M), size=(W, N))
    if N in (8, 16):  # bidiagonal: the left-to-right scorer
        A = np.zeros((W, N, N))
        for i in range(N):
            A[:, i, i] = 0.6 if i + 1 < N else 1.0
            if i + 1 < N:
                A[:, i, i + 1] = 0.4
    pi[1] = np.nan; A[1] = 0.0; B[1] = 0.0
    B[2] = -B[2]
    pi[3, 0] = np.nan
    ll, arg = engine.score(obs, off, N, M, pi, A, B)
    want = O.score_batch(U, [(A[w], B[w], pi[w]) for w in range(W)])
    assert not np.isnan(ll).any()
    assert np.array_equal(np.isneginf(ll), np.isneginf(want)) and np.isneginf(ll[:, 1:3]).all()
    assert_close(ll, want, "score against degenerate models")
    assert np.array_equal(arg, O.argmax_first(want))


@pytest.mark.parametrize("N,M", [(4, 256), (6, 32), (16, 1024), (4, 512), (4, 513), (5, 4096), (32, 64), (1, 7)])
def test_scoring_matches_oracle_with_structural_zeros(N, M):
    rng = np.random.default_rng(N + M)
    W, U = 5, 70
    pi = rng.dirichlet(np.ones(N), size=W); A = rng.dirichlet(np.ones(N), size=(W, N))
    B = rng.dirichlet(np.ones(M), size=(W, N))
    pi[1] = 0; pi[1, 0] = 1.0
    A[1] = np.triu(A[1]); A[1] /= A[1].sum(axis=1, keepdims=True)
    B[2, :, : M // 2] = 0.0  # model 2 cannot emit the lower half of the codebook -> many -inf
    B[3, 0, :] = 0.0
    seqs = [rng.integers(0, M, size=int(rng.integers(1, 60))) for _ in range(U)]
    seqs[5] = rng.integers(M // 2, M, size=30)  # possible under model 2
    obs, offsets = np.concatenate(seqs), np.concatenate([[0], np.cumsum([len(s) for s in seqs])])
    ll, arg = engine.score(obs.astype(np.int64), offsets, N, M, pi, A, B)
    ref = O.score_batch(seqs, [(A[w], B[w], pi[w]) for w in range(W)])
    assert_close(ll, ref, "score")
    assert np.array_equal(np.isneginf(ll), np.isneginf(ref))
    assert np.isneginf(ll[:, 2]).sum() > U // 2 and np.isfinite(ll[5, 2])
    assert np.array_equal(arg, O.argmax_first(ref))
    allbad = engine.score(np.zeros(4, np.uint8), np.array([0, 4]), N, M, pi[2:3], A[2:3], B[2:3])
    assert allbad[1][0] == -1 and np.isneginf(allbad[0]).all()  # "unknown" (hmm_testing.py:161)


@pytest.mark.parametrize("N,M,kind", [(16, 1024, "random"), (16, 200, "zeros"), (8, 64, "random"), (8, 300, "zeros")])
def test_scoring_left_to_right_kernels(N, M, kind, monkeypatch):
    """Recognition with upper-bidiagonal models at N = 8 / 16 runs k_scoreL (one utterance per
    thread); checked against the oracle and against the generic lanes-per-state scorer."""
    rng = np.random.default_rng(3 * N + M)
    W, U = 5, 150
    pi, A, B = _ltr_init(rng, W, N, M, kind)
    seqs = [rng.integers(0, M, size=int(rng.integers(1, 90))) for _ in range(U)]
    seqs += synthetic.clustered_sequences(rng, 40, N=N, M=M, tmin=20, tmax=60, spread=max(2, M // (2 * N)))
    if kind == "zeros":
        seqs[3] = np.zeros(25, np.int64)  # symbol 0 is emitted by every state: finite under every model
    obs, offsets = np.concatenate(seqs), np.concatenate([[0], np.cumsum([len(q) for q in seqs])])
    dt = np.uint8 if M <= 256 else np.uint16
    monkeypatch.delenv("HMMB_NO_LTR", raising=False)
    ll, arg = engine.score(obs.astype(dt), offsets, N, M, pi, A, B)
    ref = O.score_batch(seqs, [(A[w], B[w], pi[w]) for w in range(W)])
    assert_close(ll, ref, "ltr score")
    assert np.array_equal(np.isneginf(ll), np.isneginf(ref))
    # the all-zeros utterance scores 25*log(1e-3) under EVERY model (rows of A sum to 1): an exact tie
    # on paper, decided by the last bit — compare the winner only where the runner-up is clearly behind
    top = np.sort(ref, axis=1)[:, ::-1]
    with np.errstate(invalid="ignore"):
        clear = ~(np.abs(top[:, 0] - top[:, 1]) <= 1e-7 * np.abs(top[:, 0]))
    assert clear.sum() >= len(seqs) - 8
    assert np.array_equal(arg[clear], O.argmax_first(ref)[clear])
    assert np.array_equal(arg, O.argmax_first(ll))  # and always the first maximum of our own scores
    if kind == "zeros":
        assert np.isneginf(ref).sum() > U and np.isfinite(ref[3]).all()
    monkeypatch.setenv("HMMB_NO_LTR", "1")
    llg, argg = engine.score(obs.astype(dt), offsets, N, M, pi, A, B)
    assert_close(ll, llg, "ltr vs generic score")
    assert np.array_equal(arg[clear], argg[clear])


@pytest.mark.parametrize("N,M,dense_family", [(4, 64, "n4_dense"), (8, 40, "generic")])
def test_dense_a_switch_in_trainer_scorer_and_decoder(N, M, dense_family, monkeypatch):
    """HMMB_FORCE_DENSE_A=1 treats an upper-bidiagonal A as dense in all three entry points: N = 4 then trains, scores
    and decodes on the dense N = 4 kernels, N = 8 on the lanes-per-state kernels.  Both runs must match the oracle.
    At N = 4 Viterbi only adds and compares, and the terms the bidiagonal kernel skips are -inf, so its results must
    equal the default run's bit for bit.  Scores and trained models come out of different floating-point code in the two
    kernel families and differ in the last bits, so they are held to each other at the parity tolerance."""
    from test_gpu_viterbi import check_against_oracle

    rng = np.random.default_rng(N * 31 + M)
    W = 3
    corpus = [synthetic.clustered_sequences(rng, 40, N=N, M=M, tmin=1, tmax=70, shift=5 * w, spread=max(2, M // (2 * N)))
              for w in range(W)]
    obs, offsets, wos = synthetic.pack_corpus(corpus, M)
    seqs = [s for word in corpus for s in word]
    pi0, A0, B0 = _ltr_init(rng, W, N, M, "random")
    iters_max = 4
    runs = {}
    for dense in (False, True):
        if dense:
            monkeypatch.setenv("HMMB_FORCE_DENSE_A", "1")
        else:
            monkeypatch.delenv("HMMB_FORCE_DENSE_A", raising=False)
        with engine.BaumWelch(obs, offsets, wos, W, N, M) as bw:
            bw.set_params(pi0, A0, B0)
            family = bw.kernel_family()
            bw.iterate(iters_max, 1e-6, iters_max)
            trained = bw.params() + bw.history(iters_max)
        runs[dense] = (family, trained, engine.score(obs, offsets, N, M, pi0, A0, B0),
                       engine.viterbi(obs, offsets, wos, N, M, pi0, A0, B0))
    assert runs[False][0] == ("n4_left_to_right" if N == 4 else "left_to_right")
    family, (pi, A, B, hist, iters), (ll, arg), (vscore, vpath) = runs[True]
    assert family == dense_family
    for w in range(W):
        Ao, Bo, pio, h, it = O.hmm_training(corpus[w], N=N, M=M, max_iterations=iters_max,
                                            init=(pi0[w], A0[w], B0[w]), return_history=True)
        assert it == iters[w]
        assert_close(hist[w, :it], h, f"dense N{N} w{w} ll")
        assert_close(A[w], Ao, f"dense N{N} w{w} A")
        assert_close(B[w], Bo, f"dense N{N} w{w} B")
        assert_close(pi[w], pio, f"dense N{N} w{w} pi")
        assert_same_support(A[w], Ao); assert_same_support(pi[w], pio)
        assert np.array_equal(floored_set(B[w], M), floored_set(Bo, M))
    ref = O.score_batch(seqs, [(A0[w], B0[w], pi0[w]) for w in range(W)])
    assert_close(ll, ref, f"dense N{N} score")
    assert np.array_equal(np.isneginf(ll), np.isneginf(ref))
    assert np.array_equal(arg, O.argmax_first(ll))
    check_against_oracle(seqs, wos, pi0, A0, B0, vscore, vpath, offsets, f"dense N{N} viterbi")
    if N == 4:
        (_, (ll_b, _), (vscore_b, vpath_b)) = runs[False][1:]
        assert np.array_equal(vscore, vscore_b) and np.array_equal(vpath, vpath_b)
        assert_close(ll, ll_b, "dense vs bidiagonal N = 4 scores")
        for x, y, what in zip(runs[True][1], runs[False][1], ("pi", "A", "B", "ll history")):
            assert_close(x[np.isfinite(y)], y[np.isfinite(y)], f"dense vs bidiagonal N = 4 kernels: trained {what}")
        assert np.array_equal(runs[True][1][4], runs[False][1][4])


def _tiny_models(rng, W, N, M):
    """Left-to-right models whose emission rows hold denormal / 1e-300-range / zero entries:
    what saved reference models look like after safe_exp underflow (hmm_training.py:524-526)."""
    pi = np.zeros((W, N)); pi[:, 0] = 1.0
    A = np.zeros((W, N, N))
    for i in range(N):
        A[:, i, i] = 0.7
        A[:, i, min(i + 1, N - 1)] += 0.3
    B = rng.dirichlet(np.ones(M), size=(W, N))
    tiny = np.array([1e-300, 3e-310, 1e-320, 4.9e-324, 0.0, 1e-250])
    for w in range(W):
        for k in range(M):
            if k % 3 != w % 3:
                continue
            keep = rng.integers(0, N)  # one state keeps a normal probability for this symbol
            for j in range(N):
                if j != keep:
                    B[w, j, k] = tiny[rng.integers(0, len(tiny))]
    return pi, A, B


def test_scoring_long_utterances():
    """Utterances of 3000 frames against trained (peaked, 1e-20-floored) left-to-right models, own and foreign:
    k_score4 switches to the per-state error bound above 1000 frames (the scalar bound would hand every such
    utterance to the exact kernel); results against the oracle's log-space forward pass."""
    rng = np.random.default_rng(77)
    N, M, T, S, W = 4, 256, 3000, 3, 3
    corpus = [synthetic.clustered_sequences(rng, S, N=N, M=M, tmin=T - 200, tmax=T, shift=11 * w, spread=24) for w in range(W)]
    obs, offsets, wos = synthetic.pack_corpus(corpus, M)
    pi0, A0, B0 = engine.default_init(N, M)
    pi, A, B, _, _ = engine.bw_fit(obs, offsets, wos, W, N, M, np.tile(pi0, (W, 1)), np.tile(A0, (W, 1, 1)),
                                   np.tile(B0, (W, 1, 1)), max_iterations=3)
    ll, arg = engine.score(obs, offsets, N, M, pi, A, B)
    ref = O.score_batch([u for c in corpus for u in c], [(A[w], B[w], pi[w]) for w in range(W)])
    assert not np.isnan(ll).any()
    assert_close(ll, ref, "long utterances", rtol=1e-8)
    assert np.array_equal(arg, O.argmax_first(ref)) and np.array_equal(arg, wos)


@pytest.mark.parametrize("N,M", [(4, 16), (6, 16)])
def test_scoring_with_denormal_emissions(N, M):
    """Steps whose total probability is ~1e-320 (denormal B on the only live path) must keep
    the reference's log-space precision (exponent-split slow path)."""
    rng = np.random.default_rng(11 + N)
    W, U = 6, 200
    pi, A, B = _tiny_models(rng, W, N, M)
    seqs = [rng.integers(0, M, size=int(rng.integers(1, 40))) for _ in range(U)]
    obs, offsets = np.concatenate(seqs), np.concatenate([[0], np.cumsum([len(s) for s in seqs])])
    ll, arg = engine.score(obs.astype(np.uint8), offsets, N, M, pi, A, B)
    ref = O.score_batch(seqs, [(A[w], B[w], pi[w]) for w in range(W)])
    assert np.isfinite(ref).sum() > 100 and (ref[np.isfinite(ref)] < -700).sum() > 50  # the case is exercised
    assert np.array_equal(np.isneginf(ll), np.isneginf(ref))
    assert_close(ll, ref, "denormal scoring")
    assert np.array_equal(arg, O.argmax_first(ref))


@pytest.mark.parametrize("N,M", [(4, 16), (6, 16)])
def test_training_from_denormal_emissions(N, M):
    rng = np.random.default_rng(5 + N)
    W = 3
    pi0, A0, B0 = _tiny_models(rng, W, N, M)
    corpus = [[rng.integers(0, M, size=int(rng.integers(2, 30))) for _ in range(30)] for _ in range(W)]
    obs, offsets, wos = synthetic.pack_corpus(corpus, M)
    pi, A, B, hist, iters = engine.bw_fit(obs, offsets, wos, W, N, M, pi0, A0, B0, max_iterations=3)
    for w in range(W):
        Ao, Bo, pio, h, it = O.hmm_training(corpus[w], N=N, M=M, max_iterations=3, init=(pi0[w], A0[w], B0[w]),
                                            return_history=True)
        assert it == iters[w]
        assert_close(hist[w, :it], h, f"w{w} ll")
        assert_close(A[w], Ao, f"w{w} A"); assert_close(B[w], Bo, f"w{w} B"); assert_close(pi[w], pio, f"w{w} pi")
        assert_same_support(A[w], Ao); assert_same_support(pi[w], pio)


def test_vq_encode_matches_reference_golden():
    g = load_golden("vq_2000x256")
    idx = engine.vq_encode(g["X"], g["C"])
    assert np.array_equal(idx, g["idx"])


@pytest.mark.parametrize("F,K", [(1, 1), (33, 7), (5000, 256), (3000, 700), (257, 1024)])
def test_vq_encode_matches_oracle(F, K):
    X = synthetic.mfcc_mixture(F + K, F, K=min(K, 64))
    C = synthetic.random_codebook(K, K)
    if K > 3:
        C[K - 1] = C[1]
    idx = engine.vq_encode(X, C)
    assert np.array_equal(idx, vq_oracle.encode(X, C))


@pytest.mark.parametrize("case", ["nan_inf_frames", "nan_inf_centroids", "all_centroids_nan", "one_centroid", "huge", "fp32_overflow",
                                  "tiny", "fp32_underflow"])
def test_vq_encode_edge_values_match_oracle(case):
    """Values the fp32 prefilter cannot represent (overflow, underflow, NaN, inf) must not change a single index: the
    reference's `distance < min_distance` (hmm_training.py:102-114) never selects a NaN or an infinite distance and keeps
    index 0 when nothing is selected.  The C oracle was compared with the reference on each of these (scripts/
    edge_probe.py); the device path is held to the oracle, bit for bit."""
    from oracle import vq_oracle as V
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
    assert np.array_equal(engine.vq_encode(X, C), V.encode(X, C))


def test_vq_encode_empty():
    assert engine.vq_encode(np.zeros((0, 13)), synthetic.random_codebook(0, 4)).shape == (0,)


def test_lbg_degenerate_duplicates_near_tie():
    """60 frames drawn from 3 distinct points: every split puts a point exactly between the
    twin children c*1.001 / c*0.999, so the winner is decided by the last bit of the centroid
    mean.  The reference sums frames sequentially (np.mean), the GPU in a tree, so WHICH twin
    keeps the points may differ (documented near-tie, DESIGN.md); the multiset of non-empty
    centroids, the number of all-zero centroids (codevector_functions.py:435) and the
    partition of the frames must still agree."""
    g = load_golden("lbg_empty_clusters")
    C, gens, assign, iters, _ = engine.lbg_fit(g["X"], int(g["K"]), int(g["max_iterations"]), float(g["epsilon"]))
    assert C.shape == g["C"].shape and np.array_equal(iters, g["iters"])
    nz, nz_ref = C[np.any(C != 0, axis=1)], g["C"][np.any(g["C"] != 0, axis=1)]
    assert nz.shape == nz_ref.shape
    assert_close(nz[np.lexsort(nz.T)], nz_ref[np.lexsort(nz_ref.T)], "non-empty centroids", rtol=1e-9, atol=1e-12)
    relabel = {}
    for a, b in zip(assign, g["assign"]):
        assert relabel.setdefault(int(a), int(b)) == int(b)


def _with_residence(argname, values):
    """Parameter sets (value, residence) for the LBG tests: every value with host frames (id: the value) and with
    frames already in device memory (id: value-device)."""
    return pytest.mark.parametrize(
        f"{argname},residence", [(v, "host") for v in values] + [(v, "device") for v in values],
        ids=list(values) + [f"{v}-device" for v in values])


def _lbg_fit_from(residence, X, *args):
    """engine.lbg_fit on host frames, or on a device copy of them (hmmb_lbg_fit_ex with x_on_device = 1)."""
    if residence == "host":
        return engine.lbg_fit(X, *args)
    import torch
    dX = torch.from_numpy(np.ascontiguousarray(X, dtype=np.float64)).cuda()
    torch.cuda.synchronize()
    return engine.lbg_fit(None, *args, x_dev_ptr=dX.data_ptr(), F=len(X))


@_with_residence("name", ["lbg_600_k32", "lbg_1200_k256_it3", "lbg_k1", "lbg_k24_nonpow2"])
def test_lbg_matches_reference_golden(name, residence):
    g = load_golden(name)
    C, gens, assign, iters, _ = _lbg_fit_from(residence, g["X"], int(g["K"]), int(g["max_iterations"]),
                                              float(g["epsilon"]))
    assert C.shape == g["C"].shape
    assert np.array_equal(iters, g["iters"])
    assert_close(C, g["C"], "centroids", rtol=1e-9, atol=1e-12)
    assert_close(np.concatenate(gens), g["gens"], "generations", rtol=1e-9, atol=1e-12)
    if len(g["iters"]):
        assert np.array_equal(assign, g["assign"])


def test_lbg_no_data():
    with pytest.raises(ValueError):
        engine.lbg_fit(np.zeros((0, 13)), 4)


@_with_residence("case", ["max_iterations_0", "max_iterations_1", "epsilon_0", "k2", "k3", "k_above_frames", "one_frame",
                          "identical_frames", "nan_coordinate"])
def test_lbg_edge_inputs_match_oracle(case, residence):
    """Edge inputs of createCodeVector (CodeVector/codevector_functions.py:442-531).  The C oracle was compared with the
    reference itself on every one of them (same centroids, assignments and iteration counts: scripts/edge_probe.py has
    the list); here the device path is held to the oracle — a NaN coordinate included, which the reference carries
    through its distances and means without complaint — with the frames passed from host memory and from device
    memory."""
    from oracle import vq_oracle as V
    X = synthetic.mfcc_mixture(3, 200, K=8)
    K, mi, eps = 8, 20, 1e-3
    if case == "max_iterations_0": mi = 0
    elif case == "max_iterations_1": mi = 1
    elif case == "epsilon_0": eps = 0.0
    elif case == "k2": K = 2
    elif case == "k3": K = 3
    elif case == "k_above_frames": X, K = X[:5], 16
    elif case == "one_frame": X, K = X[:1], 4
    elif case == "identical_frames": X = np.tile(X[:1], (30, 1))
    elif case == "nan_coordinate":
        X = X.copy(); X[3, 4] = np.nan; K, mi = 4, 5
    C, gens, assign, iters, gdist = _lbg_fit_from(residence, X, K, mi, eps)
    Co, genso, assigno, iterso, gdisto = V.lbg(X, K, mi, eps)
    assert C.shape == Co.shape and np.array_equal(iters, iterso)
    assert np.allclose(C, Co, rtol=1e-9, atol=0, equal_nan=True)
    assert np.array_equal(assign[:len(X)], assigno)
    for a, b in zip(gens, genso):
        assert np.allclose(a, b, rtol=1e-9, atol=0, equal_nan=True)


def test_large_roundtrip_properties():
    """BASELINE-size properties that need no oracle: rows sum to 1, VQ idempotence
    (a centroid encodes to itself or an identical earlier twin), scoring the training
    data with the trained model reproduces the E-step's per-sequence log-likelihood."""
    N, M, W, S, T = 4, 256, 10, 2000, 200
    obs, offsets, wos = synthetic.fixed_length_codewords(0, W, S, T, N, M)
    pi0, A0, B0 = engine.default_init(N, M)
    with engine.BaumWelch(obs, offsets, wos, W, N, M) as bw:
        bw.set_params(np.tile(pi0, (W, 1)), np.tile(A0, (W, 1, 1)), np.tile(B0, (W, 1, 1)))
        bw.iterate(3, 1e-6, 100)
        pi_raw, A_raw, B_raw = bw.params(finalize=False)
        bw.iterate(1, 1e-6, 100)  # E-step with the parameters above; seq_ll belongs to them
        ll_seq = bw.seq_ll()
        pi, A, B = bw.params(finalize=True)
        hist, iters = bw.history(100)
    assert np.all(iters == 4)
    assert np.allclose(pi.sum(axis=1), 1) and np.allclose(A.sum(axis=2), 1) and np.allclose(B.sum(axis=2), 1)
    assert np.all(np.diff(hist[:, :4], axis=1) > -1e-6)  # EM does not decrease the statistic here
    sub = slice(0, 500)
    ll, _ = engine.score(obs[: 500 * T], offsets[:501], N, M, pi_raw, A_raw, B_raw)
    assert_close(ll[np.arange(500), wos[sub]], ll_seq[sub], "E-step LL vs scorer", rtol=1e-12, atol=0)
    C = synthetic.random_codebook(3, 256)
    assert np.array_equal(engine.vq_encode(C, C), np.arange(256))


@pytest.mark.parametrize("cfg", ["config3", "config4"])
def test_baseline_full_size_properties(cfg):
    """BASELINE configs 3 and 4 IN FULL (10 words x 100 000 sequences x T = 200, N = 4, M = 256 = 200 M frames;
    1000 words x 500 sequences x T = 200, N = 16, M = 1024 = 100 M frames — 7 / 13 GB on the device), through
    properties that need the oracle only on a sample:
      (1) the E-step's per-sequence log-likelihood equals the oracle's forward pass on sequences drawn from
          the first, the last and random CTAs of the launch;
      (2) checksum of checksums: every word's convergence statistic is the log_sum_exp (hmm_training.py:503)
          of its per-sequence values;
      (3) words are independent: one word trained alone (its own CTA partition) gives the same model;
      (4) EM does not decrease the statistic, rows of pi / A / B sum to 1, the left-to-right zero pattern of A
          is preserved."""
    N, M, W, S, T, family = (4, 256, 10, 100_000, 200, "n4_left_to_right") if cfg == "config3" else \
                            (16, 1024, 1000, 500, 200, "left_to_right")
    obs, offsets, wos = synthetic.fixed_length_codewords(1000, W, S, T, N, M)
    R = W * S
    pi0, A0, B0 = engine.default_init(N, M)
    with engine.BaumWelch(obs, offsets, wos, W, N, M) as bw:
        bw.set_params(np.tile(pi0, (W, 1)), np.tile(A0, (W, 1, 1)), np.tile(B0, (W, 1, 1)))
        assert bw.kernel_family() == family
        bw.iterate(2, 1e-6, 100)
        pi_raw, A_raw, B_raw = bw.params(finalize=False)
        bw.iterate(1, 1e-6, 100)  # E-step with the parameters above; seq_ll belongs to them
        ll_seq = bw.seq_ll()
        pi, A, B = bw.params(finalize=True)
        hist, iters = bw.history(100)
    assert np.all(iters == 3)
    # (4)
    assert np.allclose(pi.sum(axis=1), 1, atol=1e-12) and np.allclose(A.sum(axis=2), 1, atol=1e-12)
    assert np.allclose(B.sum(axis=2), 1, atol=1e-9)
    assert np.all(np.diff(hist[:, :3], axis=1) > -1e-6)
    assert np.array_equal(A == 0, np.tile(A0 == 0, (W, 1, 1)))
    assert np.all(ll_seq > -np.inf)
    # (1)
    rng = np.random.default_rng(4)
    sample = np.unique(np.concatenate([np.arange(64), np.arange(R - 64, R), rng.choice(R, 272, replace=False)]))
    for r in sample:
        w = int(wos[r])
        ref = O.calculate_log_likelihood(obs[offsets[r]:offsets[r + 1]].astype(np.int64), A_raw[w], B_raw[w], pi_raw[w])
        assert_close(ll_seq[r:r + 1], np.array([ref]), f"full-size E-step LL of sequence {r} vs oracle forward")
    # (2)
    x = ll_seq.reshape(W, S)
    m = x.max(axis=1)
    assert_close(hist[:, 2], m + np.log(np.exp(x - m[:, None]).sum(axis=1)), "statistic = log_sum_exp of sequence LLs",
                 rtol=1e-12, atol=0)
    # (3)
    w = 7
    off_w = offsets[w * S:(w + 1) * S + 1] - offsets[w * S]
    with engine.BaumWelch(obs[offsets[w * S]:offsets[(w + 1) * S]], off_w, np.zeros(S, dtype=np.int32), 1, N, M) as bw:
        bw.set_params(pi0[None], A0[None], B0[None])
        bw.iterate(3, 1e-6, 100)
        pi1, A1, B1 = bw.params(finalize=True)
        h1, _ = bw.history(100)
    assert_close(h1[0, :3], hist[w, :3], "word alone: statistic", rtol=1e-12, atol=0)
    assert_close(A1[0], A[w], "word alone: A", rtol=1e-10)
    assert_close(pi1[0], pi[w], "word alone: pi", rtol=1e-10)
    assert_close(B1[0], B[w], "word alone: B", rtol=1e-10)


def test_backward_mass_recovering_through_tiny_state(kernel_family):
    """DESIGN.md §4 / VERDICT r1 weak #1: beta mass that sinks below 1e-308 of its step (a run of symbols that only
    the last state emits, the others at 1e-160) and then grows back by 1e20 per step over a run that only the
    FIRST state emits — the backward-only gradual loss.  Whatever route a sequence takes (lean step, careful step,
    norm-consistency hand-over to the exact kernel), pi / A / B and the log-likelihoods must meet the oracle at
    the contract's 1e-9, and the zero / floor patterns must be the reference's."""
    N, M = 4, 8
    pi0 = np.array([0.97, 0.02, 0.005, 0.005])
    A0 = np.zeros((N, N))
    for i in range(3):
        A0[i, i], A0[i, i + 1] = 0.6, 0.4
    A0[3, 3] = 1.0
    B0 = np.full((N, M), 0.1)
    B0[:, 0] = [0.3, 1e-20, 1e-20, 1e-20]       # 'y': only state 0 emits it
    B0[:, 1] = [1e-160, 1e-160, 1e-160, 0.3]    # 'x': only state 3 emits it
    B0[:, 2] = [1e-300, 0.2, 1e-250, 1e-20]
    B0 /= B0.sum(axis=1, keepdims=True)
    rng = np.random.default_rng(3)
    seqs = []
    for ny in range(1, 22):
        for nx in range(1, 6):
            head = list(rng.integers(2, M, size=int(rng.integers(0, 4))))
            tail = list(rng.integers(2, M, size=int(rng.integers(0, 3))))
            seqs.append(np.array(head + [0] * ny + [1] * nx + tail))
            seqs.append(np.array(head + [1] * nx + [0] * ny + tail))
    for _ in range(40):  # long mixtures: several sink / recover cycles per sequence
        parts = []
        for _ in range(6):
            parts += [0] * int(rng.integers(1, 20)) + [1] * int(rng.integers(1, 4)) + list(rng.integers(2, M, size=2))
        seqs.append(np.array(parts))
    corpus = [seqs]
    obs, offsets, wos = synthetic.pack_corpus(corpus, M)
    with engine.BaumWelch(obs, offsets, wos, 1, N, M) as bw:
        bw.set_params(pi0[None], A0[None], B0[None])
        bw.iterate(3, -1.0, 3)
        pi, A, B = bw.params()
        hist, iters = bw.history(3)
        diag = bw.diagnostics()
    Ao, Bo, pio, h, it = O.hmm_training(seqs, N=N, M=M, epsilon=-1.0, max_iterations=3, init=(pi0, A0, B0),
                                        return_history=True)
    assert np.isfinite(h).all()
    assert_close(hist[0, :3], h, f"ll (exact passes, backward hand-overs = {diag})")
    assert_close(A[0], Ao, "A"); assert_close(B[0], Bo, "B"); assert_close(pi[0], pio, "pi")
    assert_same_support(A[0], Ao); assert_same_support(pi[0], pio)
    assert np.array_equal(floored_set(B[0], M), floored_set(Bo, M))
    print(f"exact passes, backward hand-overs = {diag}")
    assert diag[1] > 0  # both kernel families hand these sequences over from the backward pass

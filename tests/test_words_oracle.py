"""CPU checks of the connected-word oracle (oracle/words_oracle.py) — the yardstick of tests/test_gpu_words.py — and
of the argument checks of engine.decode_words / hmm_testing.recognize_connected that run before any device work.

The reference recognises one word per recording, so the oracle is checked against brute force: every (word, first
frame, last frame) segment is scored once by enumerating its state paths, and every segmentation x word assignment is
scored from those.  The oracle's score must be the optimum and its segmentation one of the optimal ones."""
import itertools

import numpy as np
import pytest

from hmm_training_b200 import engine, hmm_testing
from hmm_training_b200.hmm_classes import HMMTrained
from oracle.hmm_oracle import safe_log
from oracle.words_oracle import decode_words_batch

RTOL = 1e-12


def _random_models(rng, W, N, M, ltr, zeros):
    models = []
    for _ in range(W):
        pi = rng.random(N)
        if ltr:
            A = np.zeros((N, N))
            for i in range(N):
                A[i, i] = rng.random()
                if i + 1 < N:
                    A[i, i + 1] = rng.random()
        else:
            A = rng.random((N, N))
        B = rng.random((N, M))
        if zeros:
            pi[rng.random(N) < 0.3] = 0.0
            A[rng.random((N, N)) < 0.3] = 0.0
            B[rng.random((N, M)) < 0.3] = 0.0
        models.append((A, B, pi))
    return models


def _segment_scores(o, models):
    """best[w][a][b]: the best in-word path of word w over frames [a, b], entered in any state, left from N - 1."""
    T = len(o)
    best = {}
    for w, (A, B, pi) in enumerate(models):
        lA, lB, lpi = safe_log(A), safe_log(B), safe_log(pi)
        N = lA.shape[0]
        for a in range(T):
            for b in range(a, T):
                top = -np.inf
                for p in itertools.product(range(N), repeat=b - a):
                    path = p + (N - 1,)
                    s = lpi[path[0]] + lB[path[0], o[a]]
                    for k in range(1, len(path)):
                        s = s + lA[path[k - 1], path[k]] + lB[path[k], o[a + k]]
                    top = max(top, s)
                best[w, a, b] = top
    return best


def _brute_force(o, models, pen):
    """(optimal score, {segmentation: score}) over every segmentation x word assignment."""
    T, W = len(o), len(models)
    seg = _segment_scores(o, models)
    totals = {}
    for cuts in itertools.product((False, True), repeat=T - 1):
        starts = [0] + [t + 1 for t, c in enumerate(cuts) if c]
        ends = [s - 1 for s in starts[1:]] + [T - 1]
        for words in itertools.product(range(W), repeat=len(starts)):
            totals[tuple(zip(words, starts))] = sum(seg[w, a, b] for w, a, b in zip(words, starts, ends)) + len(starts) * pen
    return max(totals.values()), totals


def _close(x, y):
    return (np.isneginf(x) and np.isneginf(y)) or abs(x - y) <= RTOL * max(abs(x), abs(y), 1e-300)


@pytest.mark.parametrize("seed", range(18))
def test_oracle_equals_brute_force(seed):
    rng = np.random.default_rng(seed)
    W = int(rng.integers(1, 4))
    N = int(rng.integers(1, 4))
    M = int(rng.integers(2, 5))
    ltr, zeros = seed % 2 == 0, seed % 3 == 1
    pen = (0.0, -5.0, 2.0)[seed % 3]
    models = _random_models(rng, W, N, M, ltr, zeros)
    obs = [rng.integers(0, M, size=int(rng.integers(1, 8))) for _ in range(5)]
    score, seg_off, seg_word, seg_start, margin = decode_words_batch(obs, models, pen)
    assert seg_off[0] == 0 and len(seg_off) == len(obs) + 1 and len(seg_word) == len(seg_start) == seg_off[-1]
    for u, o in enumerate(obs):
        best, totals = _brute_force(o, models, pen)
        assert _close(score[u], best), (u, score[u], best)
        segs = tuple(zip(seg_word[seg_off[u]:seg_off[u + 1]].tolist(), seg_start[seg_off[u]:seg_off[u + 1]].tolist()))
        if np.isneginf(best):
            assert segs == () and margin[u] == np.inf
        else:
            assert segs in totals and _close(totals[segs], best), (u, segs, totals.get(segs), best)
            assert segs[0][1] == 0 and all(a < b for (_, a), (_, b) in zip(segs, segs[1:]))
            assert margin[u] >= 0


def test_impossible_utterance_has_no_segments():
    A = np.array([[0.5, 0.5], [0.0, 1.0]])
    B = np.array([[1.0, 0.0], [1.0, 0.0]])  # codeword 1 cannot be emitted
    pi = np.array([1.0, 0.0])
    score, seg_off, seg_word, _, margin = decode_words_batch([np.array([0, 1, 0]), np.array([0, 0])], [(A, B, pi)])
    assert score[0] == -np.inf and seg_off[1] == 0 and margin[0] == np.inf
    assert np.isfinite(score[1]) and seg_off[2] >= 1


def test_one_frame_gives_one_segment():
    rng = np.random.default_rng(5)
    models = _random_models(rng, 3, 3, 4, True, False)
    score, seg_off, seg_word, seg_start, _ = decode_words_batch([np.array([2])], models, -3.0)
    assert list(seg_off) == [0, 1] and seg_start[0] == 0
    ends = [safe_log(pi)[-1] + safe_log(B)[-1, 2] for A, B, pi in models]
    assert seg_word[0] == int(np.argmax(ends)) and score[0] == max(ends) + -3.0


def test_duplicate_models_smallest_word_wins():
    rng = np.random.default_rng(7)
    m = _random_models(rng, 2, 3, 6, True, False)
    models = [m[0], m[1], m[1], m[0]]
    obs = [rng.integers(0, 6, size=int(T)) for T in (1, 5, 40, 90)]
    _, seg_off, seg_word, _, margin = decode_words_batch(obs, models, -1.0)
    assert set(seg_word.tolist()) <= {0, 1}
    assert (margin == 0).all()  # every word end is an exact tie


def test_entry_equal_to_in_word_keeps_the_word():
    """One single-state word with self-loop a and penalty log(a): entering again ties with staying, and the in-word
    candidate must win (one segment); a slightly larger penalty makes every frame a word of its own."""
    a = 0.25
    models = [(np.array([[a]]), np.array([[0.5, 0.5]]), np.array([1.0]))]
    o = np.array([0, 1, 1, 0, 1])
    _, seg_off, _, seg_start, margin = decode_words_batch([o], models, float(np.log(a)))
    assert seg_off[1] == 1 and seg_start[0] == 0 and margin[0] == 0
    _, seg_off, _, seg_start, _ = decode_words_batch([o], models, float(np.log(a)) + 1e-3)
    assert seg_off[1] == 5 and list(seg_start) == [0, 1, 2, 3, 4]


def test_equal_predecessors_smallest_state_wins():
    """Frame 2 of a three-state word: predecessor 0 (in the word since frame 0) and predecessor 1 (entered at frame 1)
    reach the exit with exactly the same value log(q).  The smallest predecessor carries the word's first frame 0, so
    the utterance is one segment; taking predecessor 1 would split it at frame 1."""
    q = 0.5
    A = np.zeros((3, 3))
    A[0, 0] = A[0, 2] = A[1, 2] = 1.0
    B = np.ones((3, 1))
    pi = np.array([q, 1.0, 1.0])
    score, seg_off, seg_word, seg_start, margin = decode_words_batch([np.zeros(3, np.int64)], [(A, B, pi)], float(np.log(q)))
    assert list(seg_off) == [0, 1] and list(seg_start) == [0] and list(seg_word) == [0]
    assert score[0] == 2 * np.log(q) and margin[0] == 0


def test_nonfinite_penalty_is_rejected_by_the_oracle():
    models = _random_models(np.random.default_rng(0), 1, 2, 2, True, False)
    for p in (np.inf, -np.inf, np.nan):
        with pytest.raises(ValueError):
            decode_words_batch([np.array([0, 1])], models, p)


# ---------------------------------------------------------------- Python layer (checks before any device work)
def _params(W=2, N=3, M=8):
    return (np.tile(x, (W,) + (1,) * x.ndim) for x in engine.default_init(N, M))


def test_decode_words_argument_errors():
    N, M = 3, 8
    pi, A, B = _params(2, N, M)
    obs = np.zeros(5, np.uint8)
    offsets = np.array([0, 3, 5], np.int64)
    for bad in (np.zeros(5), np.zeros(5, np.float32), np.zeros(5, bool)):
        with pytest.raises(TypeError):
            engine.decode_words(bad, offsets, N, M, pi, A, B)
    with pytest.raises(ValueError):
        engine.decode_words(obs, offsets, N, M, pi[:, :2], A, B)
    with pytest.raises(ValueError):
        engine.decode_words(obs, offsets, N, M, pi, A[:1], B)
    with pytest.raises(ValueError):
        engine.decode_words(obs, offsets, N, M + 1, pi, A, B)
    for p in (np.inf, -np.inf, np.nan):
        with pytest.raises(ValueError):
            engine.decode_words(obs, offsets, N, M, pi, A, B, log_penalty=p)


def test_recognize_connected_argument_errors():
    def hmm(word, N, M):
        pi, A, B = engine.default_init(N, M)
        return HMMTrained(word=word, states=N, symbols=M, A=A, B=B, Pi=pi)

    with pytest.raises(ValueError):
        hmm_testing.recognize_connected([np.array([0, 1])], [hmm("one", 4, 8), hmm("two", 5, 8)])
    with pytest.raises(ValueError):
        hmm_testing.recognize_connected([np.array([0, 1])], [hmm("one", 4, 8), hmm("two", 4, 16)])
    with pytest.raises(IndexError):
        hmm_testing.recognize_connected([np.array([0, 1]), np.array([], np.int64)], [hmm("one", 4, 8)])

"""CPU checks of the Viterbi oracle (oracle/viterbi_oracle.py) — the yardstick of tests/test_gpu_viterbi.py.

The reference has no Viterbi, so the oracle is checked against brute force: every one of the N^T state paths of
tiny random models (with structural zeros) is scored with the same additions in the same order, and the best one
(ties broken towards the smallest last state, then the smallest predecessor, ...) must be what the oracle returns."""
import itertools

import numpy as np
import pytest

from oracle.hmm_oracle import forward_log, safe_log
from oracle.viterbi_oracle import viterbi_batch


def _random_model(rng, N, M, zeros):
    pi = rng.random(N)
    A = rng.random((N, N))
    B = rng.random((N, M))
    if zeros:
        pi[rng.random(N) < 0.3] = 0.0
        A[rng.random((N, N)) < 0.3] = 0.0
        B[rng.random((N, M)) < 0.3] = 0.0
        if N > 1:
            A[0, 0] = np.nan  # NaN is a structural zero too
    pi /= max(np.nansum(pi), 1e-300)
    return A, B, pi


def _brute_force(o, A, B, pi):
    lA, lB, lpi = safe_log(A), safe_log(B), safe_log(pi)
    N, T = lA.shape[0], len(o)
    best, best_key, best_path = -np.inf, None, None
    for p in itertools.product(range(N), repeat=T):
        s = lpi[p[0]] + lB[p[0], o[0]]
        for t in range(1, T):
            s = (s + lA[p[t - 1], p[t]]) + lB[p[t], o[t]]
        key = tuple(reversed(p))  # smallest last state, then smallest predecessor, ...
        if s > best or (s == best and s > -np.inf and key < best_key):
            best, best_key, best_path = s, key, p
    if best == -np.inf:
        return best, np.full(T, -1, dtype=np.int8)
    return best, np.array(best_path, dtype=np.int8)


@pytest.mark.parametrize("seed", range(12))
def test_viterbi_batch_equals_brute_force(seed):
    rng = np.random.default_rng(seed)
    N = int(rng.integers(1, 5))
    M = int(rng.integers(2, 6))
    zeros = seed % 2 == 1
    models = [_random_model(rng, N, M, zeros) for _ in range(3)]
    obs = [rng.integers(0, M, size=int(rng.integers(1, 7))) for _ in range(10)]
    mou = rng.integers(0, len(models), size=len(obs))
    score, paths, margin = viterbi_batch(obs, models, mou)
    for u, o in enumerate(obs):
        A, B, pi = models[mou[u]]
        bs, bp = _brute_force(o, A, B, pi)
        assert score[u] == bs, (u, score[u], bs)  # same additions in the same order: bit-exact
        assert np.array_equal(paths[u], bp), (u, paths[u], bp)
        assert paths[u].dtype == np.int8 and len(paths[u]) == len(o)
        assert margin[u] >= 0


def test_impossible_utterance_gives_minus_one_path():
    A = np.array([[0.5, 0.5], [0.0, 1.0]])
    B = np.array([[1.0, 0.0], [1.0, 0.0]])  # codeword 1 cannot be emitted
    pi = np.array([1.0, 0.0])
    score, paths, margin = viterbi_batch([np.array([0, 1, 0]), np.array([0, 0])], [(A, B, pi)], [0, 0])
    assert score[0] == -np.inf and np.array_equal(paths[0], [-1, -1, -1]) and margin[0] == np.inf
    assert np.isfinite(score[1]) and np.array_equal(paths[1], [0, 0])


@pytest.mark.parametrize("seed", range(6))
def test_score_never_exceeds_forward_log_likelihood(seed):
    rng = np.random.default_rng(100 + seed)
    N, M = 4, 16
    models = [_random_model(rng, N, M, seed % 2 == 1) for _ in range(2)]
    obs = [rng.integers(0, M, size=int(rng.integers(1, 60))) for _ in range(40)]
    mou = rng.integers(0, 2, size=len(obs))
    score, _, _ = viterbi_batch(obs, models, mou)
    for w, (A, B, pi) in enumerate(models):
        us = np.nonzero(mou == w)[0]
        for u in us:
            o = np.asarray(obs[u])[None, :]
            _, logP, _ = forward_log(o, np.array([o.shape[1]]), safe_log(pi), safe_log(A), safe_log(B))
            assert score[u] <= logP[0] + 1e-12 * abs(logP[0]) if np.isfinite(logP[0]) else True
            assert (score[u] == -np.inf) == (logP[0] == -np.inf)


def test_uniform_model_path_is_all_state_zero():
    N, M = 5, 7
    A = np.full((N, N), 1.0 / N)
    B = np.full((N, M), 1.0 / M)
    pi = np.full(N, 1.0 / N)
    rng = np.random.default_rng(3)
    obs = [rng.integers(0, M, size=T) for T in (1, 2, 9, 30)]
    score, paths, margin = viterbi_batch(obs, [(A, B, pi)], [0] * len(obs))
    for u, o in enumerate(obs):
        assert np.array_equal(paths[u], np.zeros(len(o), np.int8))
        assert margin[u] == 0.0  # every decision is a tie
        assert np.isfinite(score[u])

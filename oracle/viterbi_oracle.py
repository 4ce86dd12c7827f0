"""TEST INFRASTRUCTURE — CPU oracle for Viterbi decoding.  NOT part of the product.

An EXTENSION: the reference (DemianMArin/HMM_Training) has no Viterbi, so no reference lines stand behind
this module, and it lives apart from ``hmm_oracle.py``, which restates the reference.  It is a numpy fp64
statement of the semantics ``hmmb_viterbi`` implements (include/hmmb200.h), itself checked against
brute-force enumeration of every state path in ``tests/test_viterbi_oracle.py``:

  * log values from LINEAR pi / A / B with ``hmm_oracle.safe_log`` (entries <= 0 or NaN -> -inf);
  * delta_0(j) = log pi_j + log b_j(o_0);
    delta_t(j) = (max_i (delta_{t-1}(i) + log a_ij)) + log b_j(o_t), additions in exactly this order;
  * psi_t(j) = the smallest i that reaches the max; the last state is the smallest j that reaches
    max_j delta_{T-1}(j), and the score is that max;
  * score -inf (impossible utterance): every frame's state is -1.
"""
from __future__ import annotations

from typing import List, Sequence, Tuple

import numpy as np

from .hmm_oracle import safe_log

NEG_INF = float("-inf")


def _pad(observations: Sequence[np.ndarray]):
    """Utterances -> (codewords [R, Tmax] zero-padded, lengths [R])."""
    lens = np.array([len(o) for o in observations], dtype=np.int64)
    if len(lens) and lens.min() == 0:
        raise IndexError("empty utterance")
    obs = np.zeros((len(lens), int(lens.max()) if len(lens) else 0), dtype=np.int64)
    for r, o in enumerate(observations):
        obs[r, : len(o)] = np.asarray(o, dtype=np.int64)
    return obs, lens


def _rel_margin(cand: np.ndarray, axis: int) -> np.ndarray:
    """Relative gap between the largest and the second largest entry along ``axis``: (best - second) /
    max(|best|, |second|); inf when the runner-up is -inf (or there is none), 0 for a tie."""
    n = cand.shape[axis]
    if n == 1:
        return np.full(cand.shape[:axis] + cand.shape[axis + 1:], np.inf)
    part = -np.partition(-cand, 1, axis=axis)
    best = np.take(part, 0, axis=axis)
    second = np.take(part, 1, axis=axis)
    with np.errstate(invalid="ignore", divide="ignore"):
        diff = best - second
        denom = np.maximum(np.abs(best), np.abs(second))
        m = np.where(denom > 0, diff / denom, np.where(diff > 0, np.inf, 0.0))
    return np.where(np.isneginf(second), np.inf, m)


def viterbi_batch(observations: Sequence[np.ndarray], models, model_of_utt) -> Tuple[np.ndarray, List[np.ndarray], np.ndarray]:
    """Viterbi decoding of every utterance against ``models[model_of_utt[u]]`` (``models``: sequence of
    (A, B, Pi) in linear space, as ``hmm_oracle.score_batch`` takes them), vectorised over the utterances
    of one model.

    Returns (score [U], paths: int8 array per utterance, margin [U]).  margin[u] is the smallest relative
    margin (see _rel_margin) between the winner and the runner-up over every decision on the returned path:
    the choice of the last state and psi_t(s_t) for t >= 1.  Where it is at the level of a few ulps, a log()
    that differs in the last bit may legitimately pick another, equally good path; inf for -inf scores."""
    U = len(observations)
    mou = np.asarray(model_of_utt, dtype=np.int64).reshape(-1)
    if len(mou) != U:
        raise ValueError("one model index per utterance")
    score = np.full(U, NEG_INF)
    margin = np.full(U, np.inf)
    paths: List[np.ndarray] = [None] * U
    for w in np.unique(mou):
        us = np.nonzero(mou == w)[0]
        A, B, Pi = models[int(w)]
        lA = safe_log(np.asarray(A, float))
        lB = safe_log(np.asarray(B, float))
        lpi = safe_log(np.asarray(Pi, float))
        obs, lens = _pad([observations[u] for u in us])
        R, Tmax = obs.shape
        N = lA.shape[0]
        rows = np.arange(R)
        lb = np.transpose(lB[:, obs], (1, 2, 0))  # [R, Tmax, N]
        delta = lpi[None, :] + lb[:, 0, :]
        psi = np.zeros((R, Tmax, N), dtype=np.int8)
        marg = np.full((R, Tmax, N), np.inf)
        for t in range(1, Tmax):
            cand = delta[:, :, None] + lA[None, :, :]  # [R, i, j] = delta_{t-1}(i) + log a_ij
            arg = np.argmax(cand, axis=1)  # first (smallest i) of the maxima
            best = np.take_along_axis(cand, arg[:, None, :], axis=1)[:, 0, :]
            act = (t < lens)[:, None]
            delta = np.where(act, best + lb[:, t, :], delta)
            psi[:, t, :] = arg
            marg[:, t, :] = _rel_margin(cand, axis=1)
        last = np.argmax(delta, axis=1)
        sc = delta[rows, last]
        m = _rel_margin(delta, axis=1)
        state = last.copy()
        path = np.full((R, Tmax), -1, dtype=np.int8)
        for t in range(Tmax - 1, -1, -1):
            on = t < lens
            path[on, t] = state[on]
            if t > 0:
                m = np.where(on, np.minimum(m, marg[rows, t, state]), m)
                state = np.where(on, psi[rows, t, state], state)
        dead = np.isneginf(sc)
        for k, u in enumerate(us):
            score[u] = sc[k]
            if dead[k]:
                paths[u] = np.full(int(lens[k]), -1, dtype=np.int8)
            else:
                paths[u] = path[k, : lens[k]].copy()
                margin[u] = m[k]
    return score, paths, margin

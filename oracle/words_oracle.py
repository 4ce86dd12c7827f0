"""TEST INFRASTRUCTURE — CPU oracle for connected-word decoding.  NOT part of the product.

An EXTENSION: the reference recognises one word per recording, so no reference lines stand behind this module.  It is
a numpy fp64 restatement of the contract ``hmmb_decode_words`` implements (include/hmmb200.h), itself checked against
brute-force enumeration of every segmentation in ``tests/test_words_oracle.py``.  With lpi / lA / lb the logs of the
LINEAR models (``hmm_oracle.safe_log``: entries <= 0 or NaN -> -inf), additions in exactly this order:

  * delta_0(w,j) = lpi[w][j] + lb[w][j](o_0),  token_0(w,j) = 0;
  * t >= 1: in(w,j) = max_i (delta_{t-1}(w,i) + lA[w][i][j]) (smallest i on ties), en(w,j) = E_{t-1} + lpi[w][j],
    delta_t(w,j) = (en > in ? en : in) + lb[w][j](o_t), token_t(w,j) = en > in ? t : token_{t-1}(w, argmax i);
  * e_t = max_w delta_t(w, N-1) (smallest w on ties), E_t = e_t + log_penalty, record_t = (argmax w, its token);
  * score = E_{T-1}; the backtrace reads record_t = (w, s) from t = T-1 ("word w on frames [s, t]") and continues at
    t = s - 1.  An utterance with score -inf has no segments.
"""
from __future__ import annotations

from typing import Sequence

import numpy as np

from .hmm_oracle import safe_log
from .viterbi_oracle import _pad, _rel_margin

NEG_INF = float("-inf")

_CHUNK_CELLS = 1 << 21  # utterances x frames x states held at once


def decode_words_batch(observations: Sequence[np.ndarray], models, log_penalty: float = 0.0):
    """Connected-word decoding of every utterance over the word models ``models`` (a sequence of (A, B, Pi) in linear
    space, one shape, as ``viterbi_oracle.viterbi_batch`` takes them), vectorised over utterances.

    Returns (score [U], seg_offsets int64 [U+1], seg_word int32 [S], seg_start int32 [S], margin [U]).  margin[u] is
    the smallest relative margin (viterbi_oracle._rel_margin) over every decision on the returned segmentation: the
    word-end choice at each segment end, entry against in-word at each frame, and psi along each segment; inf for
    -inf scores."""
    p = float(log_penalty)
    if not np.isfinite(p):
        raise ValueError("log_penalty must be finite")
    lA = np.stack([safe_log(np.asarray(A, float)) for A, _, _ in models])
    lB = np.stack([safe_log(np.asarray(B, float)) for _, B, _ in models])
    lpi = np.stack([safe_log(np.asarray(Pi, float)) for _, _, Pi in models])
    U = len(observations)
    W, N = lpi.shape
    score = np.full(U, NEG_INF)
    margin = np.full(U, np.inf)
    segs = [None] * U
    obs_all, lens_all = _pad(observations)
    Tmax = obs_all.shape[1] if U else 1
    chunk = max(1, _CHUNK_CELLS // max(1, Tmax * W * N))
    for c0 in range(0, U, chunk):
        c1 = min(U, c0 + chunk)
        lens = lens_all[c0:c1]
        obs = obs_all[c0:c1, : int(lens.max())]
        sc, sg, mg = _decode_chunk(obs, lens, lpi, lA, lB, p)
        score[c0:c1] = sc
        margin[c0:c1] = mg
        segs[c0:c1] = sg
    seg_off = np.zeros(U + 1, dtype=np.int64)
    seg_off[1:] = np.cumsum([len(s) for s in segs])
    seg_word = np.array([w for s in segs for w, _ in s], dtype=np.int32)
    seg_start = np.array([a for s in segs for _, a in s], dtype=np.int32)
    return score, seg_off, seg_word, seg_start, margin


def _decode_chunk(obs, lens, lpi, lA, lB, p):
    R, Tmax = obs.shape
    W, N = lpi.shape
    rows = np.arange(R)
    lb = np.transpose(lB[:, :, obs], (2, 3, 0, 1))  # [R, Tmax, W, N]
    delta = lpi[None] + lb[:, 0]
    tok = np.zeros((R, W, N), dtype=np.int64)
    rec_w = np.zeros((R, Tmax), dtype=np.int64)
    rec_s = np.zeros((R, Tmax), dtype=np.int64)
    m_end = np.full((R, Tmax), np.inf)
    psi = np.zeros((R, Tmax, W, N), dtype=np.int8)
    m_psi = np.full((R, Tmax, W, N), np.inf)
    m_ent = np.full((R, Tmax, W, N), np.inf)

    def word_end(t):
        ends = delta[:, :, N - 1]  # [R, W]
        w = np.argmax(ends, axis=1)  # first (smallest w) of the maxima
        rec_w[:, t] = w
        rec_s[:, t] = tok[rows, w, N - 1]
        m_end[:, t] = _rel_margin(ends, axis=1)
        return ends[rows, w] + p

    E = word_end(0)
    for t in range(1, Tmax):
        act = t < lens
        cand = delta[:, :, :, None] + lA[None]  # [R, w, i, j] = delta_{t-1}(w, i) + lA[w][i][j]
        arg = np.argmax(cand, axis=2)  # first (smallest i) of the maxima
        inn = np.take_along_axis(cand, arg[:, :, None, :], axis=2)[:, :, 0, :]
        en = E[:, None, None] + lpi[None]
        enter = en > inn
        new_delta = np.where(enter, en, inn) + lb[:, t]
        new_tok = np.where(enter, t, np.take_along_axis(tok, arg, axis=2))
        delta = np.where(act[:, None, None], new_delta, delta)
        tok = np.where(act[:, None, None], new_tok, tok)
        psi[:, t] = arg
        m_psi[:, t] = _rel_margin(cand, axis=2)
        m_ent[:, t] = _rel_margin(np.stack([np.broadcast_to(en, inn.shape), inn], axis=-1), axis=-1)
        E = np.where(act, word_end(t), E)

    segs, margin = [], np.full(R, np.inf)
    for k in range(R):
        if np.isneginf(E[k]):
            segs.append([])
            continue
        out, m, t = [], np.inf, int(lens[k]) - 1
        while t >= 0:
            w, s = int(rec_w[k, t]), int(rec_s[k, t])
            out.append((w, s))
            m = min(m, m_end[k, t])
            j = N - 1
            for tau in range(t, s, -1):  # in-word frames: the in-word candidate won, psi gives the predecessor
                m = min(m, m_ent[k, tau, w, j], m_psi[k, tau, w, j])
                j = int(psi[k, tau, w, j])
            if s > 0:  # the entry frame: the entry won
                m = min(m, m_ent[k, s, w, j])
            t = s - 1
        segs.append(out[::-1])
        margin[k] = m
    return E, segs, margin

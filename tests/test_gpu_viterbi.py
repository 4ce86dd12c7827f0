"""Viterbi decoding on the GPU (hmmb_viterbi, engine.viterbi, hmm_testing.viterbi_align) against the numpy oracle
oracle/viterbi_oracle.py (itself checked against brute force in tests/test_viterbi_oracle.py).

Scores must agree to 1e-9 relative with the same -inf pattern.  Paths must be equal wherever the oracle's smallest
decision margin on its path exceeds 1e-9; below that, a log() differing in the last bit may pick another path of
(within tolerance) the same score, so there the GPU path must only be a valid path whose score is within tolerance.
"""
import numpy as np
import pytest
import torch

from helpers import RTOL, assert_close, load_golden
from hmm_training_b200 import _lib, engine, hmm_testing
from hmm_training_b200.hmm_classes import HMMTrained
from oracle.hmm_oracle import safe_log
from oracle.viterbi_oracle import viterbi_batch

pytestmark = pytest.mark.gpu

MARGIN = 1e-9


@pytest.fixture(params=["native", "generic"])
def family(request, monkeypatch):
    """Every case once with the kernels the shape selects and once with the lanes-per-state kernels forced."""
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
    pi[:, 0] += 1e-3 if zeros else 0.0
    pi /= pi.sum(1, keepdims=True)
    A /= np.maximum(A.sum(2, keepdims=True), 1e-300)
    B /= np.maximum(B.sum(2, keepdims=True), 1e-300)
    return pi, A, B


def make_corpus(rng, U, W, M, tmax=80, long_T=None):
    lens = rng.integers(1, tmax + 1, size=U)
    lens[0] = 1
    if long_T:
        lens[1] = long_T
    seqs = [rng.integers(0, M, size=int(T)) for T in lens]
    mou = rng.integers(0, W, size=U).astype(np.int32)  # mixed, unsorted
    return seqs, mou


def pack(seqs, dtype=None):
    offsets = np.zeros(len(seqs) + 1, np.int64)
    offsets[1:] = np.cumsum([len(s) for s in seqs])
    flat = np.concatenate(seqs) if seqs else np.zeros(0, np.int64)
    if dtype is None:
        dtype = np.uint8 if flat.max(initial=0) < 256 else np.uint16
    return np.ascontiguousarray(flat.astype(dtype)), offsets


def path_logp(o, p, A, B, pi):
    lA, lB, lpi = safe_log(np.asarray(A, float)), safe_log(np.asarray(B, float)), safe_log(np.asarray(pi, float))
    s = lpi[p[0]] + lB[p[0], o[0]]
    for t in range(1, len(o)):
        s = (s + lA[p[t - 1], p[t]]) + lB[p[t], o[t]]
    return s


def check_against_oracle(seqs, mou, pi, A, B, score, path, offsets, what=""):
    models = [(A[w], B[w], pi[w]) for w in range(pi.shape[0])]
    osc, opaths, omarg = viterbi_batch(seqs, models, mou)
    assert np.array_equal(np.isneginf(score), np.isneginf(osc)), f"{what}: -inf pattern differs"
    assert_close(score, osc, what + " score")
    N = pi.shape[1]
    n_near = 0
    for u, o in enumerate(seqs):
        p = path[offsets[u] - offsets[0]: offsets[u + 1] - offsets[0]]
        if np.isneginf(osc[u]):
            assert (p == -1).all(), f"{what}: utterance {u} is impossible but its path is not all -1"
        elif omarg[u] > MARGIN:
            assert np.array_equal(p, opaths[u]), f"{what}: utterance {u} (T={len(o)}, margin {omarg[u]:.3g}) path differs"
        else:
            n_near += 1
            assert ((p >= 0) & (p < N)).all(), f"{what}: utterance {u} path has invalid states"
            w = mou[u]
            lp = path_logp(o, p.astype(np.int64), A[w], B[w], pi[w])
            assert abs(lp - osc[u]) <= RTOL * abs(osc[u]) + 1e-300, f"{what}: utterance {u} near-tie path scores {lp} vs {osc[u]}"
    return n_near


LAYOUTS = [  # (N, M, left-to-right A)
    (4, 64, False), (4, 64, True), (8, 32, True), (16, 64, True), (8, 32, False), (16, 64, False),
    (1, 8, False), (3, 16, False), (5, 16, True), (6, 20, False), (32, 40, False), (4, 513, False),
]


@pytest.mark.parametrize("N,M,ltr", LAYOUTS)
def test_every_layout_against_oracle(N, M, ltr, family):
    rng = np.random.default_rng(N * 1000 + M + (1 if ltr else 0))
    W = 3
    pi, A, B = make_models(rng, W, N, M, ltr)
    seqs, mou = make_corpus(rng, 150, W, M, long_T=3000)
    obs, offsets = pack(seqs)
    score, path = engine.viterbi(obs, offsets, mou, N, M, pi, A, B)
    assert path.dtype == np.int8 and path.shape == (offsets[-1],)
    check_against_oracle(seqs, mou, pi, A, B, score, path, offsets, f"N={N} M={M} ltr={ltr} {family}")


@pytest.mark.parametrize("N,M,ltr", [(4, 32, False), (4, 32, True), (16, 48, True), (7, 24, False)])
def test_structural_zeros_impossible_and_denormal(N, M, ltr, family):
    rng = np.random.default_rng(7 + N)
    W = 4
    pi, A, B = make_models(rng, W, N, M, ltr, zeros=True)
    B[1, :, M - 1] = 0.0                  # codeword M-1 impossible under model 1
    B[2, :, 0] *= 1e-300                  # denormal emissions under model 2
    B[2, 0, 1] = 5e-324
    pi[3, :] = 0.0                        # model 3: no state can start (every utterance impossible)
    pi[3, N - 1] = np.nan                 # NaN is a structural zero too
    seqs, mou = make_corpus(rng, 120, W, M, tmax=60)
    seqs[2] = np.full(5, M - 1)
    mou[2] = 1
    obs, offsets = pack(seqs)
    score, path = engine.viterbi(obs, offsets, mou, N, M, pi, A, B)
    assert np.isneginf(score[2]) and np.isneginf(score[mou == 3]).all()
    check_against_oracle(seqs, mou, pi, A, B, score, path, offsets, f"zeros N={N} {family}")


@pytest.mark.parametrize("N,M,ltr", [(4, 16, False), (4, 16, True), (8, 16, True), (16, 16, True), (5, 16, False)])
def test_fully_tied_model_path_is_state_zero(N, M, ltr, family):
    pi = np.full((1, N), 1.0 / N)
    if ltr:
        A = np.zeros((1, N, N))
        for i in range(N - 1):
            A[0, i, i] = A[0, i, i + 1] = 0.5
        A[0, N - 1, N - 1] = 0.5  # (every transition equally likely: every decision is a tie)
    else:
        A = np.full((1, N, N), 1.0 / N)
    B = np.full((1, N, M), 1.0 / M)
    rng = np.random.default_rng(5)
    seqs = [rng.integers(0, M, size=T) for T in (1, 2, 17, 300)]
    obs, offsets = pack(seqs)
    score, path = engine.viterbi(obs, offsets, np.zeros(len(seqs), np.int32), N, M, pi, A, B)
    assert (path == 0).all()
    assert np.isfinite(score).all()


@pytest.mark.parametrize("N,M,ltr", [(4, 40, False), (16, 40, True), (6, 40, False)])
def test_idx_bytes_device_resident_score_only_and_repeat(N, M, ltr):
    rng = np.random.default_rng(11)
    W = 3
    pi, A, B = make_models(rng, W, N, M, ltr)
    seqs, mou = make_corpus(rng, 90, W, M)
    ref = None
    for dt in (np.uint8, np.uint16, np.uint32, np.uint64):
        obs, offsets = pack(seqs, dt)
        score, path = engine.viterbi(obs, offsets, mou, N, M, pi, A, B)
        if ref is None:
            ref = (score, path)
            check_against_oracle(seqs, mou, pi, A, B, score, path, offsets, f"N={N}")
        else:
            assert np.array_equal(score, ref[0]) and np.array_equal(path, ref[1]), f"idx_bytes={np.dtype(dt).itemsize}"
        # codewords resident on the device: a torch buffer, complete before the call (library's own stream)
        d = torch.from_numpy(obs.view(np.uint8).copy()).to("cuda")
        torch.cuda.synchronize()
        dscore, dpath = engine.viterbi(None, offsets, mou, N, M, pi, A, B, obs_dev_ptr=d.data_ptr(),
                                       idx_bytes=np.dtype(dt).itemsize)
        assert np.array_equal(dscore, ref[0]) and np.array_equal(dpath, ref[1])
    obs, offsets = pack(seqs)
    s_only, p_none = engine.viterbi(obs, offsets, mou, N, M, pi, A, B, want_path=False)
    assert p_none is None
    assert np.array_equal(s_only.view(np.int64), ref[0].view(np.int64)), "score-only differs from the call with path"
    again = engine.viterbi(obs, offsets, mou, N, M, pi, A, B)
    assert np.array_equal(again[0].view(np.int64), ref[0].view(np.int64)) and np.array_equal(again[1], ref[1])
    # offsets need not start at 0: the path is indexed from offsets[0]
    sub_s, sub_p = engine.viterbi(obs, offsets[5:], mou[5:], N, M, pi, A, B)
    assert np.array_equal(sub_s, ref[0][5:]) and np.array_equal(sub_p, ref[1][offsets[5]:])


def test_phase_times_are_recorded():
    lib = _lib.load()
    _lib.check(lib.hmmb_set_profiling(1))
    try:
        rng = np.random.default_rng(2)
        pi, A, B = make_models(rng, 2, 4, 32, False)
        seqs, mou = make_corpus(rng, 64, 2, 32)
        obs, offsets = pack(seqs)
        engine.viterbi(obs, offsets, mou, 4, 32, pi, A, B)
        ms, n = _lib.phase_ms("viterbi")
        assert ms >= 0 and n >= 1
        ms, n = _lib.phase_ms("viterbi_backtrace")
        assert ms >= 0 and n >= 1
    finally:
        _lib.check(lib.hmmb_set_profiling(0))


@pytest.mark.parametrize("N,M,ltr", [(4, 32, False), (4, 32, True), (8, 32, True), (16, 32, False)])
def test_score_never_exceeds_forward_log_likelihood(N, M, ltr):
    rng = np.random.default_rng(21 + N)
    W = 3
    pi, A, B = make_models(rng, W, N, M, ltr, zeros=True)
    seqs, mou = make_corpus(rng, 100, W, M)
    obs, offsets = pack(seqs)
    score, _ = engine.viterbi(obs, offsets, mou, N, M, pi, A, B, want_path=False)
    ll, _ = engine.score(obs, offsets, N, M, pi, A, B)
    fwd = ll[np.arange(len(seqs)), mou]
    assert np.array_equal(np.isneginf(score), np.isneginf(fwd))
    fin = np.isfinite(fwd)
    assert (score[fin] <= fwd[fin] + 1e-12 * np.abs(fwd[fin])).all()


def test_errors():
    rng = np.random.default_rng(3)
    pi, A, B = make_models(rng, 2, 4, 16, False)
    seqs, mou = make_corpus(rng, 10, 2, 16)
    obs, offsets = pack(seqs)
    bad = obs.copy()
    bad[3] = 16
    with pytest.raises(IndexError):  # HMMB_ERR_RANGE
        engine.viterbi(bad, offsets, mou, 4, 16, pi, A, B)
    off_empty = offsets.copy()
    off_empty[2] = off_empty[1]
    with pytest.raises(IndexError):  # HMMB_ERR_EMPTY
        engine.viterbi(obs, off_empty, mou, 4, 16, pi, A, B)
    m2 = mou.copy()
    m2[4] = 2
    with pytest.raises(_lib.HmmbError) as e:
        engine.viterbi(obs, offsets, m2, 4, 16, pi, A, B)
    assert e.value.code == _lib.ERR_ARG
    m2[4] = -1
    with pytest.raises(_lib.HmmbError) as e:
        engine.viterbi(obs, offsets, m2, 4, 16, pi, A, B)
    assert e.value.code == _lib.ERR_ARG
    p33, A33, B33 = make_models(rng, 1, 33, 16, False)
    with pytest.raises(_lib.HmmbError) as e:
        engine.viterbi(obs, offsets, np.zeros(10, np.int32), 33, 16, p33, A33, B33)
    assert e.value.code == _lib.ERR_UNSUPPORTED
    # the library still works after the errors
    score, path = engine.viterbi(obs, offsets, mou, 4, 16, pi, A, B)
    check_against_oracle(seqs, mou, pi, A, B, score, path, offsets, "after errors")


@pytest.mark.parametrize("shape", ["config3", "config4"])
def test_at_size_against_oracle(shape):
    rng = np.random.default_rng(33 if shape == "config3" else 44)
    if shape == "config3":
        N, M, W, U, ltr = 4, 256, 10, 20000, True
        lens = rng.integers(150, 251, size=U)
    else:
        N, M, W, U, ltr = 16, 1024, 24, 2400, True
        lens = rng.integers(60, 141, size=U)
    pi, A, B = make_models(rng, W, N, M, ltr)
    seqs = [rng.integers(0, M, size=int(T)) for T in lens]
    mou = rng.integers(0, W, size=U).astype(np.int32)
    obs, offsets = pack(seqs)
    score, path = engine.viterbi(obs, offsets, mou, N, M, pi, A, B)
    n_near = check_against_oracle(seqs, mou, pi, A, B, score, path, offsets, shape)
    assert n_near < U // 100


def test_viterbi_align_on_reference_pipeline():
    g = load_golden("pipeline_ref")
    words = [str(w) for w in g["words"]]
    C = g["C"]
    X = g["test"]
    d = ((X[:, None, 1:] - C[None, :, 1:]) ** 2).sum(-1)
    codes = np.argmin(d, axis=1)
    lens = g["test_len"].reshape(-1)
    offs = np.concatenate([[0], np.cumsum(lens)])
    seqs = [codes[offs[u]:offs[u + 1]] for u in range(len(lens))]
    M = C.shape[0]
    hmms = [HMMTrained(states=4, symbols=M, A=g["A"][w], B=g["B"][w], Pi=g["pi"][w], word=words[w]) for w in range(len(words))]
    models = [(g["A"][w], g["B"][w], g["pi"][w]) for w in range(len(words))]
    true_idx = np.array([words.index(str(t)) for t in g["true"]])
    pred_idx = np.array([words.index(str(p)) if str(p) in words else -1 for p in g["pred"]])
    for idx in (true_idx, pred_idx):
        scores, paths = hmm_testing.viterbi_align(seqs, hmms, idx)
        known = idx >= 0
        osc, opaths, _ = viterbi_batch([seqs[u] for u in np.nonzero(known)[0]], models, idx[known])
        assert_close(scores[known], osc, "viterbi_align")
        for k, u in enumerate(np.nonzero(known)[0]):
            assert np.array_equal(paths[u], opaths[k])
        assert np.isneginf(scores[~known]).all() and all((paths[u] == -1).all() for u in np.nonzero(~known)[0])
    # -1 indices and models of mixed (N, M) in one call
    rng = np.random.default_rng(9)
    p8, A8, B8 = make_models(rng, 1, 8, 24, True)
    extra = HMMTrained(states=8, symbols=24, A=A8[0], B=B8[0], Pi=p8[0], word="eight")
    mixed = hmms + [extra]
    idx = np.array([0, 3, -1, 1, 3, 2, -1, 0, 3, 1, 2, 3])
    scores, paths = hmm_testing.viterbi_align(seqs, mixed, idx)
    for u in range(len(seqs)):
        if idx[u] < 0:
            assert np.isneginf(scores[u]) and (paths[u] == -1).all() and len(paths[u]) == len(seqs[u])
            continue
        h = mixed[idx[u]]
        osc, opaths, _ = viterbi_batch([seqs[u]], [(h.A, h.B, h.Pi)], [0])
        assert_close(scores[u:u + 1], osc, f"mixed {u}")
        assert np.array_equal(paths[u], opaths[0])

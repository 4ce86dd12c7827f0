"""Hand-over to the exact log-space kernels on every trainer and scorer path (DESIGN.md §4, precision guard).

The fast kernels compute in the linear domain with one power-of-two scale per step.  A sequence whose value the linear
pass cannot hold to the reference's precision is marked, and k_bw_exact (training) or k_score_exact (recognition)
recomputes it with the reference's log-space recursions.  Every GPU case here proves three things: the guard fired
(a positive counter: exact passes or backward hand-overs of BaumWelch.diagnostics(), or engine.score_diagnostics()),
the case ran on the kernel family it names, and the results meet the oracle at the parity contract.  Hand-over
sequences share 32-sequence blocks with ordinary ones, in several words, so that the fast kernels have to skip exactly
the marked lanes and the exact kernel's atomics have to land in the right word.

Forward construction (_forward_model): a left-to-right model with pi = e_0, a_ii = 0.7, a_i,i+1 = 0.3, and two
special symbols.  P is emitted by state 0 with a normal probability and by every other state with d (1e-320 or
4.9e-324); Q cannot be emitted by states 0 and 1.  An utterance P^a Q^b ... with a >= 2 must sit in state 1 on the last
P frame, so its whole probability runs through a denormal: the unguarded linear pass is off by 1e-7 .. 1e-4 relative,
or returns -inf, while the reference's log P is finite.  The step after the denormal has a total below 2^-960, so the
kernels take their exponent-split branch there, which marks any sequence that carries a denormal.

Error-bound construction (_bound_model): a denormal born in state 2 survives while state 0, emitting 1e-200 per frame,
keeps every step's total far above 2^-960, and a few frames later the denormal carries the utterance.  The
exponent-split branch never runs; the sequence is handed over only because the forward error bound exceeds 1e-12 of
the step's mass (ERR_LIMIT).

test_constructions_defeat_the_linear_pass checks on the CPU, for every model and hand-over utterance used here, that the
unguarded linear pass gets it wrong and that its step totals take the trigger its construction names.

Backward construction (_backward_model, from test_gpu_parity.py::test_backward_mass_recovering_through_tiny_state):
Y is emitted only by state 0 (1e-20 elsewhere) and X only by the last state (1e-160 elsewhere); runs of Y^n X^m in
both orders sink the backward mass below fp64's range of the step and let it grow back, which the backward pass's
norm check hands over.
"""
import ctypes
import zlib

import numpy as np
import pytest

from helpers import assert_close, run_virtual_ranks
from oracle import hmm_oracle as O

P, Q = 0, 1  # forward construction
R, Z = 0, 1  # error-bound construction (models of its own)
Y, X = 0, 1  # backward construction
ROUTES = ("HMMB_FORCE_GENERIC", "HMMB_NO_LTR", "HMMB_FORCE_DENSE_A")


# ------------------------------------------------------------------------------------------------ constructions
def _forward_model(rng, N, M, d, dense=False, lean=False):
    """(pi, A, B) of the forward construction.  dense: row 0 of A stays (0.7, 0.3, 0, ...) so that state 0 cannot
    jump past state 1, every other row is dense.  lean: no zero in B (b_0(Q) = b_1(Q) = 4.9e-324), so that k_score4r
    takes its lean path."""
    pi = np.zeros(N)
    pi[0] = 1.0
    A = np.zeros((N, N))
    if dense:
        A[1:] = rng.dirichlet(np.ones(N), size=N - 1)
        A[0, 0], A[0, 1] = 0.7, 0.3
    else:
        for i in range(N - 1):
            A[i, i], A[i, i + 1] = 0.7, 0.3
        A[N - 1, N - 1] = 1.0
    B = rng.uniform(0.5, 1.5, size=(N, M))
    B /= B.sum(axis=1, keepdims=True)  # normalise first: a denormal divided by the row sum may round to zero
    B[0, P] = 0.3  # a fixed value: with some others the rounding of the denormal happens to be exact for one length
    B[1:, P] = d   # of the P run (test_constructions_defeat_the_linear_pass finds such a choice)
    B[:2, Q] = 4.9e-324 if lean else 0.0
    return pi, A, B


def _forward_models(rng, W, N, M, d=None, dense=False, lean=False):
    ds = [1e-320, 4.9e-324] if d is None else [d]
    ms = [_forward_model(rng, N, M, ds[w % len(ds)], dense, lean) for w in range(W)]
    return tuple(np.stack([m[k] for m in ms]) for k in range(3))


def _handover_utt(rng, M, T):
    a, b = int(rng.integers(2, 5)), int(rng.integers(1, 4))
    return np.array([P] * a + [Q] * b + list(rng.integers(2, M, size=T - a - b)), dtype=np.int64)


def _ordinary_utt(rng, M, T):
    return rng.integers(2, M, size=T).astype(np.int64)


def _bound_model(rng, N, M, d):
    """(pi, A, B) of the error-bound construction: left-to-right as above, two special symbols in models of their own.
    R is emitted by state 0 (normally) and state 2 (with d) and by no other state; Z by state 0 with 1e-200, not by
    state 1, by every other state normally.  After k >= 2 ordinary frames, R Z^m (m >= 2) leaves state 2 with a
    denormal that soon carries the utterance, while state 0 keeps every step's total far above 2^-960 (the
    exponent-split branch never runs).  Only the forward error bound (ERR_LIMIT) can notice that the denormal's rounding
    error has become a sizeable part of the step's mass."""
    pi = np.zeros(N)
    pi[0] = 1.0
    A = np.zeros((N, N))
    for i in range(N - 1):
        A[i, i], A[i, i + 1] = 0.7, 0.3
    A[N - 1, N - 1] = 1.0
    B = rng.uniform(0.5, 1.5, size=(N, M))
    B /= B.sum(axis=1, keepdims=True)
    B[:, R] = 0.0
    B[0, R], B[2, R] = 0.3, d
    B[0, Z], B[1, Z] = 1e-200, 0.0
    return pi, A, B


def _bound_models(rng, W, N, M):
    ms = [_bound_model(rng, N, M, (1e-322, 3e-323)[w % 2]) for w in range(W)]
    return tuple(np.stack([m[k] for m in ms]) for k in range(3))


def _bound_utt(rng, M, T):
    k, m = int(rng.integers(2, 5)), int(rng.integers(2, 5))
    return np.array(list(rng.integers(2, M, size=k)) + [R] + [Z] * m + list(rng.integers(2, M, size=T - k - 1 - m)),
                    dtype=np.int64)


def _forward_corpus(rng, W, M, S, n_ho, lo, hi, ho_words, utt=_handover_utt):
    """S ordinary sequences per word and n_ho hand-over sequences (utt) in each of ho_words, lengths from one range and
    shuffled, so that both kinds share blocks.  Returns (seqs, word_of_seq, is_handover)."""
    seqs, wos, ho = [], [], []
    for w in range(W):
        kinds = rng.permutation(np.r_[np.ones(n_ho if w in ho_words else 0, bool), np.zeros(S, bool)])
        for h in kinds:
            T = int(rng.integers(lo, hi + 1))
            seqs.append(utt(rng, M, T) if h else _ordinary_utt(rng, M, T))
            wos.append(w)
            ho.append(bool(h))
    return seqs, np.array(wos, dtype=np.int32), np.array(ho)


def _backward_model(N, M):
    pi = np.full(N, 0.03 / (N - 1))
    pi[0] = 0.97
    A = np.zeros((N, N))
    for i in range(N - 1):
        A[i, i], A[i, i + 1] = 0.6, 0.4
    A[N - 1, N - 1] = 1.0
    B = np.full((N, M), 0.1)
    B[:, Y] = 1e-20
    B[0, Y] = 0.3
    B[:, X] = 1e-160
    B[N - 1, X] = 0.3
    B[:, 2] = np.resize([1e-300, 0.2, 1e-250, 1e-20], N)
    B /= B.sum(axis=1, keepdims=True)
    return pi, A, B


def _backward_corpus(rng, W, M, n_ordinary=60):
    """Per word: Y^n X^m in both orders with short heads / tails, long mixtures of several sink / recover cycles, and
    n_ordinary sequences without Y or X.  is_handover marks the constructed sequences."""
    seqs, wos, ho = [], [], []
    for w in range(W):
        mine = []
        for ny in range(1, 22):
            for nx in range(1, 6):
                head = list(rng.integers(3, M, size=int(rng.integers(0, 4))))
                tail = list(rng.integers(3, M, size=int(rng.integers(0, 3))))
                mine.append((np.array(head + [Y] * ny + [X] * nx + tail), True))
                mine.append((np.array(head + [X] * nx + [Y] * ny + tail), True))
        for _ in range(40):
            parts = []
            for _ in range(6):
                parts += [Y] * int(rng.integers(1, 20)) + [X] * int(rng.integers(1, 4)) + list(rng.integers(3, M, size=2))
            mine.append((np.array(parts), True))
        for _ in range(n_ordinary):
            mine.append((_ordinary_utt(rng, M, int(rng.integers(3, 40))), False))
        for i in rng.permutation(len(mine)):
            seqs.append(mine[i][0].astype(np.int64))
            wos.append(w)
            ho.append(mine[i][1])
    return seqs, np.array(wos, dtype=np.int32), np.array(ho)


def _tile(model, W):
    return tuple(np.tile(x, (W,) + (1,) * x.ndim) for x in model)


def _seed(name):
    return zlib.crc32(name.encode())


# ------------------------------------------------------------------------------------------------ scorer cases
# name: (N, M, dense, lean, d, (lo, hi) frames, ordinary utterances, hand-over utterances, family, rtol)
SCORE_CASES = {
    "score4r_bidiag": (4, 16, False, False, None, (8, 40), 300, 30, "n4_left_to_right", 1e-9),
    "score4r_bidiag_lean": (4, 16, False, True, 4.9e-324, (8, 40), 300, 30, "n4_left_to_right", 1e-9),
    "score4r_dense": (4, 16, True, False, None, (8, 40), 300, 30, "n4_dense", 1e-9),
    "score4r_dense_lean": (4, 16, True, True, 4.9e-324, (8, 40), 300, 30, "n4_dense", 1e-9),
    "score4_m300_bidiag": (4, 300, False, False, None, (8, 40), 300, 30, "n4_left_to_right", 1e-9),
    "score4_m300_dense": (4, 300, True, False, None, (8, 40), 300, 30, "n4_dense", 1e-9),
    "score4r_vecb": (4, 16, False, False, 4.9e-324, (1500, 1510), 56, 8, "n4_left_to_right", 1e-7),
    "scoreL_n8": (8, 40, False, False, None, (12, 40), 300, 30, "left_to_right", 1e-9),
    "scoreL_n16": (16, 1024, False, False, None, (20, 50), 300, 30, "left_to_right", 1e-9),
    "scoreG_n5_u8": (5, 16, False, False, None, (8, 40), 300, 30, "generic", 1e-9),
    "scoreG_n6_u16": (6, 600, False, False, None, (8, 40), 300, 30, "generic", 1e-9),
    "scoreG_n32": (32, 64, False, False, None, (36, 60), 300, 30, "generic", 1e-9),
}
# the same for the error-bound construction (dense, lean and d unused): fwd4_run (k_score4r, k_score4, the per-state
# bound above 1000 frames), k_scoreL and the lanes-per-state pass
BOUND_SCORE_CASES = {
    "bound_score4r": (4, 16, False, False, None, (12, 40), 300, 30, "n4_left_to_right", 1e-9),
    "bound_score4r_vecb": (4, 16, False, False, None, (1500, 1510), 56, 8, "n4_left_to_right", 1e-7),
    "bound_score4_m300": (4, 300, False, False, None, (12, 40), 300, 30, "n4_left_to_right", 1e-9),
    "bound_scoreL_n8": (8, 40, False, False, None, (12, 40), 300, 30, "left_to_right", 1e-9),
    "bound_scoreL_n16": (16, 1024, False, False, None, (20, 50), 300, 30, "left_to_right", 1e-9),
    "bound_scoreG_n5_u8": (5, 16, False, False, None, (12, 40), 300, 30, "generic", 1e-9),
    "bound_scoreG_n32": (32, 64, False, False, None, (36, 60), 300, 30, "generic", 1e-9),
}


def _score_case(name):
    """(seqs, is_handover, (pi, A, B), family, rtol) of a scorer case: W = 3 models of its construction."""
    bound = name in BOUND_SCORE_CASES
    N, M, dense, lean, d, (lo, hi), S, n_ho, family, rtol = (BOUND_SCORE_CASES if bound else SCORE_CASES)[name]
    rng = np.random.default_rng(_seed(name))
    model = _bound_models(rng, 3, N, M) if bound else _forward_models(rng, 3, N, M, d, dense, lean)
    seqs, _, ho = _forward_corpus(rng, 1, M, S, n_ho, lo, hi, (0,), _bound_utt if bound else _handover_utt)
    return seqs, ho, model, family, rtol


# ------------------------------------------------------------------------------------------------ trainer cases
# name: (N, M, dense A, routing switch, family, codeword dtype)
FORWARD_TRAIN = {
    "n4_m16": (4, 16, False, None, "n4_left_to_right", np.uint8),
    "n4_m256": (4, 256, False, None, "n4_left_to_right", np.uint8),
    "n4_m300": (4, 300, False, None, "n4_left_to_right", np.uint16),
    "n4_dense": (4, 64, True, None, "n4_dense", np.uint8),
    "ltr_n8_m40": (8, 40, False, None, "left_to_right", np.uint8),
    "ltr_n16_m1024": (16, 1024, False, None, "left_to_right", np.uint16),
    "generic_n8": (8, 40, False, "HMMB_NO_LTR", "generic", np.uint8),
    "generic_n5_u8": (5, 16, False, None, "generic", np.uint8),
    "generic_n6_m600_u16": (6, 600, False, None, "generic", np.uint16),
    "generic_n32": (32, 64, False, None, "generic", np.uint8),
}
# the error-bound construction on k_bw_fwd4, k_bw_fwdL and the lanes-per-state pass
BOUND_TRAIN = {
    "bound_n4_m16": (4, 16, False, None, "n4_left_to_right", np.uint8),
    "bound_ltr_n8_m40": (8, 40, False, None, "left_to_right", np.uint8),
    "bound_ltr_n16_m1024": (16, 1024, False, None, "left_to_right", np.uint16),
    "bound_generic_n8": (8, 40, False, "HMMB_NO_LTR", "generic", np.uint8),
    "bound_generic_n5_u8": (5, 16, False, None, "generic", np.uint8),
}
TRAIN_CASES = {**FORWARD_TRAIN, **BOUND_TRAIN}


def _forward_train_case(name, W=3):
    N, M, dense, _, _, _ = TRAIN_CASES[name]
    rng = np.random.default_rng(_seed(name))
    bound = name in BOUND_TRAIN
    init = _bound_models(rng, W, N, M) if bound else _forward_models(rng, W, N, M, None, dense)
    lo, hi = (12, 40) if N <= 16 else (36, 60)
    seqs, wos, ho = _forward_corpus(rng, W, M, 90, 12, lo, hi, (0, 1), _bound_utt if bound else _handover_utt)
    return seqs, wos, ho, init


# ------------------------------------------------------------------------------------------------ CPU: the constructions
def _linear_forward(o, pi, A, B, totals=False):
    """log P of utterance o under every model (pi [W,N], A [W,N,N], B [W,N,M]) from the unguarded linear forward pass:
    fp64 with gradual underflow and one power-of-two rescale per step that brings the step's total into [0.5, 1) (what
    the fast kernels do before their guard).  totals=True also returns the smallest step total per model, each taken
    before its rescale from the previous step's rescaled values."""
    alpha = pi * B[:, :, o[0]]
    k = np.zeros(len(pi))
    low = alpha.sum(axis=1)
    for t in range(1, len(o) + 1):
        m = alpha.sum(axis=1)
        e = np.where(m > 0, np.frexp(np.where(m > 0, m, 1.0))[1], 0)
        alpha = np.ldexp(alpha, -e[:, None])
        k += e
        if t < len(o):
            alpha = np.einsum("wi,wij->wj", alpha, A) * B[:, :, o[t]]
            low = np.minimum(low, alpha.sum(axis=1))
    s = alpha.sum(axis=1)
    with np.errstate(divide="ignore"):
        ll = np.where(s > 0, np.log(s) + k * np.log(2.0), -np.inf)
    return (ll, low) if totals else ll


TINY_STEP = 2.0 ** -960  # below it the kernels switch to exponent-split products (hmm_device.cuh)


def _assert_linear_pass_fails(seqs, model, what, bound):
    """The linear pass is wrong on every pair, and the pairs reach the guard through the trigger their construction
    names: the error-bound construction keeps every step total at least 2^10 above TINY_STEP (a margin for kernels that
    rescale to another binade), the others take a step below it."""
    pi, A, B = model
    ref = O.score_batch(seqs, [(A[w], B[w], pi[w]) for w in range(len(pi))])
    assert np.isfinite(ref).all(), f"{what}: the reference gives up on a constructed utterance"
    lin, low = (np.array(x) for x in zip(*[_linear_forward(o, pi, A, B, totals=True) for o in seqs]))
    with np.errstate(invalid="ignore"):
        teeth = np.isneginf(lin) | (np.abs(lin - ref) > 1e-7 * np.abs(ref))
    assert teeth.all(), f"{what}: the linear pass gets {int((~teeth).sum())} of {teeth.size} pairs right"
    if bound:
        assert (low >= 2.0 ** 10 * TINY_STEP).all(), f"{what}: a step total of {low.min()!r} takes the exponent-split branch"
    else:
        assert (low < TINY_STEP).all(), f"{what}: a pair never takes the exponent-split branch"


@pytest.mark.parametrize("case", [f"score:{n}" for n in (*SCORE_CASES, *BOUND_SCORE_CASES)] +
                         [f"train:{n}" for n in TRAIN_CASES] + ["score:pipelined", "train:pipelined_ltr_n16"])
def test_constructions_defeat_the_linear_pass(case):
    """Every forward construction this file hands to the GPU must be one the fast path cannot get right without the
    guard: the unguarded linear forward pass is more than 1e-7 relative off the oracle, or -inf where the oracle is
    finite, on every (hand-over utterance, model) pair.  If a construction is ever edited into one the linear pass
    handles exactly, the GPU cases would prove nothing, and this fails on any machine.  It also pins which of the
    guard's triggers each construction needs: the error-bound cases never take a step below 2^-960, so only the
    comparison with ERR_LIMIT can hand them over; the others always do."""
    kind, name = case.split(":")
    bound = name.startswith("bound_")
    if name == "pipelined":
        seqs, ho, model = _pipelined_score_data(handover_only=True)
        _assert_linear_pass_fails(seqs, model, case, bound)
        return
    if name == "pipelined_ltr_n16":
        seqs, wos, ho, init, _ = _pipelined_forward_data(construction_words_only=True)
    elif kind == "score":
        seqs, ho, model, _, _ = _score_case(name)
        _assert_linear_pass_fails([s for s, h in zip(seqs, ho) if h], model, case, bound)
        return
    else:
        seqs, wos, ho, init = _forward_train_case(name)
    for w in np.unique(wos[ho]):
        mine = [s for s, h, v in zip(seqs, ho, wos) if h and v == w]
        _assert_linear_pass_fails(mine, tuple(x[w:w + 1] for x in init), f"{case} word {w}", bound)


def test_linear_pass_statement_is_exact_on_ordinary_utterances():
    """The statement above is the fast path on ordinary input: on utterances without the special symbols it meets the
    oracle to 1e-12, so the failures above come from the constructions, not from the statement."""
    seqs, ho, model, _, _ = _score_case("scoreG_n5_u8")
    pi, A, B = model
    plain = [s for s, h in zip(seqs, ho) if not h][:40]
    ref = O.score_batch(plain, [(A[w], B[w], pi[w]) for w in range(len(pi))])
    lin = np.array([_linear_forward(o, pi, A, B) for o in plain])
    assert_close(lin, ref, "linear pass on ordinary utterances", rtol=1e-12)


# ------------------------------------------------------------------------------------------------ GPU helpers
def _route(monkeypatch, switch):
    for env in ROUTES:
        monkeypatch.delenv(env, raising=False)
    if switch:
        monkeypatch.setenv(switch, "1")


def _pack(seqs, dtype):
    off = np.concatenate([[0], np.cumsum([len(s) for s in seqs])]).astype(np.int64)
    return np.concatenate(seqs).astype(dtype), off


def _assert_mixed(seqs, wos, ho, min_words):
    """Hand-over and ordinary sequences share blocks: the library sorts a word's sequences by descending length
    (stably) and cuts the blocked layouts' 32-sequence blocks from that order."""
    lens = np.array([len(s) for s in seqs])
    words = blocks = 0
    for w in np.unique(wos):
        idx = np.flatnonzero(wos == w)
        idx = idx[np.argsort(-lens[idx], kind="stable")]
        n = sum(1 for b in range(0, len(idx), 32) if ho[idx[b:b + 32]].any() and not ho[idx[b:b + 32]].all())
        words += n > 0
        blocks += n
    assert words >= min_words and blocks >= 2, f"hand-over sequences mixed into {blocks} blocks of {words} words"


def _family_of(N, M, model):
    """The kernel family the library picks for these models (hmmb_score and the trainer choose it in one place)."""
    from hmm_training_b200 import engine
    W = len(model[0])
    with engine.BaumWelch(np.zeros(2, np.uint8), np.array([0, 2]), np.zeros(1, np.int32), W, N, M) as bw:
        bw.set_params(*model)
        return bw.kernel_family()


def _train(seqs, wos, W, N, M, init, dtype, iters=3, dev=None):
    """3 iterations with sync_each: ((pi, A, B, hist, iters, thin states), family, diagnostics)."""
    from hmm_training_b200 import engine
    obs, off = _pack(seqs, dtype)
    kw = {}
    if dev is not None:
        kw = dict(obs_dev_ptr=dev(obs).data_ptr(), idx_bytes=obs.itemsize)
        obs = None
    with engine.BaumWelch(obs, off, wos, W, N, M, **kw) as bw:
        bw.set_params(*init)
        family = bw.kernel_family()
        bw.iterate(iters, -1.0, iters, sync_each=True)
        got = bw.params() + bw.history(iters) + (bw.thin_states(),)
        return got, family, bw.diagnostics()


def _check_training(got, seqs, wos, W, N, M, init, iters=3, words=None):
    from test_gpu_thin_states import _check
    if words is None:
        _check(got, seqs, wos, W, N, M, init, iters)
        return
    for w in words:  # a sample of words, each against its own oracle run
        mine = [seqs[r] for r in range(len(seqs)) if wos[r] == w]
        sub = tuple(x[w:w + 1] for x in got[:3]) + (got[3][w:w + 1], got[4][w:w + 1], got[5])
        _check(sub, mine, np.zeros(len(mine), np.int32), 1, N, M, tuple(x[w:w + 1] for x in init), iters)


def _check_scores(ll, arg, seqs, model, rtol, what):
    pi, A, B = model
    ref = O.score_batch(seqs, [(A[w], B[w], pi[w]) for w in range(len(pi))])
    assert np.array_equal(np.isneginf(ll), np.isneginf(ref)), f"{what}: -inf pattern"
    assert_close(ll, ref, what, rtol=rtol)
    assert np.array_equal(arg, O.argmax_first(ref)), f"{what}: argmax"


def _pinned_copy(a):
    """numpy view of pinned host memory (hmmb_host_alloc) holding a copy of `a`, and its handle."""
    from hmm_training_b200 import _lib
    p = _lib.load().hmmb_host_alloc(a.nbytes)
    assert p
    buf = np.ctypeslib.as_array((ctypes.c_uint8 * a.nbytes).from_address(p)).view(a.dtype).reshape(a.shape)
    buf[...] = a
    return buf, p


def _host_free(p):
    from hmm_training_b200 import _lib
    _lib.load().hmmb_host_free(p)


@pytest.fixture
def dev():
    """dev(a) -> a uint8 CUDA tensor holding the bytes of numpy array `a`, complete before it is returned."""
    import torch
    keep = []

    def copy(a):
        t = torch.from_numpy(np.ascontiguousarray(a).reshape(-1).view(np.uint8).copy()).to("cuda")
        torch.cuda.synchronize()
        keep.append(t)
        return t

    yield copy
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ GPU: trainer
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TRAIN_CASES))
def test_forward_handover_in_every_estep_family(name, monkeypatch):
    """Warm start from saved-looking models with denormal / zero emissions: the forward pass of every E-step family
    marks the constructed sequences, through the exponent-split branch (the first construction) or through the error
    bound (bound_*), and k_bw_exact recomputes them; parameters and history against the oracle."""
    N, M, _, switch, family, dtype = TRAIN_CASES[name]
    _route(monkeypatch, switch)
    W = 3
    seqs, wos, ho, init = _forward_train_case(name, W)
    _assert_mixed(seqs, wos, ho, min_words=2)
    got, fam, diag = _train(seqs, wos, W, N, M, init, dtype)
    print(f"{name}: family {fam}, exact passes / backward hand-overs {diag}")
    assert fam == family
    # the forward pass handed them over: had it missed them, the backward pass's norm check would catch them and the
    # redone E-step would still meet the oracle, but only with sync_each
    assert diag[0] > 0 and diag[1] == 0
    _check_training(got, seqs, wos, W, N, M, init)


# name: (N, M, routing switch, family)
BACKWARD_TRAIN = {
    "n4": (4, 8, None, "n4_left_to_right"),
    "n4_dense": (4, 8, "HMMB_FORCE_DENSE_A", "n4_dense"),
    "ltr_n8": (8, 40, None, "left_to_right"),
    "ltr_n16": (16, 64, None, "left_to_right"),
    "generic_n5": (5, 8, None, "generic"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(BACKWARD_TRAIN))
def test_backward_handover_redoes_the_estep(name, monkeypatch):
    """Backward mass that sinks below fp64's range of its step and grows back: the backward pass's norm check hands
    the sequence over and, with sync_each, the host redoes the E-step; results against the oracle."""
    N, M, switch, family = BACKWARD_TRAIN[name]
    _route(monkeypatch, switch)
    W = 2
    rng = np.random.default_rng(_seed(name))
    seqs, wos, ho = _backward_corpus(rng, W, M)
    init = _tile(_backward_model(N, M), W)
    _assert_mixed(seqs, wos, ho, min_words=2)
    got, fam, diag = _train(seqs, wos, W, N, M, init, np.uint8)
    print(f"backward {name}: family {fam}, exact passes / backward hand-overs {diag}")
    assert fam == family
    assert diag[1] > 0
    _check_training(got, seqs, wos, W, N, M, init)


BULK_WORDS = 16  # ordinary words behind the constructed ones in the pipelined-create cases


def _bulk_words(rng, Wb, S, T, M, dtype):
    """Wb words of S ordinary sequences of T frames each (already in the library's sorted order)."""
    obs = rng.integers(3, M, size=Wb * S * T).astype(dtype)
    return obs, np.full(Wb * S, T, np.int64)


def _pipelined_forward_data(construction_words_only=False):
    """Left-to-right N = 16, M = 1024: four words of the forward construction (hand-overs in three of them) ahead of
    sixteen bulk words, 36 MB of u16 codewords in sorted order (two upload chunks).  Returns (seqs of the construction
    words, their words, is_handover, init of all words, (bulk obs, bulk lengths))."""
    N, M, Wc, Wb = 16, 1024, 4, BULK_WORDS
    rng = np.random.default_rng(_seed("pipelined_ltr_n16"))
    init = _forward_models(rng, Wc + Wb, N, M)
    seqs, wos, ho = _forward_corpus(rng, Wc, M, 150, 10, 20, 60, ho_words=(0, 1, 3))
    if construction_words_only:
        return seqs, wos, ho, init, None
    return seqs, wos, ho, init, _bulk_words(rng, Wb, 11250, 100, M, np.uint16)


def _sorted_pack(seqs, wos, bulk, Wc, dtype):
    """Codewords and offsets of the construction words (each word's sequences by descending length) followed by the
    bulk words, in the library's sorted order; also the permuted (seqs, wos) and the full word_of_seq."""
    lens = np.array([len(s) for s in seqs])
    order = np.lexsort((-lens, wos))  # by word, then descending length; ties keep their order
    seqs, wos = [seqs[i] for i in order], wos[order]
    bobs, blens = bulk
    obs = np.concatenate([np.concatenate(seqs).astype(dtype), bobs])
    lens = np.concatenate([[len(s) for s in seqs], blens])
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    wall = np.concatenate([wos, Wc + np.repeat(np.arange(BULK_WORDS), len(blens) // BULK_WORDS)]).astype(np.int32)
    return seqs, wos, obs, off, wall


def _pipelined_vs_plain(obs, off, wall, W, N, M, init):
    """The pipelined create (pinned codewords, staged first E-step) and the plain path on the same corpus."""
    from hmm_training_b200 import engine
    assert obs.nbytes >= 32 << 20  # two upload chunks: a staged first E-step of two stages
    pinned, handle = _pinned_copy(obs)
    try:
        with engine.BaumWelch(pinned, off, wall, W, N, M, pipeline_upload=True, init=init) as bw:
            fam = bw.kernel_family()
            bw.iterate(3, -1.0, 3, sync_each=True)
            a = bw.params() + bw.history(3) + (bw.thin_states(),)
            diag_a = bw.diagnostics()
    finally:
        _host_free(handle)
    with engine.BaumWelch(obs, off, wall, W, N, M) as bw:
        bw.set_params(*init)
        bw.iterate(3, -1.0, 3, sync_each=True)
        b = bw.params() + bw.history(3) + (bw.thin_states(),)
        diag_b = bw.diagnostics()
    # the first statistic is reduced in a fixed order: bit-identical; what follows the exact kernel's fp64 atomics
    # agrees to rounding
    assert np.array_equal(a[3][:, 0], b[3][:, 0])
    assert np.array_equal(a[4], b[4])
    for x, y, what in zip(a[:4], b[:4], ("pi", "A", "B", "history")):
        assert_close(x, y, f"pipelined vs plain {what}", rtol=1e-11)
    return a, fam, diag_a, diag_b


@pytest.mark.gpu
def test_pipelined_create_forward_handover_left_to_right(monkeypatch):
    """Pipelined create on the left-to-right kernels, N = 16: the staged first E-step's forward passes hand sequences
    over, the exact kernel runs after the stages; the result equals the plain path and, on a sample of words, the
    oracle."""
    _route(monkeypatch, None)
    N, M, Wc = 16, 1024, 4
    seqs, wos, ho, init, bulk = _pipelined_forward_data()
    _assert_mixed(seqs, wos, ho, min_words=2)
    seqs, wos, obs, off, wall = _sorted_pack(seqs, wos, bulk, Wc, np.uint16)
    W = len(init[0])
    got, fam, diag_a, diag_b = _pipelined_vs_plain(obs, off, wall, W, N, M, init)
    print(f"pipelined forward ltr N = 16: family {fam}, pipelined {diag_a}, plain {diag_b}")
    assert fam == "left_to_right"
    assert diag_a[0] > 0 and diag_b[0] > 0 and diag_a[1] == diag_b[1] == 0
    sample = [0, 2, Wc + 5]
    allseqs = seqs + [obs[off[r]:off[r + 1]].astype(np.int64) for r in range(len(seqs), len(wall)) if wall[r] == Wc + 5]
    allwos = np.concatenate([wos, np.full(len(allseqs) - len(seqs), Wc + 5, np.int32)])
    _check_training(got, allseqs, allwos, W, N, M, init, words=sample)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["ltr_n16", "n4"])
def test_pipelined_create_backward_handover(name, monkeypatch):
    """Pipelined create whose staged first E-step meets backward hand-overs (N = 4 and left-to-right N = 16): the
    redo of the E-step must give the plain path's result and, on a sample of words, the oracle's."""
    _route(monkeypatch, None)
    N, M, family, dtype = (16, 64, "left_to_right", np.uint8) if name == "ltr_n16" else (4, 8, "n4_left_to_right", np.uint8)
    Wc = 3
    rng = np.random.default_rng(_seed("pipelined_backward_" + name))
    seqs, wos, ho = _backward_corpus(rng, Wc, M)
    _assert_mixed(seqs, wos, ho, min_words=2)
    bulk = _bulk_words(rng, BULK_WORDS, 75000 if N == 4 else 22500, 30 if N == 4 else 100, M, dtype)
    seqs, wos, obs, off, wall = _sorted_pack(seqs, wos, bulk, Wc, dtype)
    W = Wc + BULK_WORDS
    init = _tile(_backward_model(N, M), W)
    got, fam, diag_a, diag_b = _pipelined_vs_plain(obs, off, wall, W, N, M, init)
    print(f"pipelined backward {name}: family {fam}, pipelined {diag_a}, plain {diag_b}")
    assert fam == family
    assert diag_a[1] > 0 and diag_b[1] > 0
    _check_training(got, seqs, wos, W, N, M, init, words=range(Wc))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["n4_m16", "generic_n5_u8"])
def test_forward_handover_with_device_resident_codewords(name, dev, monkeypatch):
    """Codewords already in HBM, 4 bytes wide, on one blocked family (N = 4) and on the lanes-per-state family."""
    N, M, _, switch, family, _ = FORWARD_TRAIN[name]
    _route(monkeypatch, switch)
    W = 3
    seqs, wos, ho, init = _forward_train_case(name, W)
    got, fam, diag = _train(seqs, wos, W, N, M, init, np.uint32, dev=dev)
    print(f"device-resident {name}: family {fam}, exact passes / backward hand-overs {diag}")
    assert fam == family
    assert diag[0] > 0 and diag[1] == 0
    _check_training(got, seqs, wos, W, N, M, init)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["forward", "backward"])
def test_handover_on_one_of_two_virtual_ranks(kind, monkeypatch):
    """Two virtual ranks with every hand-over sequence in rank 0's shard: the exact kernel's contributions enter the
    summed accumulators, and a backward hand-over's redo of the E-step is taken by both ranks in step; the result
    equals the one-rank run and the oracle."""
    _route(monkeypatch, None)
    W, N, iters = 2, 4, 3
    rng = np.random.default_rng(_seed("ranks_" + kind))
    if kind == "forward":
        M = 16
        init = _forward_models(rng, W, N, M)
        seqs, wos, ho = _forward_corpus(rng, W, M, 90, 12, 8, 40, ho_words=(0, 1))
    else:
        M = 8
        init = _tile(_backward_model(N, M), W)
        seqs, wos, ho = _backward_corpus(rng, W, M, n_ordinary=120)
    want, fam, diag = _train(seqs, wos, W, N, M, init, np.uint8, iters)
    assert fam == "n4_left_to_right"
    _check_training(want, seqs, wos, W, N, M, init, iters)
    plain = np.flatnonzero(~ho)
    shards = [np.sort(np.r_[np.flatnonzero(ho), plain[::2]]), plain[1::2]]
    got, diags, _ = run_virtual_ranks(shards, lambda idx: _pack([seqs[i] for i in idx], np.uint8), wos, W, N, M,
                                      init, iters)
    print(f"{kind}: one rank {diag}, two ranks {diags}")
    col = 0 if kind == "forward" else 1
    assert diag[col] > 0 and diags[0][col] > 0 and diags[1][0] == 0
    if kind == "forward":
        assert diag[1] == diags[0][1] == diags[1][1] == 0
    for x, y, what in zip(got[:5], want[:5], ("pi", "A", "B", "statistic", "iterations")):
        assert_close(x, y, f"2 virtual ranks: {what}", rtol=1e-9, atol=1e-12)
    _check_training(got, seqs, wos, W, N, M, init, iters)


# ------------------------------------------------------------------------------------------------ GPU: scorer
@pytest.mark.gpu
@pytest.mark.parametrize("name", [*SCORE_CASES, *BOUND_SCORE_CASES])
def test_scorer_hands_over_in_every_family(name, monkeypatch):
    """k_score4r (lean and full, bidiagonal and dense), k_score4 (M = 300), the per-state error bound above 1000
    frames, k_scoreL (N = 8 / 16) and k_scoreG (u8 / u16 codewords, N = 32), with both constructions (bound_*: the
    error-bound trigger): the constructed pairs are recomputed by k_score_exact — counted by hmmb_score_diagnostics —
    and every score meets the oracle."""
    from hmm_training_b200 import engine
    _route(monkeypatch, None)
    seqs, ho, model, family, rtol = _score_case(name)
    N, M = model[2].shape[1:]
    assert _family_of(N, M, model) == family
    _assert_mixed(seqs, np.zeros(len(seqs), np.int32), ho, min_words=1)
    obs, off = _pack(seqs, np.uint8 if M <= 256 else np.uint16)
    ll, arg = engine.score(obs, off, N, M, *model)
    n = engine.score_diagnostics()
    print(f"{name}: family {family}, pairs recomputed {n} of {int(ho.sum()) * len(model[0])} constructed")
    assert n == int(ho.sum()) * len(model[0])  # every constructed pair, and no ordinary one
    _check_scores(ll, arg, seqs, model, rtol, name)
    # the counter belongs to the last call
    plain = [s for s, h in zip(seqs, ho) if not h][:64]
    obs, off = _pack(plain, np.uint8 if M <= 256 else np.uint16)
    engine.score(obs, off, N, M, *model)
    assert engine.score_diagnostics() == 0


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["score4r_bidiag", "scoreG_n5_u8"])
def test_scorer_handover_with_device_resident_codewords(name, dev, monkeypatch):
    from hmm_training_b200 import engine
    _route(monkeypatch, None)
    seqs, ho, model, family, rtol = _score_case(name)
    N, M = model[2].shape[1:]
    assert _family_of(N, M, model) == family
    obs, off = _pack(seqs, np.uint32)
    ll, arg = engine.score(None, off, N, M, *model, obs_dev_ptr=dev(obs).data_ptr(), idx_bytes=4)
    n = engine.score_diagnostics()
    print(f"device-resident {name}: pairs recomputed {n}")
    assert n == int(ho.sum()) * len(model[0])
    _check_scores(ll, arg, seqs, model, rtol, f"device-resident {name}")


def _pipelined_score_data(handover_only=False):
    """400 000 utterances of 90 frames (36 MB of u8 codewords: two upload chunks), every 1000th one a hand-over
    utterance, against three N = 4 models of the forward construction."""
    U, T, M = 400_000, 90, 16
    rng = np.random.default_rng(_seed("pipelined_score"))
    model = _forward_models(rng, 3, 4, M)
    ho_at = np.arange(500, U, 1000)
    hos = [_handover_utt(rng, M, T) for _ in ho_at]
    if handover_only:
        return hos, np.ones(len(hos), bool), model
    obs = rng.integers(2, M, size=(U, T)).astype(np.uint8)
    obs[ho_at] = np.array(hos, dtype=np.uint8)
    ho = np.zeros(U, bool)
    ho[ho_at] = True
    return obs, ho, model


@pytest.mark.gpu
def test_pipelined_scorer_hands_over_like_the_plain_scorer(monkeypatch):
    """The pipelined scorer (pinned codewords, two stages) with a pageable and with a pinned result matrix and
    argmax-only must equal the unpipelined call bit for bit and recompute the same number of pairs; the hand-over
    utterances and a sample of the others against the oracle."""
    from hmm_training_b200 import engine
    _route(monkeypatch, None)
    obs2d, ho, model = _pipelined_score_data()
    U, T = obs2d.shape
    N, M = 4, 16
    assert _family_of(N, M, model) == "n4_left_to_right"
    offsets = np.arange(U + 1, dtype=np.int64) * T
    pinned, handle = _pinned_copy(obs2d.reshape(-1))
    try:
        monkeypatch.setenv("HMMB_SCORE_NO_PIPELINE", "1")
        ll0, arg0 = engine.score(pinned, offsets, N, M, *model)
        n0 = engine.score_diagnostics()
        monkeypatch.delenv("HMMB_SCORE_NO_PIPELINE")
        ll1, arg1 = engine.score(pinned, offsets, N, M, *model)
        n1 = engine.score_diagnostics()
        ll_pin, hll = _pinned_copy(np.zeros((U, len(model[0]))))
        try:
            ll2, arg2 = engine.score(pinned, offsets, N, M, *model, out_ll=ll_pin)
            ll2 = ll2.copy()
        finally:
            _host_free(hll)
        n2 = engine.score_diagnostics()
        _, arg3 = engine.score(pinned, offsets, N, M, *model, want_ll=False)
        n3 = engine.score_diagnostics()
    finally:
        _host_free(handle)
    print(f"pipelined scorer: pairs recomputed {n0} (plain), {n1} / {n2} / {n3} (pipelined: pageable, pinned, argmax)")
    assert n0 == int(ho.sum()) * len(model[0]) and n0 == n1 == n2 == n3
    for ll in (ll1, ll2):
        assert np.array_equal(ll.view(np.int64), ll0.view(np.int64))
    for arg in (arg1, arg2, arg3):
        assert np.array_equal(arg, arg0)
    sample = np.r_[np.arange(300), np.flatnonzero(ho)]
    _check_scores(ll0[sample], arg0[sample], [obs2d[u].astype(np.int64) for u in sample], model, 1e-9,
                  "pipelined scorer vs oracle")

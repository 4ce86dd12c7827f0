"""Thin states: rows of A / B whose whole posterior mass over the training set is below what fp64 can hold.

The kernels accumulate posteriors (gamma, xi in [0, 1]) in the linear domain; the reference keeps log sums
(HMM/hmm_training.py:429-497) and still forms the ratios that become a row of A or B when numerator and denominator
are both 1e-340.  The property tests found the case (16 states, one 15-frame sequence: state 13 is entered before the
last step with negligible posterior, and the denominator of A excludes the last step) — here it is pinned, together
with the more ordinary way to get there: tail states of a left-to-right model that the data never reaches, whose
posterior decays super-exponentially from one EM iteration to the next.  The M-step flags such a state
(denominator below 2^-200), and from then on its rows come from log-space sums (hmm_device.cuh, "thin-state rescue").
"""
import numpy as np
import pytest

from helpers import assert_close, assert_same_support, floored_set, run_virtual_ranks
from oracle import hmm_oracle as O
from test_properties import _pack, _random_corpus, _random_model

pytestmark = pytest.mark.gpu


def _fit(engine, seqs, wos, W, N, M, init, iters, sync_each=True, calls=1):
    obs, off = _pack(seqs)
    with engine.BaumWelch(obs, off, wos, W, N, M) as bw:
        bw.set_params(*init)
        for _ in range(calls):
            bw.iterate(iters // calls, -1.0, iters, sync_each=sync_each)
        return bw.params() + bw.history(iters) + (bw.thin_states(),)


def _check(got, seqs, wos, W, N, M, init, iters, rtol=1e-9):
    pi, A, B, hist, it, _ = got
    for w in range(W):
        mine = [seqs[r] for r in range(len(seqs)) if wos[r] == w]
        Ao, Bo, pio, ho, _ = O.hmm_training(mine, N=N, M=M, epsilon=-1.0, max_iterations=iters,
                                            init=(init[0][w], init[1][w], init[2][w]), return_history=True)
        assert_close(A[w], Ao, f"A of word {w}", rtol=rtol); assert_close(B[w], Bo, f"B of word {w}", rtol=rtol)
        assert_close(pi[w], pio, f"pi of word {w}", rtol=rtol)
        assert_same_support(A[w], Ao, "A"); assert_same_support(pi[w], pio, "pi")
        assert np.array_equal(floored_set(B[w], M), floored_set(Bo, M))
        assert_close(hist[w, :iters], np.array(ho), "statistic", rtol=rtol, atol=1e-12)


def test_property_test_counterexample_is_pinned():
    """N = 16, M = 5, one sequence per word of 15 / 6 / 28 frames, 4 iterations: the reference keeps
    a_13,13 = 0.39397 for word 0 while the row's posterior mass is ~1e-340."""
    from hmm_training_b200 import engine
    N, M, W, S, seed = 16, 5, 3, 1, 1333002
    rng = np.random.default_rng(seed)
    init = _random_model(rng, W, N, M, True, 0.0)
    seqs, wos = _random_corpus(rng, W, S, 1, 60, M)
    assert [len(s) for s in seqs] == [15, 6, 28]
    got = _fit(engine, seqs, wos, W, N, M, init, 4)
    _check(got, seqs, wos, W, N, M, init, 4)
    assert got[5] >= 1  # at least one state was rescued


@pytest.mark.parametrize("N,M,kernel", [(4, 256, "n4"), (4, 24, "n4"), (8, 40, "ltr"), (5, 16, "generic")])
def test_tail_states_the_data_never_reaches(N, M, kernel):
    """Utterances with two acoustic segments on a model with N >= 4 states: the tail states die — their posterior
    shrinks super-exponentially with the iterations, through 1e-100, 1e-250, below 1e-308 — while the reference's
    rows for them stay well defined.  15 iterations, every iterate against the oracle."""
    from hmm_training_b200 import engine
    rng = np.random.default_rng(7 * N + M)
    W, S = 2, 40
    seqs, wos = [], []
    for w in range(W):
        for _ in range(S):
            T = int(rng.integers(30, 50))
            cut = int(rng.integers(10, T - 10))
            a = rng.integers(0, max(M // 4, 2), size=cut) + w
            b = rng.integers(M // 2, M // 2 + max(M // 4, 2), size=T - cut)
            seqs.append(np.concatenate([a, b]).astype(np.int64) % M)
            wos.append(w)
    wos = np.array(wos, dtype=np.int32)
    pi0 = np.zeros((W, N)); pi0[:, 0] = 1.0
    A0 = np.zeros((W, N, N))
    for i in range(N):
        A0[:, i, i] = 0.6
        if i + 1 < N:
            A0[:, i, i + 1] = 0.4
        else:
            A0[:, i, i] = 1.0
    B0 = rng.random((W, N, M)) + 0.2
    B0 /= B0.sum(axis=2, keepdims=True)
    init = (pi0, A0, B0)
    iters = 15
    got = _fit(engine, seqs, wos, W, N, M, init, iters)
    _check(got, seqs, wos, W, N, M, init, iters)


def test_states_flagged_between_calls_without_host_sync():
    """sync_each = 0 queues the iterations: a state flagged on the device gets its slot at the end of the call, i.e.
    from the next hmmb_bw_iterate on (DESIGN.md section 4).  Iterations run one per call here, so the flag of
    iteration k is in force in iteration k + 1 — early enough as long as the row's mass is still representable when
    it is flagged (2^-200 leaves 800 binades)."""
    from hmm_training_b200 import engine
    N, M, W, S, seed = 16, 5, 3, 1, 1333002
    rng = np.random.default_rng(seed)
    init = _random_model(rng, W, N, M, True, 0.0)
    seqs, wos = _random_corpus(rng, W, S, 1, 60, M)
    got = _fit(engine, seqs, wos, W, N, M, init, 4, sync_each=False, calls=4)
    _check(got, seqs, wos, W, N, M, init, 4)


def test_thin_states_over_virtual_ranks():
    """Two virtual ranks on one device (tests/test_properties.py): the rescue slots ride behind the accumulators in
    the buffer the hook sums, one region per rank, and a newly flagged state repeats the iteration — i.e. the hook
    runs twice in that iteration, with a longer buffer the second time."""
    from hmm_training_b200 import dist, engine
    N, M, W, G, iters = 16, 5, 2, 2, 4
    rng = np.random.default_rng(99)
    init = _random_model(rng, W, N, M, True, 0.0)
    seqs, wos = [], []
    for w in range(W):  # one short sequence (the thin state) and a few more per word
        for T in (15, 17, 16, 18):
            seqs.append(rng.integers(0, M, size=T).astype(np.int64)); wos.append(w)
    wos = np.array(wos, dtype=np.int32)
    want = _fit(engine, seqs, wos, W, N, M, init, iters)
    _check(want, seqs, wos, W, N, M, init, iters)
    shards = [dist.shard_sequences_round_robin(wos, r, G) for r in range(G)]
    got, _, calls = run_virtual_ranks(shards, lambda idx: _pack([seqs[i] for i in idx]), wos, W, N, M, init, iters)
    assert calls > iters  # at least one iteration was repeated
    for x, y, name in zip(got[:5], want[:5], ("pi", "A", "B", "statistic", "iterations")):
        assert_close(x, y, f"{G} virtual ranks: {name}", rtol=1e-9, atol=1e-12)
    assert got[5] == want[5] >= 1


@pytest.mark.parametrize("family", ["left_to_right", "generic"])
def test_backward_rescale_keeps_denormal_markers(family, monkeypatch):
    """Second find of the property tests (N = 16, M = 256, one sequence of 8 / 5 / 13 frames per word, 4 iterations):
    b_0(253) of word 2 is 0.0 in the reference — a finite log value below -745 — but came out as the 1e-20 floor
    ("no finite term") because the careful backward step rescaled beta-hat by a power of two BELOW one (the sum of
    N states' values can reach 2 N) and flushed the denormal marker of state 0 to zero, after which gamma had no
    way to stay positive."""
    from hmm_training_b200 import engine
    if family == "generic":
        monkeypatch.setenv("HMMB_NO_LTR", "1")
    N, M, W, S, seed = 16, 256, 3, 1, 197
    rng = np.random.default_rng(seed)
    init = _random_model(rng, W, N, M, True, 0.0)
    seqs, wos = _random_corpus(rng, W, S, 1, 60, M)
    assert [len(s) for s in seqs] == [8, 5, 13]
    obs, off = _pack(seqs)
    with engine.BaumWelch(obs, off, wos, W, N, M) as bw:
        bw.set_params(*init)
        assert bw.kernel_family() == family
        bw.iterate(4, -1.0, 4)
        got = bw.params() + bw.history(4) + (bw.thin_states(),)
    _check(got, seqs, wos, W, N, M, init, 4)

"""The N = 4 E-step rebuilds odd-step alpha-hat rows in the backward pass (DESIGN.md §3).

k_bw_fwd4 writes the alpha-hat row of every even step, and of an odd step only for the lanes whose step was not plain
(all four states alive, t > 0, no exponent-split products); k_bw_bwd4 recomputes the other odd rows from the even row
before them with the forward pass's own step (fwd4_rebuild).  The rebuilt values must be the forward pass's bits, so
every case here trains the same problem twice, with the default rows and with HMMB_FULL_SPILL=1 (every row written and
read back), and asks for exactly equal parameters, log-likelihood history, per-sequence log-likelihoods, thin-state
count and hand-over counters (to rounding only where the exact kernel's atomics ran, see _same).  A few cases also meet
the oracle.

Cases: a reduced config-3 corpus (every odd row rebuilt), the same from pi = e_0 (t = 1 is a masked step whose row
comes from the spill), dense A, M = 300 (the runtime-M kernel), a word whose B holds exact zeros (codewords kill states
at odd steps, the lean backward path is off), ragged lengths from 1 frame on with odd and even T in one block, the
forward and backward hand-over constructions of test_gpu_handover.py (exponent-split steps at odd t: after the first
frame such a step always hands the sequence over, the error bound being positive), the pipelined create, codewords
already on the device, and three queued iterations.
"""
import numpy as np
import pytest

from helpers import assert_close
from test_gpu_handover import (_backward_corpus, _backward_model, _check_training, _forward_train_case, _pack, _seed,
                               _tile, dev)  # noqa: F401 (dev: fixture)

ROUTES = ("HMMB_FORCE_GENERIC", "HMMB_NO_LTR", "HMMB_FORCE_DENSE_A", "HMMB_FULL_SPILL")


def _config3(W=10, S=3000, T=200):
    from hmm_training_b200 import engine, synthetic
    obs, off, wos = synthetic.fixed_length_codewords(_seed("spill_c3"), W, S, T, 4, 256)
    pi0, A0, B0 = engine.default_init(4, 256)
    return obs, off, wos, (np.tile(pi0, (W, 1)), np.tile(A0, (W, 1, 1)), np.tile(B0, (W, 1, 1)))


def _run(monkeypatch, full, obs, off, wos, W, N, M, init, iters=3, sync_each=True, switch=None, **kw):
    """Train with or without HMMB_FULL_SPILL: (family, outputs by name)."""
    from hmm_training_b200 import engine
    for env in ROUTES:
        monkeypatch.delenv(env, raising=False)
    if switch:
        monkeypatch.setenv(switch, "1")
    if full:
        monkeypatch.setenv("HMMB_FULL_SPILL", "1")
    pipelined = kw.pop("pipeline_upload", False)
    with engine.BaumWelch(obs, off, wos, W, N, M, pipeline_upload=pipelined, init=init if pipelined else None,
                          **kw) as bw:
        if not pipelined:
            bw.set_params(*init)
        family = bw.kernel_family()
        bw.iterate(iters, -1.0, iters, sync_each=sync_each)
        pi, A, B = bw.params()
        hist, its = bw.history(iters)
        out = dict(pi=pi, A=A, B=B, hist=hist, iters=its, seq_ll=bw.seq_ll(),
                   diag=np.array(bw.diagnostics()), thin=np.array(bw.thin_states()))
    return family, out


def _same(monkeypatch, family, *args, **kw):
    """Default rows against every row spilled: bit-identical outputs.  Returns the default run's outputs.

    Where the exact log-space kernel ran (hand-overs), its fp64 atomics make everything that follows the first
    iteration's statistic agree between two runs only to rounding, whichever rows are spilled (test_gpu_handover.py
    holds the pipelined create to the same rule); there the counters, the first statistic and the iteration counts
    must still be equal, the rest agree to 1e-11."""
    fam0, got = _run(monkeypatch, False, *args, **kw)
    fam1, ref = _run(monkeypatch, True, *args, **kw)
    assert fam0 == fam1 == family
    assert np.array_equal(got["diag"], ref["diag"])
    if got["diag"].sum() == 0:
        for k in got:
            assert np.array_equal(got[k], ref[k], equal_nan=True), f"{k}: rebuilt rows differ from spilled rows"
    else:
        assert np.array_equal(got["hist"][:, 0], ref["hist"][:, 0]), "first statistic"
        assert np.array_equal(got["iters"], ref["iters"])
        for k in ("pi", "A", "B", "hist"):
            assert_close(got[k], ref[k], f"{k}: rebuilt against spilled rows", rtol=1e-11)
    return got


def _as_tuple(out):
    return (out["pi"], out["A"], out["B"], out["hist"], out["iters"], int(out["thin"]))


@pytest.mark.gpu
def test_config3_every_odd_row_rebuilt(monkeypatch):
    obs, off, wos, init = _config3()
    got = _same(monkeypatch, "n4_left_to_right", obs, off, wos, 10, 4, 256, init)
    assert tuple(got["diag"]) == (0, 0)


@pytest.mark.gpu
def test_config3_pi_e0_masked_first_steps(monkeypatch):
    obs, off, wos, init = _config3(W=4, S=1500)
    pi = np.zeros_like(init[0])
    pi[:, 0] = 1.0
    _same(monkeypatch, "n4_left_to_right", obs, off, wos, 4, 4, 256, (pi,) + init[1:])


@pytest.mark.gpu
def test_dense_a(monkeypatch):
    obs, off, wos, init = _config3(W=4, S=800, T=101)
    rng = np.random.default_rng(_seed("spill_dense"))
    A = rng.dirichlet(np.ones(4), size=(4, 4))
    _same(monkeypatch, "n4_dense", obs, off, wos, 4, 4, 256, (init[0], A, init[2]))


@pytest.mark.gpu
def test_dense_a_forced(monkeypatch):
    obs, off, wos, init = _config3(W=3, S=600, T=77)
    _same(monkeypatch, "n4_dense", obs, off, wos, 3, 4, 256, init, switch="HMMB_FORCE_DENSE_A")


@pytest.mark.gpu
def test_runtime_m300(monkeypatch):
    from hmm_training_b200 import engine, synthetic
    W, S, T, M = 3, 700, 151, 300
    obs, off, wos = synthetic.fixed_length_codewords(_seed("spill_m300"), W, S, T, 4, M)
    pi0, A0, B0 = engine.default_init(4, M)
    init = (np.tile(pi0, (W, 1)), np.tile(A0, (W, 1, 1)), np.tile(B0, (W, 1, 1)))
    _same(monkeypatch, "n4_left_to_right", obs, off, wos, W, 4, M, init)


def _ragged(rng, W, S, M, lo, hi):
    seqs = []
    for _ in range(W * S):
        T = int(rng.integers(lo, hi + 1))
        seqs.append(rng.integers(0, M, size=T).astype(np.int64))
    seqs[:6] = [s[:n] for s, n in zip(seqs[:6], (1, 2, 3, 1, 2, 3))]  # the shortest lengths, in word 0
    return seqs, np.repeat(np.arange(W, dtype=np.int32), S)


@pytest.mark.gpu
def test_zeros_in_b_kill_states_at_odd_steps(monkeypatch):
    from hmm_training_b200 import engine
    W, S, M = 2, 160, 16
    rng = np.random.default_rng(_seed("spill_zero_b"))
    seqs, wos = _ragged(rng, W, S, M, 4, 40)
    pi0, A0, B0 = engine.default_init(4, M)
    B = np.tile(B0, (W, 1, 1))
    B[0, 1, 3] = B[0, 2, 3] = 0.0  # codeword 3 kills states 1 and 2 of word 0
    B[0, 0, 5] = 0.0               # codeword 5 kills state 0
    B /= B.sum(axis=2, keepdims=True)
    init = (np.tile(pi0, (W, 1)), np.tile(A0, (W, 1, 1)), B)
    obs, off = _pack(seqs, np.uint8)
    got = _same(monkeypatch, "n4_left_to_right", obs, off, wos, W, 4, M, init)
    _check_training(_as_tuple(got), seqs, wos, W, 4, M, init)


@pytest.mark.gpu
def test_ragged_lengths_from_one_frame(monkeypatch):
    from hmm_training_b200 import engine
    W, S, M = 3, 200, 16
    rng = np.random.default_rng(_seed("spill_ragged"))
    seqs, wos = _ragged(rng, W, S, M, 1, 45)
    pi0, A0, B0 = engine.default_init(4, M)
    init = (np.tile(pi0, (W, 1)), np.tile(A0, (W, 1, 1)), np.tile(B0, (W, 1, 1)))
    obs, off = _pack(seqs, np.uint8)
    got = _same(monkeypatch, "n4_left_to_right", obs, off, wos, W, 4, M, init)
    _check_training(_as_tuple(got), seqs, wos, W, 4, M, init)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["n4_m16", "n4_m256", "n4_m300", "n4_dense", "bound_n4_m16"])
def test_forward_handover_lanes_share_blocks(name, monkeypatch):
    from test_gpu_handover import TRAIN_CASES
    N, M, _, _, family, dtype = TRAIN_CASES[name]
    W = 3
    seqs, wos, ho, init = _forward_train_case(name, W)
    obs, off = _pack(seqs, dtype)
    got = _same(monkeypatch, family, obs, off, wos, W, N, M, init)
    assert got["diag"][0] > 0
    _check_training(_as_tuple(got), seqs, wos, W, N, M, init)


@pytest.mark.gpu
@pytest.mark.parametrize("switch,family", [(None, "n4_left_to_right"), ("HMMB_FORCE_DENSE_A", "n4_dense")])
def test_backward_handover_redo(switch, family, monkeypatch):
    W, N, M = 2, 4, 8
    rng = np.random.default_rng(_seed("n4"))
    seqs, wos, ho = _backward_corpus(rng, W, M)
    init = _tile(_backward_model(N, M), W)
    obs, off = _pack(seqs, np.uint8)
    got = _same(monkeypatch, family, obs, off, wos, W, N, M, init, switch=switch)
    assert got["diag"][1] > 0


@pytest.mark.gpu
def test_pipelined_create(monkeypatch):
    obs, off, wos, init = _config3(W=10, S=3000)
    _same(monkeypatch, "n4_left_to_right", obs, off, wos, 10, 4, 256, init, pipeline_upload=True)


@pytest.mark.gpu
def test_codewords_on_device(monkeypatch, dev):
    obs, off, wos, init = _config3(W=4, S=1000, T=120)
    _same(monkeypatch, "n4_left_to_right", None, off, wos, 4, 4, 256, init, obs_dev_ptr=dev(obs).data_ptr(),
          idx_bytes=obs.itemsize)


@pytest.mark.gpu
def test_three_queued_iterations(monkeypatch):
    obs, off, wos, init = _config3(W=4, S=1000, T=200)
    _same(monkeypatch, "n4_left_to_right", obs, off, wos, 4, 4, 256, init, sync_each=False)

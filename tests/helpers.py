"""Shared test helpers: tolerances from BASELINE.md §4 / SURVEY.md §8c."""
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# |x - x_ref| <= RTOL*|x_ref| + ATOL.  ATOL sits 10 orders below the reference's 1e-20
# emission floor so a mis-floored B entry is still caught.
RTOL = 1e-9
ATOL = 1e-30


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def split_corpus(g):
    """golden npz -> list (per word) of list of int64 sequences."""
    obs, off, wos = g["obs"], g["offsets"], g["word_of_seq"]
    W = int(wos.max()) + 1 if len(wos) else 0
    corpus = [[] for _ in range(W)]
    for r in range(len(wos)):
        corpus[int(wos[r])].append(obs[off[r]:off[r + 1]].astype(np.int64))
    return corpus


def assert_close(x, ref, what="", rtol=RTOL, atol=ATOL):
    x = np.asarray(x, dtype=float)
    ref = np.asarray(ref, dtype=float)
    assert x.shape == ref.shape, f"{what}: shape {x.shape} vs {ref.shape}"
    both_nan = np.isnan(x) & np.isnan(ref)
    same_inf = np.isinf(ref) & (x == ref)
    with np.errstate(invalid="ignore"):
        ok = both_nan | same_inf | (np.abs(x - ref) <= rtol * np.abs(ref) + atol)
    if not ok.all():
        bad = np.argwhere(~ok)[:5]
        msgs = [f"{tuple(b)}: got {x[tuple(b)]!r} want {ref[tuple(b)]!r}" for b in bad]
        raise AssertionError(f"{what}: {int((~ok).sum())} of {ok.size} outside tolerance; " + "; ".join(msgs))


def assert_same_support(x, ref, what=""):
    """Zero pattern must match exactly (structural zeros of A / pi)."""
    assert np.array_equal(np.asarray(x) == 0, np.asarray(ref) == 0), f"{what}: zero pattern differs"


def floored_set(B, M):
    """Entries produced by the reference's log(1e-20) floor (HMM/hmm_training.py:497):
    after the final row renormalisation they are 1e-20/rowsum, i.e. within a factor
    ~[1/(1+M*1e-20), 1] of 1e-20 — anything in [0.5e-20, 1.5e-20] qualifies."""
    B = np.asarray(B)
    return (B > 0.5e-20) & (B < 1.5e-20)


def run_virtual_ranks(shards, pack, wos, W, N, M, init, iters):
    """G "virtual ranks" on one device in lock step: rank r trains on the sequences shards[r] (pack(indices) ->
    (obs, offsets)) with an all-reduce hook that the emulation serves.  Pass k runs every rank and records each rank's
    buffer of hook call k; the hook calls before it are served the sums recorded so far, so that each rank sees the
    reduced buffers up to that call and produces its next one from correct parameters.  A pass whose hook calls were all
    served is the G-rank run.  Returns (pi, A, B, history, iterations, thin states) of that run, every rank's
    diagnostics() in it, and the number of hook calls per rank."""
    import ctypes

    from hmm_training_b200 import engine
    rt = ctypes.CDLL("libcudart.so.12")
    rt.cudaMemcpy.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int]
    rt.cudaDeviceSynchronize.argtypes = []
    G = len(shards)
    sums = []
    for _ in range(64):
        recorded, diags = [], []
        for r in range(G):
            mine, k = [], [0]

            def hook(ptr, n, mine=mine, k=k):
                assert rt.cudaDeviceSynchronize() == 0
                if k[0] < len(sums):
                    assert n == len(sums[k[0]])
                    assert rt.cudaMemcpy(ptr, sums[k[0]].ctypes.data, n * 8, 1) == 0
                else:
                    buf = np.empty(n)
                    assert rt.cudaMemcpy(buf.ctypes.data, ptr, n * 8, 2) == 0
                    mine.append(buf)
                k[0] += 1

            obs, off = pack(shards[r])
            with engine.BaumWelch(obs, off, wos[shards[r]], W, N, M) as bw:
                bw.set_params(*init)
                bw.set_dist(r, G, hook)
                bw.iterate(iters, -1.0, iters)
                got = bw.params() + bw.history(iters) + (bw.thin_states(),)
                diags.append(bw.diagnostics())
            recorded.append(mine)
        if not recorded[0]:
            return got, diags, len(sums)
        assert all(len(m) >= 1 for m in recorded)
        sums.append(np.sum([m[0] for m in recorded], axis=0))
    raise AssertionError("the hook calls did not settle")

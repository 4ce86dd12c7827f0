"""How the trainer and the scorer cut large, skewed, ragged corpora into work items, against the numpy oracle.

The other oracle comparisons use a few small words: each becomes one CTA work item.  Here the corpora are shaped like
real vocabularies — one giant word, a few mid-sized ones, hundreds of tiny ones (partial blocks), empty words, a word
of T = 1 recordings, a word with one recording of thousands of frames among short ones, heavy-tailed lengths — and
large enough that the host-side partition (seqset_build in csrc/bw.cu) takes the regimes that only exist at scale:

  * N = 4: exactly 2 x sm backward work items shared out to the words by largest remainder (more items than that when
    there are more words), a separate forward list, fat backward CTAs running several warp-rounds per item (16 warps
    for a bidiagonal A, 12 for a dense one), and the finer list of the staged first E-step of a pipelined create;
  * N = 5: the lanes-per-state kernels with several sequences per group, so that groups span word boundaries;
  * N = 8 / 16 left-to-right: several serpentine rounds per CTA, and the backward pass in word groups with the
    all-reduce hook called per group (hmmb_bw_set_overlap), run here on one device with two virtual ranks;
  * scoring: k_score4r, k_score4, k_scoreL (several rounds), k_scoreG and the pipelined scorer.

Every threshold is computed from the device's SM count and asserted with a margin, so a case cannot silently fall
back to a smaller regime.  Training is checked word by word and sequence by sequence: a block visited twice or
skipped, or a partial combined into the wrong word, hides in no aggregate property but shows in the per-word
parameters and in the per-sequence log-likelihoods.
"""
import ctypes
import os
import time

import numpy as np
import pytest

from helpers import assert_close, assert_same_support, floored_set
from oracle import hmm_oracle as O

pytestmark = pytest.mark.gpu

# Tuning constants of csrc/bw.cu, bw4_kernels.cuh, bwltr_kernels.cuh that decide the partition.
BWD4_MAX_WARPS = 16   # warps of the fat N = 4 backward CTA (bidiagonal A)
LTR_WARPS = 8         # warps of a left-to-right CTA
BW_WARPS = 4          # warps of the generic (lanes-per-state) CTA
MARGIN = 1.05         # every case exceeds its regime's threshold by at least 5 %


# ---------------------------------------------------------------------------------------------- corpora
def _heavy_tailed_lengths(rng, n):
    """1..64 frames, with 6 % of the recordings from a log-uniform tail up to 300."""
    T = rng.integers(1, 65, size=n)
    tail = rng.random(n) < 0.06
    T[tail] = np.exp(rng.uniform(np.log(65), np.log(301), size=int(tail.sum()))).astype(np.int64)
    return T.astype(np.int64)


def _ltr_codewords(rng, lens, N, M, shift):
    """Left-to-right structured codewords (as synthetic.clustered_sequences, vectorised): a recording is cut into N
    segments at sorted random points and segment s emits (M // N) * s + shift + U{0..spread-1} (mod M)."""
    F = int(lens.sum())
    if F == 0:
        return np.zeros(0, np.int64)
    spread = max(2, M // (2 * N))
    start = np.concatenate([[0], np.cumsum(lens)[:-1]])
    seq = np.repeat(np.arange(len(lens)), lens)
    t = np.arange(F) - start[seq]
    seg = np.zeros(F, np.int64)
    if N > 1:
        cuts = np.sort(rng.integers(0, lens[:, None] + 1, size=(len(lens), N - 1)), axis=1)
        for c in range(N - 1):
            seg += t >= cuts[seq, c]
    return ((M // N) * seg + shift + rng.integers(0, spread, size=F)) % M


class Corpus:
    """Words in a fixed order; `lens` / `word` / `start` describe every recording (word-major, generation order)."""

    def __init__(self, N, M, sizes, seed):
        rng = np.random.default_rng(seed)
        self.N, self.M, self.W = N, M, len(sizes)
        lens, words, flat = [], [], []
        for w, (kind, S) in enumerate(sizes):
            if kind == "T1":
                L = np.ones(S, np.int64)
            elif kind == "long":  # one recording of 3000 frames among short ones: its block's tmax dwarfs the rest
                L = rng.integers(1, 41, size=S)
                L[S // 2] = 3000
            else:
                L = _heavy_tailed_lengths(rng, S)
            lens.append(L)
            words.append(np.full(S, w, np.int32))
            flat.append(_ltr_codewords(rng, L, N, M, (7 * w) % M))
        self.lens = np.concatenate(lens)
        self.word = np.concatenate(words)
        self.obs = np.concatenate(flat).astype(np.uint8 if M <= 256 else np.uint16)
        self.start = np.concatenate([[0], np.cumsum(self.lens)[:-1]]).astype(np.int64)
        self.R = len(self.lens)
        self.counts = np.bincount(self.word, minlength=self.W)
        self.nblk = int(sum((S + 31) // 32 for S in self.counts))

    def seq(self, r):
        return self.obs[self.start[r]:self.start[r] + self.lens[r]]

    def packed(self, order):
        """(obs, offsets, word_of_seq) with the recordings in `order`."""
        L = self.lens[order]
        off = np.concatenate([[0], np.cumsum(L)]).astype(np.int64)
        idx = np.repeat(self.start[order], L) + (np.arange(int(off[-1])) - np.repeat(off[:-1], L))
        return self.obs[idx], off, self.word[order]

    def shuffled(self, seed=1):
        return np.random.default_rng(seed).permutation(self.R)

    def sorted(self):
        """(word, length descending): the order the library sorts into, and that the pipelined create needs."""
        return np.lexsort((-self.lens, self.word))


def skewed_sizes(giant_blocks, n_tiny=320, n_mid=0):
    """One giant word (its last block holds 5 sequences), mid-sized words whose last items end in partial blocks
    (517 = 16 * 32 + 5), n_tiny tiny words of 1..40 sequences, an empty word in the middle and one at the end, a word
    of T = 1 recordings and a word with one 3000-frame recording; optionally n_mid more words of 40..200 blocks, each
    ending in a partial block."""
    rng = np.random.default_rng(7)
    sizes = [("ragged", 517), ("ragged", 32 * giant_blocks - 27), ("ragged", 0), ("T1", 45), ("long", 70),
             ("ragged", 1203), ("ragged", 2990)]
    sizes += [("ragged", 32 * int(rng.integers(40, 200)) + int(rng.integers(1, 32))) for _ in range(n_mid)]
    for k in range(n_tiny):
        sizes.append(("ragged", int(rng.integers(1, 41))))
        if k == n_tiny // 2:
            sizes.append(("ragged", 0))
    sizes.append(("ragged", 0))
    return sizes


def corpus_for(N, M, seed, min_blocks=0, min_seqs=0, **shape):
    """The skewed corpus with the giant word sized so that the corpus has at least min_blocks blocks and min_seqs
    sequences (and not many more).  `shape`: n_tiny / n_mid of skewed_sizes."""
    other = skewed_sizes(1, **shape)
    other_blocks = sum((S + 31) // 32 for _, S in other) - 1
    other_seqs = sum(S for _, S in other) - 5
    giant = max(1, int(np.ceil(min_blocks)) - other_blocks, -(-(int(np.ceil(min_seqs)) - other_seqs + 27) // 32))
    c = Corpus(N, M, skewed_sizes(giant, **shape), seed)
    assert c.nblk >= min_blocks and c.R >= min_seqs
    return c


def _sm_count():
    from hmm_training_b200 import _lib
    return int(_lib.device_info()["sm_count"])


# ---------------------------------------------------------------------------------------------- partition (mirror)
def n4_items(counts, sm):
    """The N = 4 partition of seqset_build in numbers: blocks, backward / forward / finer work items, the items the
    largest-remainder step hands out on top of every word's floor share, the most items one word gets besides the
    largest word, and the largest item in blocks."""
    nb = [(S + 31) // 32 for S in counts]
    nblk, target = sum(nb), 2 * sm
    bpc = max(1, -(-nblk // target))
    if bpc > 1:
        bpc = -(-bpc // BWD4_MAX_WARPS) * BWD4_MAX_WARPS
    exact = nblk >= target * BWD4_MAX_WARPS * 2
    leftover = 0
    if exact:
        q = [b * target / nblk for b in nb]
        items = [max(1, int(x)) if b else 0 for x, b in zip(q, nb)]
        rem = sorted(((x - int(x), w) for w, (x, b) in enumerate(zip(q, nb)) if b), key=lambda r: (-r[0], r[1]))
        leftover = max(0, min(len(rem), target - sum(items)))
        for _, w in rem[:leftover]:
            items[w] += 1
        items = [min(i, b) for i, b in zip(items, nb)]  # (an item of no block is dropped)
    else:
        items = [-(-b // bpc) for b in nb]
    largest = max(b / i for b, i in zip(nb, items) if i)
    bpf = max(1, -(-nblk // (8 * sm)))
    if bpf > 1:
        bpf = -(-bpf // BWD4_MAX_WARPS) * BWD4_MAX_WARPS
    fine = sum(-(-b // bpf) for b in nb) if bpf < bpc else 0
    return {"blocks": nblk, "exact_items": exact, "bwd_items": sum(items), "leftover_items": leftover,
            "most_items_of_another_word": sorted(items)[-2], "fwd_items": sum(-(-b // bpc) for b in nb),
            "fine_items": fine, "largest_item_blocks": largest}


def ltr_rounds(nblk, sm):
    """Blocks per left-to-right work item and warp-rounds of a full item (seqset_build: ~4 items per SM)."""
    bpc = max(1, -(-nblk // (4 * sm)))
    bpc = -(-bpc // LTR_WARPS) * LTR_WARPS
    return bpc, bpc // LTR_WARPS


# ---------------------------------------------------------------------------------------------- oracle
_ORACLE = None  # (sequences, per-word log parameters, M): read by the forked pool workers


def _oracle_job(job):
    w, idx = job
    seqs, logs, M = _ORACLE
    s = O.estep_logsums([seqs[r] for r in idx], *logs[w], M)
    return w, idx, s


def oracle_em(c, raw):
    """One EM iteration of every word from the raw parameters `raw` (the oracle's estep_logsums / merge_logsums /
    mstep_from_logsums / finalize_params, sequences of a word chunked and spread over a process pool).
    Returns per word (A, B, pi, statistic) and the per-sequence log-likelihood of every recording."""
    global _ORACLE
    import multiprocessing as mp
    N, M = c.N, c.M
    pi, A, B = raw
    logs = [(O.safe_log(pi[w]), O.safe_log(A[w]), O.safe_log(B[w])) for w in range(c.W)]
    jobs = []
    budget = 6_000_000 // (N * N)  # padded frames per chunk: ~50 MB for the xi terms
    for w in range(c.W):
        mine = np.flatnonzero(c.word == w)
        mine = mine[np.argsort(-c.lens[mine], kind="stable")]  # long first: little padding per chunk
        i = 0
        while i < len(mine):
            n = max(1, budget // int(c.lens[mine[i]]))
            jobs.append((w, mine[i:i + n]))
            i += n
    jobs.sort(key=lambda j: -int(c.lens[j[1]].sum()))  # big jobs first
    _ORACLE = ([c.seq(r) for r in range(c.R)], logs, M)
    try:
        procs = max(1, min(len(os.sched_getaffinity(0)), 32))
        with mp.get_context("fork").Pool(procs) as pool:
            parts = pool.map(_oracle_job, jobs, chunksize=1)
    finally:
        _ORACLE = None
    seq_ll = np.full(c.R, np.nan)
    per_word = [[] for _ in range(c.W)]
    for w, idx, s in parts:
        seq_ll[idx] = s["seq_ll"]
        per_word[w].append(s)
    out = []
    for w in range(c.W):
        if not per_word[w]:
            A_, B_, pi_, h, _ = O.hmm_training([], N=N, M=M, max_iterations=1, return_history=True)
            out.append((A_, B_, pi_, h[0]))
            continue
        s = O.merge_logsums(per_word[w])
        A_, B_, pi_ = O.finalize_params(*O.mstep_from_logsums(s, N, M))
        out.append((A_, B_, pi_, s["ll"]))
    return out, seq_ll


# ---------------------------------------------------------------------------------------------- runs and checks
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


class launches_of:
    """Counts the kernel launches of one library phase (HMMB_LAUNCH name) inside a `with` block, through the library's
    per-launch profiling events: a way to assert which path a call took."""

    def __init__(self, phase):
        self.phase, self.n = phase.encode(), None

    def __enter__(self):
        from hmm_training_b200 import _lib
        lib = _lib.load()
        _lib.check(lib.hmmb_set_profiling(1))
        _lib.check(lib.hmmb_phase_reset())
        return self

    def __exit__(self, *exc):
        from hmm_training_b200 import _lib
        lib = _lib.load()
        n = ctypes.c_int64(0)
        lib.hmmb_phase_ms(self.phase, ctypes.byref(n))
        self.n = n.value
        _lib.check(lib.hmmb_set_profiling(0))


def tiled(init, W):
    pi, A, B = init
    return np.tile(pi, (W, 1)), np.tile(A, (W, 1, 1)), np.tile(B, (W, 1, 1))


def gpu_em(c, order, init, family, pipelined=False, obs_dtype=None):
    """Two EM iterations, the raw parameters, one more iteration.  Results are returned in the corpus' own
    recording order (seq_ll) whatever `order` the recordings were fed in."""
    from hmm_training_b200 import engine
    obs, off, wos = c.packed(order)
    if obs_dtype is not None:
        obs = obs.astype(obs_dtype)
    handle = None
    if pipelined:
        obs, handle = _pinned_copy(obs)
    fwd = launches_of("bw_forward")
    try:
        with fwd, engine.BaumWelch(obs, off, wos, c.W, c.N, c.M, pipeline_upload=pipelined,
                              init=init if pipelined else None) as bw:
            if not pipelined:
                bw.set_params(*init)
            assert bw.kernel_family() == family
            bw.iterate(2, -1.0, 3)
            raw = bw.params(finalize=False)
            bw.iterate(1, -1.0, 3)
            pi, A, B = bw.params()
            hist, iters = bw.history(3)
            ll = np.empty(c.R)
            ll[order] = bw.seq_ll()
    finally:
        if handle is not None:
            _host_free(handle)
    return {"raw": raw, "pi": pi, "A": A, "B": B, "hist": hist, "iters": iters, "seq_ll": ll, "fwd_launches": fwd.n}


def check_against_oracle(what, c, got, want):
    """Every word's pi / A / B / statistic at the contract's tolerance, the zero pattern of A and pi, the floored-B
    set, the iteration counts, and every recording's log-likelihood."""
    per_word, seq_ll = want
    assert np.array_equal(got["iters"], np.full(c.W, 3)), f"{what}: iteration counts {np.unique(got['iters'])}"
    bad = []
    for w in range(c.W):
        A_, B_, pi_, stat = per_word[w]
        try:
            assert_close(got["pi"][w], pi_, f"w{w} pi")
            assert_close(got["A"][w], A_, f"w{w} A")
            assert_close(got["B"][w], B_, f"w{w} B")
            assert_close(got["hist"][w, 2], stat, f"w{w} statistic")
            assert_same_support(got["A"][w], A_, f"w{w} A")
            assert_same_support(got["pi"][w], pi_, f"w{w} pi")
            assert np.array_equal(floored_set(got["B"][w], c.M), floored_set(B_, c.M)), f"w{w}: floored B set"
        except AssertionError as e:
            bad.append(f"[{c.counts[w]} seqs] {e}")
    assert not bad, f"{what}: {len(bad)} of {c.W} words differ from the oracle: " + " | ".join(bad[:4])
    with np.errstate(invalid="ignore"):
        wrong = ~((got["seq_ll"] == seq_ll) | (np.abs(got["seq_ll"] - seq_ll) <= 1e-9 * np.abs(seq_ll)))
    if wrong.any():
        r = np.flatnonzero(wrong)[:5]
        raise AssertionError(f"{what}: {int(wrong.sum())} of {c.R} per-sequence log-likelihoods differ, e.g. recordings "
                             f"{list(r)} of words {list(c.word[r])}: {got['seq_ll'][r]} vs {seq_ll[r]}")


def check_same(what, a, b, rtol):
    for k in ("pi", "A", "B", "hist"):
        assert_close(a[k], b[k], f"{what}: {k}", rtol=rtol, atol=0)
    for k in ("raw",):
        for x, y, name in zip(a[k], b[k], ("pi", "A", "B")):
            assert_close(x, y, f"{what}: raw {name}", rtol=rtol, atol=0)
    assert_close(a["seq_ll"], b["seq_ll"], f"{what}: per-sequence LL", rtol=rtol, atol=0)
    assert np.array_equal(a["iters"], b["iters"])


# ---------------------------------------------------------------------------------------------- N = 4
@pytest.fixture(scope="module")
def n4():
    """Case (a)'s corpus and run, and the oracle from its raw parameters (shared by cases (a) and (c))."""
    from hmm_training_b200 import engine
    sm = _sm_count()
    c = corpus_for(4, 256, 41, min_blocks=MARGIN * 2 * sm * BWD4_MAX_WARPS * 2)
    part = n4_items(c.counts, sm)
    print(f"N = 4 corpus: W = {c.W}, {c.R} sequences, {len(c.obs)} frames, SMs = {sm}, partition {part}")
    assert part["exact_items"] and part["blocks"] >= MARGIN * 2 * sm * BWD4_MAX_WARPS * 2
    assert c.W > 2 * sm and part["bwd_items"] > 2 * sm      # every non-empty word gets an item
    assert part["largest_item_blocks"] > 2 * BWD4_MAX_WARPS        # fat CTAs with partial last rounds
    assert part["fine_items"] > part["fwd_items"]                  # the staged E-step has a finer list
    init = tiled(engine.default_init(4, 256), c.W)
    t0 = time.time()
    got = gpu_em(c, c.shuffled(), init, "n4_left_to_right")
    t1 = time.time()
    want = oracle_em(c, got["raw"])
    print(f"N = 4 bidiagonal: GPU {t1 - t0:.1f} s, oracle {time.time() - t1:.1f} s")
    return c, got, want


def test_n4_exact_items_bidiagonal_match_oracle(n4):
    """(a) N = 4, M = 256, default (bidiagonal) initial models, shuffled input, plain create: the exact-items
    backward list, more words than 2 x sm items, the separate forward list."""
    c, got, want = n4
    check_against_oracle("N = 4 bidiagonal", c, got, want)


def test_n4_largest_remainder_leftovers_match_oracle():
    """(a') The exact-items regime with fewer non-empty words than 2 x sm items: every word gets its floor share of the
    items and the largest-remainder step hands out the rest, so that mid-sized words get several items of uneven
    length.  (With more words than items, as in (a), the floor shares alone exceed the target.)"""
    from hmm_training_b200 import engine
    sm = _sm_count()
    c = corpus_for(4, 256, 43, min_blocks=MARGIN * 2 * sm * BWD4_MAX_WARPS * 2, n_tiny=10, n_mid=60)
    part = n4_items(c.counts, sm)
    print(f"N = 4 corpus with leftovers: W = {c.W}, {c.R} sequences, partition {part}")
    assert part["exact_items"] and (c.counts > 0).sum() < 2 * sm
    assert part["bwd_items"] == 2 * sm and part["leftover_items"] > 0 and part["most_items_of_another_word"] >= 3
    got = gpu_em(c, c.shuffled(6), tiled(engine.default_init(4, 256), c.W), "n4_left_to_right")
    check_against_oracle("N = 4 largest remainder", c, got, oracle_em(c, got["raw"]))


def test_n4_dense_transitions_match_oracle(n4):
    """(b) The same corpus with a dense random A: 12-warp backward CTAs, so the rounds of every item differ."""
    c = n4[0]
    rng = np.random.default_rng(5)
    pi0, _, B0 = tiled(O.default_init(4, 256), c.W)
    A0 = rng.dirichlet(np.ones(4), size=(c.W, 4))
    got = gpu_em(c, c.shuffled(2), (pi0, A0, B0), "n4_dense")
    t1 = time.time()
    want = oracle_em(c, got["raw"])
    print(f"N = 4 dense: oracle {time.time() - t1:.1f} s")
    check_against_oracle("N = 4 dense", c, got, want)


def test_n4_pipelined_create_matches_plain_and_oracle(n4):
    """(c) The same corpus pinned, sorted and 8-byte codewords (96 MB: several upload chunks, so several stages on
    the alternating side streams) through the pipelined create: its first E-step runs in stages from the finer work
    list and k_bw_reduce sums that E-step's partials over the finer list's word ranges.  It must equal the plain
    create of (a) to rounding (the partials are grouped differently) and the oracle at the contract's tolerance."""
    from hmm_training_b200 import engine
    c, plain, want = n4
    init = tiled(engine.default_init(4, 256), c.W)
    assert c.lens.sum() * 8 >= 2 << 24  # at least two 16 MB upload chunks
    got = gpu_em(c, c.sorted(), init, "n4_left_to_right", pipelined=True, obs_dtype=np.uint64)
    stages = min(8, int(c.lens.sum()) * 8 >> 24)  # one stage per 16 MB upload chunk, at most 8
    print(f"pipelined create: {stages} stages, forward launches {got['fwd_launches']} (plain create {plain['fwd_launches']})")
    assert plain["fwd_launches"] == 3 and got["fwd_launches"] == stages + 2  # the first E-step ran in stages
    check_same("pipelined vs plain create", got, plain, rtol=1e-12)
    # the oracle ran from (a)'s raw parameters, which the line above holds to 1e-12 of these
    check_against_oracle("N = 4 pipelined create", c, got, want)


# ---------------------------------------------------------------------------------------------- N = 5
def test_n5_generic_groups_span_words_match_oracle():
    """(d) N = 5: the lanes-per-state kernels give every lane group `per_group` consecutive sequences of the
    word-sorted order, so with more sequences than groups a group runs across word boundaries."""
    sm = _sm_count()
    groups = sm * 16 * BW_WARPS * (32 // 8)  # grid cap x warps x groups per warp (8 lanes per sequence)
    c = corpus_for(5, 64, 51, min_seqs=MARGIN * 2 * groups)
    per_group = -(-c.R // groups)
    print(f"N = 5 corpus: W = {c.W}, {c.R} sequences, {groups} lane groups, {per_group} sequences per group")
    assert c.R >= MARGIN * 2 * groups and per_group >= 3
    rng = np.random.default_rng(6)
    pi0 = rng.dirichlet(np.ones(5), size=c.W)
    A0 = rng.dirichlet(np.ones(5), size=(c.W, 5))
    B0 = rng.dirichlet(np.ones(64), size=(c.W, 5))
    got = gpu_em(c, c.shuffled(3), (pi0, A0, B0), "generic")
    check_against_oracle("N = 5 generic", c, got, oracle_em(c, got["raw"]))


# ---------------------------------------------------------------------------------------------- left-to-right
LTR_CASES = [(16, 1024, 61), (8, 200, 81)]
_ltr_cache = {}


def ltr_corpus(N, M, seed):
    if (N, M) not in _ltr_cache:
        sm = _sm_count()
        c = corpus_for(N, M, seed, min_blocks=MARGIN * 4 * sm * LTR_WARPS)
        bpc, rounds = ltr_rounds(c.nblk, sm)
        print(f"N = {N} corpus: W = {c.W}, {c.R} sequences, {len(c.obs)} frames, {c.nblk} blocks, "
              f"{bpc} blocks per work item = {rounds} serpentine rounds")
        assert c.nblk >= MARGIN * 4 * sm * LTR_WARPS and rounds >= 2
        _ltr_cache[(N, M)] = c
    return _ltr_cache[(N, M)]


@pytest.mark.parametrize("N,M,seed", LTR_CASES)
def test_left_to_right_serpentine_rounds_match_oracle(N, M, seed):
    """(e) Left-to-right N = 16 / 8 with enough blocks for at least two serpentine rounds per CTA, on ragged,
    length-sorted blocks (neighbouring blocks of a round have very different tmax)."""
    from hmm_training_b200 import engine
    c = ltr_corpus(N, M, seed)
    got = gpu_em(c, c.shuffled(4), tiled(engine.default_init(N, M), c.W), "left_to_right")
    t1 = time.time()
    want = oracle_em(c, got["raw"])
    print(f"N = {N}: oracle {time.time() - t1:.1f} s")
    check_against_oracle(f"N = {N} left-to-right", c, got, want)


def test_overlapped_backward_on_two_virtual_ranks():
    """The left-to-right backward pass in word groups with the all-reduce hook per group (hmmb_bw_set_overlap), on
    one device: each of two virtual ranks runs its shard with a hook that captures every slice it is handed (keyed by
    the slice's offset from the first one: one per word group, then the LL statistics, then the (0, 0) join); rank
    0 then runs again with a hook that writes the ranks' sum into each slice.  Overlapped and plain reduction must
    give the same statistic bit for bit and the same parameters to rounding (the accumulators take fp64 atomics, so
    two runs of the same E-step differ in the last bits), and both must equal one rank over the whole corpus — at the
    tolerances of test_properties.py::test_virtual_ranks_on_one_device_equal_single_rank: pi of the giant word, a sum
    of 150 000 gamma_0 terms of ~0.002 taken in another order, moves by 2e-12 relative (5e-15 absolute)."""
    from hmm_training_b200 import dist, engine
    N, M, seed = LTR_CASES[0]
    c = ltr_corpus(N, M, seed)
    init = tiled(engine.default_init(N, M), c.W)
    order = c.shuffled(5)
    obs, off, wos = c.packed(order)
    rt = ctypes.CDLL("libcudart.so.12")
    rt.cudaMemcpy.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int]

    def one_iteration(rows, rank=0, hook=None, groups=1):
        o, f, w = c.packed(order[rows])
        with engine.BaumWelch(o, f, w, c.W, N, M) as bw:
            bw.set_params(*init)
            assert bw.kernel_family() == "left_to_right"
            if hook is not None:
                bw.set_dist(rank, 2, hook)
                if groups > 1:
                    bw.set_overlap(groups)
            bw.iterate(1, -1.0, 1)
            return bw.params() + bw.history(1)

    want = one_iteration(np.arange(c.R))
    shards = [dist.shard_sequences_round_robin(wos, r, 2) for r in range(2)]
    results, calls = {}, {}
    for groups in (1, 3):
        captured = [{}, {}]

        def capture_into(store):
            first = []

            def hook(ptr, n):
                if n == 0:
                    return  # join
                if not first:
                    first.append(ptr)
                buf = np.empty(n)
                assert rt.cudaDeviceSynchronize() == 0
                assert rt.cudaMemcpy(buf.ctypes.data, ptr, n * 8, 2) == 0
                key = (ptr - first[0]) // 8
                assert key not in store
                store[key] = buf
            return hook

        for r in range(2):
            one_iteration(shards[r], r, capture_into(captured[r]), groups)
        assert captured[0].keys() == captured[1].keys()
        total = {k: captured[0][k] + captured[1][k] for k in captured[0]}
        calls[groups] = sorted(total)
        first = []

        def inject(ptr, n):
            if n == 0:
                return
            if not first:
                first.append(ptr)
            key = (ptr - first[0]) // 8
            assert key in total and len(total[key]) == n
            assert rt.cudaDeviceSynchronize() == 0
            assert rt.cudaMemcpy(ptr, total[key].ctypes.data, n * 8, 1) == 0

        results[groups] = one_iteration(shards[0], 0, inject, groups)
    print(f"hook slices (offsets in doubles): plain {calls[1]}, overlapped {calls[3]}")
    assert len(calls[1]) == 1 and len(calls[3]) == 3 + 1  # three word groups + the LL statistics
    plain, over = results[1], results[3]
    assert np.array_equal(over[3], plain[3]) and np.array_equal(over[4], plain[4])  # statistic, iteration counts
    for x, y, z, name in zip(over, plain, want, ("pi", "A", "B", "statistic")):
        assert_close(x, y, f"overlapped vs plain: {name}", rtol=1e-12, atol=1e-13)
        assert_close(x, z, f"two virtual ranks vs one rank: {name}", rtol=1e-12, atol=1e-13)


# ---------------------------------------------------------------------------------------------- scoring
SCORE_U = 165_001  # not a multiple of 32


def score_case(N, M, W, bidiag, seed):
    rng = np.random.default_rng(seed)
    lens = _heavy_tailed_lengths(rng, SCORE_U)
    shifts = rng.integers(0, W, size=SCORE_U)
    obs = np.empty(int(lens.sum()), np.int64)
    start = np.concatenate([[0], np.cumsum(lens)[:-1]])
    for w in range(W):
        u = np.flatnonzero(shifts == w)
        cw = _ltr_codewords(rng, lens[u], N, M, (7 * w) % M)
        idx = np.repeat(start[u], lens[u]) + (np.arange(int(lens[u].sum())) - np.repeat(np.concatenate([[0], np.cumsum(lens[u])[:-1]]), lens[u]))
        obs[idx] = cw
    pi = rng.dirichlet(np.ones(N), size=W)
    B = rng.dirichlet(np.ones(M) * 0.3, size=(W, N))
    if bidiag:
        A = np.zeros((W, N, N))
        stay = rng.uniform(0.4, 0.9, size=(W, N))
        for i in range(N):
            A[:, i, i] = stay[:, i] if i + 1 < N else 1.0
            if i + 1 < N:
                A[:, i, i + 1] = 1.0 - stay[:, i]
    else:
        A = rng.dirichlet(np.ones(N), size=(W, N))
    return obs.astype(np.uint8 if M <= 256 else np.uint16), lens, start, (pi, A, B)


def score_sample(lens, rng):
    """Rows to check: the first and last 64, both ends of every 1000th block of the length-sorted order (and of
    the last block), and 2000 random ones."""
    U = len(lens)
    srt = np.argsort(-lens, kind="stable")
    nblk = -(-U // 32)
    ends = [b * 32 for b in range(0, nblk, 1000)] + [min(U, b * 32 + 32) - 1 for b in range(0, nblk, 1000)]
    ends += [(nblk - 1) * 32, U - 1]
    rows = np.concatenate([np.arange(64), np.arange(U - 64, U), srt[ends], rng.choice(U, 2000, replace=False)])
    return np.unique(rows)


@pytest.mark.parametrize("N,M,W,bidiag,kernel", [(4, 256, 7, True, "k_score4r"), (4, 300, 5, False, "k_score4"),
                                                 (16, 1024, 4, True, "k_scoreL"), (5, 64, 4, False, "k_scoreG")])
def test_scoring_at_scale_matches_oracle(N, M, W, bidiag, kernel):
    """165 001 ragged utterances in random order against W models, each scorer family: a sample of rows against
    the oracle's forward pass, and the argmax on it."""
    from hmm_training_b200 import engine
    sm = _sm_count()
    nblk = -(-SCORE_U // 32)
    if kernel == "k_scoreL":
        bpc, rounds = ltr_rounds(nblk, sm)
        assert nblk >= MARGIN * 4 * sm * LTR_WARPS and rounds >= 2, (nblk, rounds)
    if kernel == "k_scoreG":
        assert SCORE_U >= MARGIN * 2 * sm * 16 * BW_WARPS * (32 // 8)  # several utterances per lane group
    if kernel == "k_score4r":
        bpc = -(-max(8, -(-nblk * W // (sm * 12))) // 8) * 8
        assert bpc > 8, bpc  # several blocks per CTA
    obs, lens, start, (pi, A, B) = score_case(N, M, W, bidiag, seed=N * 31 + M)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    ll, arg = engine.score(obs, off, N, M, pi, A, B)
    rows = score_sample(lens, np.random.default_rng(M))
    ref = O.score_batch([obs[start[u]:start[u] + lens[u]] for u in rows], [(A[w], B[w], pi[w]) for w in range(W)])
    print(f"{kernel}: {nblk} blocks, {len(rows)} rows checked")
    assert np.isfinite(ref).all()
    assert_close(ll[rows], ref, f"{kernel}: sampled rows")
    assert np.array_equal(arg[rows], O.argmax_first(ref))
    assert np.array_equal(arg, O.argmax_first(ll))


def test_pipelined_scorer_ragged_length_descending(monkeypatch):
    """Pinned, length-descending ragged utterances go through the pipelined scorer (stages repacked and scored as
    they land, each stage's rows of a pinned result matrix copied back on their own): it must equal the unpipelined
    scorer bit for bit with a pageable and with a pinned result matrix.  The same utterances pinned but NOT sorted
    fall back to the unpipelined path and must give the same rows in the caller's order."""
    from hmm_training_b200 import engine
    N, M, W = 4, 256, 7
    obs, lens, start, (pi, A, B) = score_case(N, M, W, True, seed=3)
    srt = np.argsort(-lens, kind="stable")
    L = lens[srt]
    off = np.concatenate([[0], np.cumsum(L)]).astype(np.int64)
    sorted_obs = np.concatenate([obs[start[u]:start[u] + lens[u]] for u in srt]).astype(np.uint64)
    assert sorted_obs.nbytes >= 2 << 24  # at least two 16 MB upload chunks: several stages
    pinned, h1 = _pinned_copy(sorted_obs)
    out, h2 = _pinned_copy(np.zeros((SCORE_U, W)))
    unsorted, h3 = _pinned_copy(obs.astype(np.uint64))
    try:
        monkeypatch.setenv("HMMB_SCORE_NO_PIPELINE", "1")
        with launches_of("score") as plain:
            ll0, arg0 = engine.score(pinned, off, N, M, pi, A, B)
        monkeypatch.delenv("HMMB_SCORE_NO_PIPELINE")
        with launches_of("score") as staged:
            ll1, arg1 = engine.score(pinned, off, N, M, pi, A, B)
        assert plain.n == 1 and staged.n >= 2, (plain.n, staged.n)  # one scoring launch per stage
        assert np.array_equal(ll1, ll0) and np.array_equal(arg1, arg0), "pipelined (pageable result) vs unpipelined"
        ll2, arg2 = engine.score(pinned, off, N, M, pi, A, B, out_ll=out)
        assert np.array_equal(ll2, ll0) and np.array_equal(arg2, arg0), "pipelined (pinned result) vs unpipelined"
        off_u = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        with launches_of("score") as fallback:
            ll3, arg3 = engine.score(unsorted, off_u, N, M, pi, A, B)
        assert fallback.n == 1  # unsorted input: the unpipelined path
        want = np.empty_like(ll0)
        want[srt] = ll0
        assert np.array_equal(ll3, want), "pinned unsorted input: rows not in the caller's order"
        wa = np.empty_like(arg0)
        wa[srt] = arg0
        assert np.array_equal(arg3, wa)
    finally:
        for h in (h1, h2, h3):
            _host_free(h)
    rows = score_sample(L, np.random.default_rng(9))
    ref = O.score_batch([obs[start[u]:start[u] + lens[u]] for u in srt[rows]], [(A[w], B[w], pi[w]) for w in range(W)])
    assert_close(ll0[rows], ref, "pipelined scorer: sampled rows")

"""Drop-in for the reference's HMM/hmm_testing.py recognition path:

    calculate_log_likelihood   HMM/hmm_testing.py:49-104
    test_hmm                   HMM/hmm_testing.py:107-163
    create_confusion_matrix    HMM/hmm_testing.py:166-218
plus ``score_all`` (every utterance against every model in one launch), ``viterbi_align`` (the most
likely state path of every utterance under a chosen model; an extension, the reference has no Viterbi) and
``recognize_connected`` (the best word sequence of every utterance; an extension, the reference recognises one word
per recording).
"""
from __future__ import annotations

import os
from typing import Dict, List, Sequence, Tuple

import numpy as np

from . import _lib, engine
from .codevector_classes import DataStorage, RawDataMFCC
from .hmm_classes import HMMTrained
from .hmm_training import get_observations


def _stack_models(all_hmm: Sequence[HMMTrained]):
    N, M = int(all_hmm[0].states), int(all_hmm[0].symbols)
    pi = np.stack([np.asarray(h.Pi, float) for h in all_hmm])
    A = np.stack([np.asarray(h.A, float) for h in all_hmm])
    B = np.stack([np.asarray(h.B, float) for h in all_hmm])
    return N, M, pi, A, B


def score_all(observations: Sequence[np.ndarray], all_hmm: Sequence[HMMTrained]):
    """[U, W] log-likelihood matrix and the index of the winning model per utterance
    (-1 = "unknown": every score is -inf, hmm_testing.py:161).  The reference scores every (recording, model)
    pair on its own (:139-153), so models of different shapes may sit in one list: they are grouped by
    (states, symbols), each group is one launch, and the columns go back to list order before the argmax."""
    seqs = [np.asarray(o) for o in observations]
    if any(len(o) == 0 for o in seqs):
        raise IndexError("index 0 is out of bounds for axis 0 with size 0")  # hmm_testing.py:75
    groups: Dict[Tuple[int, int], List[int]] = {}
    for w, h in enumerate(all_hmm):
        groups.setdefault((int(h.states), int(h.symbols)), []).append(w)
    if len(groups) == 1:
        N, M, pi, A, B = _stack_models(all_hmm)
        obs, offsets = _lib.pack_sequences(seqs, M)
        return engine.score(obs, offsets, N, M, pi, A, B)
    ll = np.empty((len(seqs), len(all_hmm)))
    for (N, M), cols in groups.items():
        _, _, pi, A, B = _stack_models([all_hmm[w] for w in cols])
        obs, offsets = _lib.pack_sequences(seqs, M)  # (a codeword >= this group's M raises IndexError, as B[:, o] would)
        ll[:, cols], _ = engine.score(obs, offsets, N, M, pi, A, B)
    # first model with the strictly largest score, from -inf (:143-153)
    arg = np.full(len(seqs), -1, dtype=np.int32)
    best = np.full(len(seqs), -np.inf)
    for w in range(len(all_hmm)):
        better = ll[:, w] > best
        arg[better] = w
        best[better] = ll[better, w]
    return ll, arg


def viterbi_align(observations: Sequence[np.ndarray], all_hmm: Sequence[HMMTrained], model_index):
    """Viterbi alignment of every utterance against the model all_hmm[model_index[u]] (for example score_all's
    argmax, or the index of the utterance's known word for forced alignment).

    Returns (scores float64 [U], paths: one int8 array of states per utterance): the log-probability of the best
    state path and that path.  Index -1 ("unknown") and utterances impossible under their model give -inf and a
    path of -1.  Models of different (states, symbols) are grouped as in score_all, one launch per group."""
    seqs = [np.asarray(o) for o in observations]
    idx = np.asarray(model_index, dtype=np.int64).reshape(-1)
    if len(idx) != len(seqs):
        raise ValueError(f"model_index has {len(idx)} entries for {len(seqs)} utterances")
    if any(len(o) == 0 for o in seqs):
        raise IndexError("index 0 is out of bounds for axis 0 with size 0")  # as score_all (hmm_testing.py:75)
    if len(idx) and (int(idx.min()) < -1 or int(idx.max()) >= len(all_hmm)):
        raise IndexError(f"model index outside [-1, {len(all_hmm)})")
    scores = np.full(len(seqs), -np.inf)
    paths = [np.full(len(o), -1, dtype=np.int8) for o in seqs]
    groups: Dict[Tuple[int, int], List[int]] = {}
    for w, h in enumerate(all_hmm):
        groups.setdefault((int(h.states), int(h.symbols)), []).append(w)
    for (N, M), cols in groups.items():
        local = np.full(len(all_hmm) + 1, -1, dtype=np.int64)  # (slot -1 stays -1: "unknown")
        local[cols] = np.arange(len(cols))
        utts = np.nonzero(local[idx] >= 0)[0]
        if len(utts) == 0:
            continue
        _, _, pi, A, B = _stack_models([all_hmm[w] for w in cols])
        obs, offsets = _lib.pack_sequences([seqs[u] for u in utts], M)
        sc, path = engine.viterbi(obs, offsets, local[idx[utts]], N, M, pi, A, B)
        scores[utts] = sc
        for k, u in enumerate(utts):
            paths[u] = path[offsets[k]:offsets[k + 1]].copy()
    return scores, paths


def recognize_connected(observations: Sequence[np.ndarray], all_hmm: Sequence[HMMTrained], log_penalty: float = 0.0):
    """Connected-word recognition: the best sequence of words from all_hmm (a free word loop, any word after any
    other) for every utterance, in one decode on the GPU (engine.decode_words).  log_penalty (natural log) is added
    once per recognised word: negative values favour fewer, longer words.

    Returns (scores float64 [U], one list per utterance of (word, first_frame, last_frame) with the word named by
    HMMTrained.word).  An utterance that no word sequence can produce gets -inf and an empty list.  One decode needs
    one model shape, so models of different (states, symbols) raise ValueError."""
    seqs = [np.asarray(o) for o in observations]
    if any(len(o) == 0 for o in seqs):
        raise IndexError("index 0 is out of bounds for axis 0 with size 0")  # as score_all (hmm_testing.py:75)
    if len({(int(h.states), int(h.symbols)) for h in all_hmm}) > 1:
        raise ValueError("connected-word recognition needs models of one (states, symbols) shape")
    if not all_hmm:
        raise ValueError("no word models")
    N, M, pi, A, B = _stack_models(all_hmm)
    obs, offsets = _lib.pack_sequences(seqs, M)
    scores, seg_off, seg_word, seg_start = engine.decode_words(obs, offsets, N, M, pi, A, B, log_penalty)
    words = []
    for u, o in enumerate(seqs):
        a, b = int(seg_off[u]), int(seg_off[u + 1])
        ends = list(seg_start[a + 1:b] - 1) + [len(o) - 1]
        words.append([(all_hmm[int(seg_word[k])].word, int(seg_start[k]), int(ends[k - a])) for k in range(a, b)])
    return scores, words


def calculate_log_likelihood(recording_observations: np.ndarray, hmm: HMMTrained) -> float:
    """log P(O | lambda) of one recording by the forward algorithm (hmm_testing.py:49-104)."""
    ll, _ = score_all([recording_observations], [hmm])
    return float(ll[0, 0])


def test_hmm(all_hmm: List[HMMTrained], test_recordings_dict: Dict[str, List[List[RawDataMFCC]]],
             base_dir="../Data", show_progress=False) -> Tuple[List[str], List[str]]:
    """hmm_testing.py:107-163: loads <base_dir>/CodeVector/codevector.json itself, encodes every
    test recording, scores it against every model, predicts the first model with the
    strictly largest log-likelihood ("unknown" if all are -inf)."""
    print("Starting HMM testing...")
    storage = DataStorage()
    centroids = storage.load_centroids(os.path.join(base_dir, "CodeVector", "codevector.json"))
    print("Phase 1: Converting recordings to observations...")
    words = list(test_recordings_dict.keys())
    for word in words:
        print(f"  Converting {len(test_recordings_dict[word])} recordings for word: '{word}'")
    all_recs = [rec for w in words for rec in test_recordings_dict[w]]
    all_obs = get_observations(all_recs, centroids)
    print("Phase 2: Testing all recording-HMM combinations...")
    true_labels: List[str] = []
    predicted_labels: List[str] = []
    if not all_obs:
        return true_labels, predicted_labels
    ll, arg = score_all(all_obs, all_hmm)
    pos = 0
    for word in words:
        n = len(test_recordings_dict[word])
        print(f"Testing {n} recordings for word: '{word}'")
        for r in range(n):
            k = int(arg[pos])
            predicted = all_hmm[k].word if k >= 0 else None
            if show_progress:
                likelihoods = {h.word: float(ll[pos, i]) for i, h in enumerate(all_hmm)}
                print(f"  Recording {r + 1} likelihoods: {likelihoods}")
                print(f"  True: '{word}' -> Predicted: '{predicted}'")
            true_labels.append(word)
            predicted_labels.append(predicted if predicted else "unknown")
            pos += 1
    return true_labels, predicted_labels


def confusion_counts(true_labels: Sequence[str], predicted_labels: Sequence[str]):
    """(cm [L,L] int64, labels): rows = true word, columns = predicted word, labels sorted as in
    the reference (hmm_testing.py:182-185; same matrix as sklearn's confusion_matrix)."""
    labels = sorted(set(true_labels) | set(predicted_labels))
    index = {w: i for i, w in enumerate(labels)}
    L = len(labels)
    t = np.fromiter((index[w] for w in true_labels), dtype=np.int64, count=len(true_labels))
    p = np.fromiter((index[w] for w in predicted_labels), dtype=np.int64, count=len(predicted_labels))
    cm = np.bincount(t * L + p, minlength=L * L).reshape(L, L) if L else np.zeros((0, 0), np.int64)
    return cm.astype(np.int64), labels


def classification_report_text(cm: np.ndarray, labels: Sequence[str], digits: int = 2) -> str:
    """Per-word precision / recall / f1 / support table in the layout of
    sklearn.metrics.classification_report (what the reference prints, hmm_testing.py:214),
    computed from the confusion counts; 0/0 ratios are reported as 0 like sklearn does."""
    cm = np.asarray(cm, dtype=np.float64)
    tp = np.diag(cm)
    support = cm.sum(axis=1)
    pred = cm.sum(axis=0)
    with np.errstate(divide="ignore", invalid="ignore"):
        prec = np.where(pred > 0, tp / pred, 0.0)
        rec = np.where(support > 0, tp / support, 0.0)
        f1 = np.where(prec + rec > 0, 2 * prec * rec / (prec + rec), 0.0)
    total = support.sum()
    names = [str(x) for x in labels]
    width = max([len(n) for n in names] + [len("weighted avg"), digits])
    head = "{:>{w}s} ".format("", w=width) + "".join(" {:>9}".format(h) for h in ("precision", "recall", "f1-score", "support"))
    lines = [head, ""]
    row = "{:>{w}s} " + " {:>9.{d}f}" * 3 + " {:>9}"
    for n, p_, r_, f_, s_ in zip(names, prec, rec, f1, support):
        lines.append(row.format(n, p_, r_, f_, int(s_), w=width, d=digits))
    lines.append("")
    acc = tp.sum() / total if total else 0.0
    lines.append("{:>{w}s} ".format("accuracy", w=width) + " {:>9}".format("") * 2 + " {:>9.{d}f}".format(acc, d=digits) +
                 " {:>9}".format(int(total)))
    wavg = lambda x: float((x * support).sum() / total) if total else 0.0
    lines.append(row.format("macro avg", prec.mean() if len(prec) else 0.0, rec.mean() if len(rec) else 0.0,
                            f1.mean() if len(f1) else 0.0, int(total), w=width, d=digits))
    lines.append(row.format("weighted avg", wavg(prec), wavg(rec), wavg(f1), int(total), w=width, d=digits))
    return "\n".join(lines) + "\n"


def create_confusion_matrix(true_labels: List[str], predicted_labels: List[str], base_dir="../Data"):
    """hmm_testing.py:166-218: confusion matrix over the sorted label set, accuracy, the
    classification report, and the matrix saved under <base_dir>/Plots.  The reference draws a
    seaborn heat map (confusion_matrix.png); that is done when matplotlib + seaborn are
    importable, and the counts are always written as confusion_matrix.csv.  Returns (cm, labels)."""
    plots_dir = os.path.join(base_dir, "Plots")
    os.makedirs(plots_dir, exist_ok=True)
    cm, unique_labels = confusion_counts(true_labels, predicted_labels)
    accuracy = (cm.diagonal().sum() / cm.sum()) * 100 if cm.sum() else float("nan")
    csv_path = os.path.join(plots_dir, "confusion_matrix.csv")
    with open(csv_path, "w") as f:
        f.write("true\\predicted," + ",".join(unique_labels) + "\n")
        for w, row in zip(unique_labels, cm):
            f.write(w + "," + ",".join(str(int(x)) for x in row) + "\n")
    plot_path = csv_path
    try:
        import matplotlib
        matplotlib.use("Agg")
        import matplotlib.pyplot as plt
        import seaborn as sns
        plt.figure(figsize=(10, 8))
        sns.heatmap(cm, annot=True, fmt="d", cmap="Blues", xticklabels=unique_labels, yticklabels=unique_labels,
                    cbar_kws={"label": "Number of Recordings"})
        plt.title(f"HMM Classification Confusion Matrix\nAccuracy: {accuracy:.2f}%", fontsize=14, fontweight="bold")
        plt.xlabel("Predicted Word", fontsize=12)
        plt.ylabel("True Word", fontsize=12)
        plt.xticks(rotation=45, ha="right")
        plt.yticks(rotation=0)
        plt.tight_layout()
        plot_path = os.path.join(plots_dir, "confusion_matrix.png")
        plt.savefig(plot_path, dpi=300, bbox_inches="tight")
        plt.close()
    except ImportError:
        pass
    print("\nClassification Report:")
    print(classification_report_text(cm, unique_labels))
    print(f"\nConfusion matrix saved to: {plot_path}")
    print(f"Overall Accuracy: {accuracy:.2f}%")
    return cm, unique_labels

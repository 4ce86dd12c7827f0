"""Viterbi decoding at BASELINE config 3's shape (1 M utterances x 200 frames, N = 4, M = 256, 10 models: 200 M
frames) and config 4's (N = 16, M = 1024, 1 M utterances x 100 frames: 100 M frames, 24 models), left-to-right
models, pinned host codewords.

Reports, warm and from CUDA events: the `viterbi` and `viterbi_backtrace` phases, the score-only `viterbi` phase,
the `score` phase of hmmb_score on the same corpus against the same models, the HBM bytes each Viterbi kernel needs
per frame and the share of the HBM roofline they reach, and the end-to-end call time.  Every input is larger than
the 126 MB L2.  The card's name and power limit are read in the same run.

    python scripts/viterbi_probe.py [--reps 3] [--out viterbi_probe.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from hmm_training_b200 import _lib, engine, synthetic  # noqa: E402

HBM_BPS = 7.7e12  # HGX B200 data sheet, one GPU


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:  # pragma: no cover
        return f"unknown ({e})"


def phases(names):
    return {k: _lib.phase_ms(k)[0] for k in names}


def run(cfg, reps):
    N, M, W, U, T = cfg["N"], cfg["M"], cfg["W"], cfg["U"], cfg["T"]
    obs, offsets, word = synthetic.fixed_length_codewords(7, W, U // W, T, N, M)
    pi, A, _ = engine.default_init(N, M)
    rng = np.random.default_rng(3)
    Bm = rng.dirichlet(np.ones(M) * 0.3, size=(W, N))
    pim, Am = np.tile(pi, (W, 1)), np.tile(A, (W, 1, 1))
    pinned = torch.empty(obs.shape, dtype=torch.uint8 if obs.dtype == np.uint8 else torch.int16, pin_memory=True).numpy()
    pinned = pinned.view(obs.dtype)
    pinned[:] = obs
    frames = int(offsets[-1])
    lib = _lib.load()
    # warm-up of every kernel at a small size
    small = offsets[: 1001]
    engine.viterbi(pinned[: small[-1]], small, word[:1000], N, M, pim, Am, Bm)
    engine.viterbi(pinned[: small[-1]], small, word[:1000], N, M, pim, Am, Bm, want_path=False)
    engine.score(pinned[: small[-1]], small, N, M, pim, Am, Bm, want_ll=False)
    out = {"config": cfg, "frames": frames, "path": [], "score_only": [], "hmmb_score": []}
    for _ in range(reps):
        for key, fn in (("path", lambda: engine.viterbi(pinned, offsets, word, N, M, pim, Am, Bm)),
                        ("score_only", lambda: engine.viterbi(pinned, offsets, word, N, M, pim, Am, Bm, want_path=False)),
                        ("hmmb_score", lambda: engine.score(pinned, offsets, N, M, pim, Am, Bm, want_ll=False))):
            _lib.check(lib.hmmb_set_profiling(1))
            _lib.check(lib.hmmb_phase_reset())
            t0 = time.perf_counter()
            res = fn()
            dt = time.perf_counter() - t0
            ph = phases(("prepare", "viterbi_load", "viterbi", "viterbi_backtrace", "score"))
            _lib.check(lib.hmmb_set_profiling(0))
            out[key].append({"call_ms": dt * 1e3, **ph})
            if key == "path":
                score, path = res
                out["n_impossible"] = int(np.isneginf(score).sum())
    # HBM bytes per frame (blocked layouts, fixed lengths: no padding): packed u16 codeword entries in, one packed
    # backpointer row out (1 B at N = 4, 2 B at N = 16); the backtrace reads that row and writes the int8 path
    row = 1 if N <= 8 else 2
    bytes_fwd, bytes_bt = 2 + row, row + 1
    best = lambda k, ph: min(r[ph] for r in out[k])
    vit, bt = best("path", "viterbi"), best("path", "viterbi_backtrace")
    out["bytes_per_frame"] = {"viterbi": bytes_fwd, "viterbi_score_only": 2, "viterbi_backtrace": bytes_bt}
    out["summary"] = {
        "viterbi_ms": vit, "viterbi_backtrace_ms": bt, "viterbi_score_only_ms": best("score_only", "viterbi"),
        "hmmb_score_ms": best("hmmb_score", "score"), "score_models": W,
        "viterbi_hbm_share": frames * bytes_fwd / HBM_BPS / (vit * 1e-3),
        "viterbi_backtrace_hbm_share": frames * bytes_bt / HBM_BPS / (bt * 1e-3),
        "viterbi_Gframes_per_s": frames / (vit * 1e-3) / 1e9,
        "end_to_end_ms": min(r["call_ms"] for r in out["path"]),
        "end_to_end_score_only_ms": min(r["call_ms"] for r in out["score_only"]),
    }
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write every run as JSON here")
    a = ap.parse_args()
    _lib.init(0)
    res = {"card": card(), "runs": []}
    print("card:", res["card"], flush=True)
    for cfg in ({"name": "config3", "N": 4, "M": 256, "W": 10, "U": 1_000_000, "T": 200},
                {"name": "config4", "N": 16, "M": 1024, "W": 24, "U": 1_000_008, "T": 100}):
        r = run(cfg, a.reps)
        res["runs"].append(r)
        print(cfg["name"], json.dumps(r["summary"]), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

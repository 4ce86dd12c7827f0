"""Connected-word decoding (hmmb_decode_words) at three shapes, left-to-right models, pinned host codewords:

  1. the reference's shape: W = 10 words, N = 4, M = 256, strings of 1-6 words of 100 frames (~70 M frames);
  2. W = 32, N = 16, M = 1024 (a 4 MB log-emission table);
  3. W = 200, N = 16, M = 256 (3200 states per utterance).

Reports, warm and from CUDA events: the `words` phase with and without segments, the same with the generic kernel
forced (HMMB_FORCE_GENERIC=1, which must give the same words), the `words_backtrace` phase, the
end-to-end call into host arrays, frames/s and state updates/s (frames x W x N / time), and the `score` phase of
hmmb_score on the same corpus against the same models.  Every codeword stream is larger than the 126 MB L2 except
shape 3's (sized to keep the run short).  The card's name and power limit are read in the same run.

    python scripts/words_probe.py [--reps 3] [--scale 1.0] [--out words_probe.json]
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


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:  # pragma: no cover
        return f"unknown ({e})"


def corpus(W, N, M, frames, T=100, seed=7):
    """Strings of 1-6 isolated words of T frames each, about `frames` frames in all."""
    pool, _, _ = synthetic.fixed_length_codewords(seed, W, 200, T, N, M)
    pool = pool.reshape(W * 200, T)
    rng = np.random.default_rng(seed)
    K = rng.integers(1, 7, size=max(1, int(frames / (3.5 * T))))
    rows = rng.integers(0, len(pool), size=int(K.sum()))
    obs = pool[rows].reshape(-1)
    offsets = np.zeros(len(K) + 1, np.int64)
    np.cumsum(K * T, out=offsets[1:])
    pinned = torch.empty(obs.shape, dtype=torch.uint8 if obs.dtype == np.uint8 else torch.int16, pin_memory=True).numpy()
    pinned = pinned.view(obs.dtype)
    pinned[:] = obs
    return pinned, offsets


def run(cfg, reps, scale):
    N, M, W = cfg["N"], cfg["M"], cfg["W"]
    obs, offsets = corpus(W, N, M, cfg["frames"] * scale)
    U, frames = len(offsets) - 1, int(offsets[-1])
    pi, A, _ = engine.default_init(N, M)
    Bm = np.random.default_rng(3).dirichlet(np.ones(M) * 0.3, size=(W, N))
    pim, Am = np.tile(pi, (W, 1)), np.tile(A, (W, 1, 1))
    lib = _lib.load()
    small = offsets[: min(U, 200) + 1]
    for seg in (True, False):
        engine.decode_words(obs[: small[-1]], small, N, M, pim, Am, Bm, -20.0, want_segments=seg)
    engine.score(obs[: small[-1]], small, N, M, pim, Am, Bm, want_ll=False)
    out = {"config": cfg, "U": U, "frames": frames, "segments": [], "generic": [], "score_only": [], "hmmb_score": []}

    def generic():  # the same call with the one-CTA-per-utterance kernel forced
        os.environ["HMMB_FORCE_GENERIC"] = "1"
        try:
            return engine.decode_words(obs, offsets, N, M, pim, Am, Bm, -20.0)
        finally:
            del os.environ["HMMB_FORCE_GENERIC"]

    for _ in range(reps):
        for key, fn in (("segments", lambda: engine.decode_words(obs, offsets, N, M, pim, Am, Bm, -20.0)),
                        ("generic", generic),
                        ("score_only", lambda: engine.decode_words(obs, offsets, N, M, pim, Am, Bm, -20.0, want_segments=False)),
                        ("hmmb_score", lambda: engine.score(obs, offsets, N, M, pim, Am, Bm, want_ll=False))):
            _lib.check(lib.hmmb_set_profiling(1))
            _lib.check(lib.hmmb_phase_reset())
            t0 = time.perf_counter()
            res = fn()
            dt = time.perf_counter() - t0
            ph = {k: _lib.phase_ms(k)[0] for k in ("prepare", "words_load", "words", "words_backtrace", "score")}
            _lib.check(lib.hmmb_set_profiling(0))
            out[key].append({"call_ms": dt * 1e3, **ph})
            if key == "segments":
                out["n_impossible"] = int(np.isneginf(res[0]).sum())
                out["words_per_utterance"] = float(res[1][-1] / U)
                ref = res
            if key == "generic":  # both kernels must return the same words
                out["generic_same_segments"] = bool(all(np.array_equal(x, y) for x, y in zip(ref[1:], res[1:])))
                fin = np.isfinite(ref[0])
                out["generic_same_inf"] = bool(np.array_equal(np.isfinite(res[0]), fin))
                out["generic_max_rel_score_diff"] = float(np.max(np.abs(res[0][fin] - ref[0][fin]) / np.abs(ref[0][fin]), initial=0.0))
    best = lambda k, ph: min(r[ph] for r in out[k])
    dec = best("segments", "words")
    out["summary"] = {
        "words_ms": dec, "words_generic_ms": best("generic", "words"), "words_score_only_ms": best("score_only", "words"),
        "words_backtrace_ms": best("segments", "words_backtrace"), "hmmb_score_ms": best("hmmb_score", "score"),
        "end_to_end_ms": min(r["call_ms"] for r in out["segments"]),
        "end_to_end_score_only_ms": min(r["call_ms"] for r in out["score_only"]),
        "Gframes_per_s": frames / (dec * 1e-3) / 1e9,
        "Gstate_updates_per_s": frames * W * N / (dec * 1e-3) / 1e9,
    }
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--scale", type=float, default=1.0, help="multiplies every shape's frame count")
    ap.add_argument("--out", default=None, help="also write every run as JSON here")
    a = ap.parse_args()
    _lib.init(0)
    res = {"card": card(), "runs": []}
    print("card:", res["card"], flush=True)
    for cfg in ({"name": "reference", "N": 4, "M": 256, "W": 10, "frames": 70e6},
                {"name": "w32_n16_m1024", "N": 16, "M": 1024, "W": 32, "frames": 20e6},
                {"name": "w200_n16", "N": 16, "M": 256, "W": 200, "frames": 2e6}):
        r = run(cfg, a.reps, a.scale)
        res["runs"].append(r)
        print(cfg["name"], r["U"], r["frames"], json.dumps(r["summary"]), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

"""bench.py on the GPU: `--dump-outputs` writes what the timed iterations computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import assert_close
from hmm_training_b200 import engine, synthetic

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dump_outputs_hold_the_model_after_the_timed_steps(tmp_path):
    """After 3 warm-up + 2 timed EM iterations on config 1's seeded inputs, the dumped model, log-likelihood
    history and per-sequence log-likelihoods equal those of a 5-iteration fit of the same inputs."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "bw_c1", "--steps", "2", "--warmup", "3",
                          "--no-extras", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout)
    assert (line["steps"], line["warmup"]) == (2, 3)
    W, S, T, N, M = 10, 20, 100, 4, 256
    obs, offsets, wos = synthetic.fixed_length_codewords(1000, W, S, T, N, M)
    pi0, A0, B0 = engine.default_init(N, M)
    with engine.BaumWelch(obs, offsets, wos, W, N, M) as bw:
        bw.set_params(np.tile(pi0, (W, 1)), np.tile(A0, (W, 1, 1)), np.tile(B0, (W, 1, 1)))
        bw.iterate(5, -1.0, 5)
        pi, A, B = bw.params()
        hist, iters = bw.history(5)
        seq_ll = bw.seq_ll()
    assert np.array_equal(iters, np.full(W, 5))
    for name, want in (("pi", pi), ("A", A), ("B", B), ("ll_hist", hist), ("seq_ll", seq_ll)):
        got = np.load(tmp_path / f"{name}.npy")
        assert got.dtype == np.float64
        assert_close(got, want, name)

"""CPU-side checks of the C-ABI boundary: the library builds/loads and exports every symbol
include/hmmb200.h declares; without a GPU compute calls fail loudly (no CPU fallback)."""
import os
import re

import numpy as np
import pytest

from hmm_training_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_functions():
    src = open(os.path.join(ROOT, "include", "hmmb200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(hmmb_[a-z0-9_]+)\s*\(", src)) - {"hmmb_allreduce_fn"})


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    declared = _header_functions()
    assert len(declared) >= 25
    bound = {name for name, _, _ in _lib.SYMBOLS}
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in hmmb200.h but not exported"
        assert name in bound, f"{name} declared in hmmb200.h but not bound in _lib.SYMBOLS"
    assert lib.hmmb_version().decode().startswith("hmmb200")


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from hmm_training_b200 import engine
    with pytest.raises(_lib.HmmbError) as ei:
        engine.vq_encode(np.zeros((4, 13)), np.zeros((2, 13)))
    assert ei.value.code == _lib.ERR_CUDA
    assert "no CPU fallback" in str(ei.value)


def test_non_integer_codewords_are_rejected_before_the_library():
    """Host codewords must be integers in every entry point: the bits of a float array are not codewords (an all-zero
    float64 array would otherwise be read as codeword 0).  The check runs before any device work."""
    from hmm_training_b200 import engine
    N, M, W = 4, 8, 2
    pi, A, B = (np.tile(x, (W,) + (1,) * x.ndim) for x in engine.default_init(N, M))
    offsets = np.array([0, 3, 5], np.int64)
    for obs in (np.zeros(5), np.zeros(5, np.float32), np.zeros(5, bool)):
        with pytest.raises(TypeError):
            engine.score(obs, offsets, N, M, pi, A, B)
        with pytest.raises(TypeError):
            engine.viterbi(obs, offsets, np.zeros(2, np.int32), N, M, pi, A, B)
        with pytest.raises(TypeError):
            engine.BaumWelch(obs, offsets, np.zeros(2, np.int32), W, N, M)


def test_product_package_never_imports_oracle():
    pkg = os.path.join(ROOT, "hmm_training_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f"{f} imports the oracle"
                assert "/root/reference" not in text, f"{f} reads the reference tree"


def test_native_communicator_api_without_ranks():
    """hmmb_comm_* (the library's own NCCL plumbing, libnccl via dlopen): without a communicator the all-reduce
    hook fails loudly, the reported world size is 1, and rank 0 can obtain a 128-byte id (no GPU needed)."""
    import ctypes
    lib = _lib.load()
    assert lib.hmmb_comm_allreduce(None, 0, None) == _lib.ERR_ARG
    assert b"no communicator" in lib.hmmb_last_error()
    r, w = ctypes.c_int32(-1), ctypes.c_int32(-1)
    assert lib.hmmb_comm_rank(ctypes.byref(r), ctypes.byref(w)) == 0 and (r.value, w.value) == (0, 1)
    assert lib.hmmb_comm_unique_id(ctypes.create_string_buffer(16), 16) == _lib.ERR_ARG  # buffer too small
    buf = ctypes.create_string_buffer(128)
    rc = lib.hmmb_comm_unique_id(buf, 128)
    if rc == _lib.ERR_UNSUPPORTED:
        pytest.skip("libnccl.so.2 not present")
    assert rc == 0 and any(buf.raw)
    assert lib.hmmb_comm_destroy() == 0  # nothing to destroy


def _build_c_caller(tmp_path):
    import shutil
    import subprocess
    if not shutil.which("gcc"):
        pytest.skip("gcc not available")
    _lib.load()  # builds the library if needed
    exe = str(tmp_path / "c_caller")
    subprocess.run(["gcc", "-std=c11", "-O2", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "examples", "c_caller.c"), "-L", os.path.join(ROOT, "hmm_training_b200"),
                    "-lhmmb200", "-lm", "-o", exe], check=True)
    env = dict(os.environ, LD_LIBRARY_PATH=os.path.join(ROOT, "hmm_training_b200") + ":" + os.environ.get("LD_LIBRARY_PATH", ""))
    return exe, env


def test_plain_c_caller_compiles_against_the_header(tmp_path):
    """include/hmmb200.h is a C header (no C++ / torch types): examples/c_caller.c builds with gcc -std=c11 -Werror
    and links against the library; without a GPU it stops at hmmb_init with the no-fallback message."""
    import subprocess
    import torch
    exe, env = _build_c_caller(tmp_path)
    if torch.cuda.is_available():
        pytest.skip("GPU present: tests/test_gpu_dropin.py runs the example")
    r = subprocess.run([exe], env=env, capture_output=True, text=True)
    assert r.returncode == 1 and "no CPU fallback" in r.stderr

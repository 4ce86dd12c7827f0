#!/usr/bin/env python
"""Benchmark of the hot path on B200 (contract: see the task statement / DESIGN.md §Measurement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

Default workload = BASELINE.json config 3: 10-word discrete HMM (N=4, M=256) Baum-Welch over
100 000 synthetic sequences per word at T=200 (200 M frames per EM iteration), per GPU (weak
scaling: every rank holds its own shard of that size; the pi/A/B accumulators are combined
with one NCCL all-reduce per iteration).  One "step" = one full EM iteration (E-step forward +
backward/accumulate, reduce, all-reduce, M-step) over the whole batch.

Printed JSON (rank 0, one line): metric/value = Baum-Welch frames/s/iteration with the
codewords resident in HBM; `e2e` = the same through the public packed-array API
(engine.bw_fit -> hmmb_bw_*) from pinned HOST buffers, H2D/D2H inside the timed region;
`roofline` for the dominant kernel from CUDA events recorded around every launch on the
launching stream; `cpu_baseline` = the CPU oracle (numpy port of the reference) on a bounded
sample using all host cores; secondary blocks `vq_encode`, `lbg`, `score` for the other
BASELINE configs.

--dump-outputs DIR writes what the timed iterations computed, as a caller of the resident trainer would
read it after the last timed step (pi, A, B, the per-iteration log-likelihood statistic of every word and
the per-sequence log-likelihoods of the last E-step), to DIR/<name>.npy; the inputs depend only on the
arguments, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import contextlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True  # the benchmark writes nothing into the source tree (which may be read-only)
sys.path.insert(0, ROOT)

HBM_FALLBACK_GBS = 6650.0  # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent

WORKLOADS = {
    # name: (W, S per word per GPU, T, N, M)
    "bw_c3": dict(W=10, S=100_000, T=200, N=4, M=256, desc="config 3: 10 words x 100k seq x T=200, N=4, M=256"),
    "bw_c4": dict(W=1000, S=500, T=200, N=16, M=1024, desc="config 4: 1000 words x 500 seq x T=200, N=16, M=1024"),
    "bw_n8": dict(W=1000, S=500, T=200, N=8, M=1024, desc="1000 words x 500 seq x T=200, N=8, M=1024 (left-to-right kernels at 8 states)"),
    "bw_c1": dict(W=10, S=20, T=100, N=4, M=256, desc="config 1: 10 words x 20 seq x T~100 (latency-bound parity config)"),
}


def measured_traffic(workload: str, kernel: str, frames: int):
    """DRAM bytes per launch of `kernel` from the committed ncu capture (profiles/traffic.json:
    dram__bytes_read.sum + dram__bytes_write.sum per frame of the captured launch, scaled to this
    launch's frame count); None if no capture is recorded for the workload."""
    try:
        rec = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[workload][kernel]
        return rec["dram_bytes_per_frame"] * frames, rec.get("source")
    except Exception:
        return None, None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock, power and throttle reasons sampled DURING the timed region (B200_PROFILING.md):
    NVML every ~2 ms from a thread (the timed region of the default workload is tens of
    milliseconds, shorter than one nvidia-smi call); nvidia-smi is the fallback."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.samples = []          # (sm_mhz, power_w, reasons bitmask)
        self.sm_max = None
        self.source = None
        self._stop = threading.Event()
        self._t = None
        self._nvml = None
        self._h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical devices: honour CUDA_VISIBLE_DEVICES
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if vis:
                ids = [v.strip() for v in vis.split(",") if v.strip()]
                if index < len(ids) and ids[index].isdigit():
                    phys = int(ids[index])
            self._h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self._nvml = pynvml
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
            self.source = "nvml"
        except Exception:
            self._nvml = None
            self.source = "nvidia-smi"

    def _sample_nvml(self):
        n = self._nvml
        sm = float(n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM))
        try:
            pw = n.nvmlDeviceGetPowerUsage(self._h) / 1000.0
        except Exception:
            pw = None
        try:
            rs = int(n.nvmlDeviceGetCurrentClocksEventReasons(self._h))
        except Exception:
            try:
                rs = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self._h))
            except Exception:
                rs = 0
        self.samples.append((sm, pw, rs))

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
        parts = [x.strip() for x in out.strip().split(",")]
        if len(parts) >= 7:
            bits = 0
            for i, b in enumerate((0x8, 0x40, 0x20, 0x4)):  # hw_slowdown, hw_thermal, sw_thermal, sw_power_cap
                if parts[3 + i].lower().startswith("active"):
                    bits |= b
            self.sm_max = float(parts[1])
            self.samples.append((float(parts[0]), float(parts[2]), bits))

    def _run(self):
        try:  # first NVML query of a thread is slow: take (and drop) it before the timed region starts
            if self._nvml:
                self._sample_nvml()
                self.samples.clear()
        except Exception:
            pass
        self._ready.set()
        while not self._stop.is_set():
            try:
                if self._nvml:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self._stop.wait(0.002 if self._nvml else 0.2)

    def __enter__(self):
        self.samples = []
        self._stop.clear()
        self._ready = threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        self._ready.wait(5.0)
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": [], "samples": 0, "source": self.source}
        sm = sorted(s[0] for s in self.samples)
        pw = [s[1] for s in self.samples if s[1] is not None]
        bits = 0
        for s in self.samples:
            bits |= s[2]
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        reasons = [n for b, n in names.items() if bits & b]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.sm_max, "power_w_max": max(pw) if pw else None,
                "reasons": reasons, "samples": len(self.samples), "source": self.source}


class SmiLoopSampler:
    """Clocks for multi-rank runs: one `nvidia-smi -lms` child process on rank 0 (the recipe's own way).  A
    Python sampler thread cannot be used there: the all-reduce hook is a Python callback, so every EM iteration
    needs the GIL, and an NVML-polling thread made rank 0 the straggler of every all-reduce (measured on 8 GPUs:
    4.0-4.5 ms per iteration with the thread, 3.53 ms without)."""

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.samples = []
        self.sm_max = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={ClockSampler.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
        return self

    def stop(self):
        if not self.proc:
            return
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        for line in out.splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) >= 7 and parts[0].replace(".", "").isdigit():
                bits = 0
                for i, b in enumerate((0x8, 0x40, 0x20, 0x4)):
                    if parts[3 + i].lower().startswith("active"):
                        bits |= b
                self.sm_max = float(parts[1])
                pw = float(parts[2]) if parts[2].replace(".", "").isdigit() else None
                self.samples.append((float(parts[0]), pw, bits))

    def summary(self):
        c = ClockSampler.__new__(ClockSampler)
        c.samples, c.sm_max, c.source = self.samples, self.sm_max, "nvidia-smi -lms 20 (rank 0, from the warm-up on)"
        return ClockSampler.summary(c)


# ----------------------------------------------------------------------------- CPU arm
# BASELINE.md §2 (survey, build container, the UNMODIFIED reference on one core; it cannot travel to the GPU box):
LITERAL_REFERENCE_SURVEY = {
    "baum_welch_frames_per_s_per_iter": 2405.0, "vq_encode_frames_per_s": 1000.0, "score_frame_models_per_s": 17600.0,
    "lbg_frame_centroid_pairs_per_s": 172000.0, "cores": 1,
    "source": "BASELINE.md section 2: unmodified reference timed in the build container at survey time (not re-measured here)"}


def _cpu_estep_job(args):
    from oracle import hmm_oracle as O
    seqs, lp, lA, lB, M = args
    return O.estep_logsums(seqs, lp, lA, lB, M)


def cpu_baum_welch(cfg, seq_per_word: int, iters: int, procs: int, max_words: int = 40):
    """One EM iteration of the CPU oracle (numpy restatement of the reference's log-space Baum-Welch) on a bounded
    sample of the workload, on `procs` host cores: every word's sequences are cut into chunks, the chunks of all
    words go through one process pool (oracle.estep_logsums), and the parent merges each word's chunks with
    log_sum_exp and applies the M-step — the whole iteration the reference runs, with all the parallelism its
    structure admits (words AND sequences are independent given the parameters)."""
    import multiprocessing as mp
    from hmm_training_b200 import engine, synthetic
    from oracle import hmm_oracle as O
    W, T, N, M = min(cfg["W"], max_words), cfg["T"], cfg["N"], cfg["M"]
    obs, offsets, wos = synthetic.fixed_length_codewords(12345, W, seq_per_word, T, N, M)
    pi0, A0, B0 = engine.default_init(N, M)
    lp, lA, lB = O.safe_log(pi0), O.safe_log(A0), O.safe_log(B0)
    rows = obs.reshape(W * seq_per_word, T)
    # ~4 chunks per core so that the pool stays busy to the end
    chunk = max(8, min(seq_per_word, (W * seq_per_word + 4 * procs - 1) // (4 * max(procs, 1))))
    jobs, owner = [], []
    for w in range(W):
        for lo in range(0, seq_per_word, chunk):
            part = rows[w * seq_per_word + lo: w * seq_per_word + min(seq_per_word, lo + chunk)]
            jobs.append(([r.astype(np.int64) for r in part], lp, lA, lB, M))
            owner.append(w)
    pool = mp.get_context("fork").Pool(procs) if procs > 1 else None
    t0 = time.perf_counter()
    for _ in range(iters):
        parts = pool.map(_cpu_estep_job, jobs, chunksize=1) if pool else [_cpu_estep_job(j) for j in jobs]
        for w in range(W):
            O.mstep_from_logsums(O.merge_logsums([p for p, o in zip(parts, owner) if o == w]), N, M)
    dt = time.perf_counter() - t0
    if pool:
        pool.close()
        pool.join()
    frames = W * seq_per_word * T
    return frames * iters / dt, dt, (f"{W} words x {seq_per_word} seq x T={T} (N={N}, M={M}), {iters} EM iteration(s), "
                                     f"{len(jobs)} chunks of <= {chunk} sequences on {procs} process(es)")


def run_reference(args, cfg, real_stdout):
    """--impl reference: the reference's algorithm on the host cores.  The reference itself is
    pure Python and only exists in the build container, so this arm times oracle/ (the
    validated numpy port, kind="port") with every host core, on the same workload shape."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    spw = int(os.environ.get("HMMB_CPU_SEQ_PER_WORD", "4000" if cfg["N"] <= 4 else "100"))
    for _ in range(max(args.warmup, 0) and 1):
        cpu_baum_welch(cfg, max(spw // 4, 1), 1, cores)
    vals, wall = [], 0.0
    for _ in range(args.steps):
        v, dt, sample = cpu_baum_welch(cfg, spw, 1, cores)  # (dt: the EM iteration alone, data generation excluded)
        vals.append(v)
        wall += dt
    value = float(np.mean(vals))
    one_core, _, one_sample = cpu_baum_welch(cfg, max(min(spw // 8, 500), 1), 1, 1, max_words=1)
    line = {
        "impl": "reference", "metric": "baum_welch_frames_per_s_per_iter", "value": value, "unit": "frames/s/iter",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": cfg["desc"], "sample": sample},
        "cpu_baseline": {"value": value, "unit": "frames/s/iter", "cores": cores, "kind": "port", "sample": sample,
                         "one_core": {"value": one_core, "sample": one_sample},
                         "literal_reference_survey": LITERAL_REFERENCE_SURVEY},
        "e2e": {"value": value, "unit": "frames/s/iter", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    _emit(real_stdout, line)


# ----------------------------------------------------------------------------- GPU arm
def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version
    line to stdout on this image), so file descriptor 1 is pointed at stderr for the whole run and
    the JSON line goes to the saved original descriptor."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return real


def _emit(real_fd: int, line: dict) -> None:
    sys.stdout.flush()
    os.write(real_fd, (json.dumps(line) + "\n").encode())


class Env:
    """What every block of the GPU arm needs: torch, the library, rank / world, barrier and max-over-ranks."""

    def __init__(self, torch, dist, lib, _lib, engine, synthetic, hdist, rank, world, local_rank):
        self.torch, self.dist, self.lib, self._lib = torch, dist, lib, _lib
        self.engine, self.synthetic, self.hdist = engine, synthetic, hdist
        self.rank, self.world, self.local_rank = rank, world, local_rank
        self.native = False  # the library's own NCCL communicator exists

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return float(x)
        t = self.torch.tensor([x], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return float(x)
        t = self.torch.tensor([x], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def allreduce_hook(self, kind: str):
        """kind = 'native' (hmmb_comm_allreduce: NCCL called from C inside the EM loop, no Python between the
        E-step and the M-step) or 'torch' (torch.distributed.all_reduce from a ctypes callback, under the GIL)."""
        if self.world == 1:
            return None
        return "native" if (kind == "native" and self.native) else self.hdist.make_allreduce()


PHASES = ("bw_forward", "bw_exact", "bw_backward", "bw_reduce", "bw_allreduce", "bw_mstep")


def time_baum_welch(env: Env, bw, steps: int, warmup: int, sampler=None, on_timed=None):
    """W untimed warm-up iterations, then `steps` iterations queued back to back between barrier + synchronize,
    CUDA events on the launching stream, profiling events OFF (this is `value`); then the same number of
    iterations once more with the library's per-launch events on, for the per-kernel times of the roofline.
    on_timed(bw) is called between the two, outside the timed region."""
    torch, lib, _lib = env.torch, env.lib, env._lib
    done = int(bw.history(1)[1].max(initial=0))  # iterations the model already ran (max_iterations counts them too)
    # max_iterations of the calls below: never reached (a word that reaches it stops being trained)
    cap = max(1 << 14, done + warmup + 2 * steps + 1)
    bw.iterate(warmup, -1.0, cap, sync_each=False)
    env.barrier()
    l0 = lib.hmmb_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with (sampler if sampler is not None else contextlib.nullcontext()):
        ev0.record()
        bw.iterate(steps, -1.0, cap, sync_each=False)
        ev1.record()
        env.barrier()
    ms = env.max_over_ranks(ev0.elapsed_time(ev1))
    launches = int(lib.hmmb_launch_count() - l0)
    if on_timed is not None:
        on_timed(bw)
    _lib.check(lib.hmmb_set_profiling(1))
    _lib.check(lib.hmmb_phase_reset())
    env.barrier()
    bw.iterate(steps, -1.0, cap, sync_each=False)
    env.barrier()
    phases = {}
    for name in PHASES:
        pms, n = _lib.phase_ms(name)
        if n:
            phases[name] = {"ms_per_launch": pms / n, "launches": n}
    _lib.check(lib.hmmb_set_profiling(0))
    return ms / steps, launches, phases


DUMP_LIMIT_BYTES = 64_000_000


def bw_outputs(bw, iterations: int):
    """What a caller of the resident trainer reads back after `iterations` EM iterations: the model, the
    per-iteration log-likelihood statistic of every word and the per-sequence log-likelihoods of the last E-step."""
    pi, A, B = bw.params()
    hist, _ = bw.history(iterations)
    return {"pi": pi, "A": A, "B": B, "ll_hist": hist, "seq_ll": bw.seq_ll()}


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Every array as out_dir/<name>.npy in float64, DUMP_LIMIT_BYTES in all at most: an array larger than its
    share is cut to a fixed, seeded sample of its rows (leading axis), the same rows on every run."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_LIMIT_BYTES // len(arrays) - 4096  # (room for the .npy header)
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float64)
        if a.nbytes > share:
            rows = np.random.default_rng(0).choice(len(a), max(1, share // (a.nbytes // len(a))), replace=False)
            a = a[np.sort(rows)]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def bw_roofline(workload, family, phases, frames_rank, N, M, hbm_peak, peak_src):
    """Roofline of the dominant E-step kernel: algorithmic bytes (DESIGN.md §6: s_idx + 8 N per frame and kernel)
    over its mean CUDA-event duration, against the measured HBM copy bandwidth."""
    sym_b = 1 if M <= 256 else 2
    alg = {"bw_forward": frames_rank * (sym_b + 8 * N), "bw_backward": frames_rank * (sym_b + 8 * N)}
    dom = max((k for k in alg if k in phases), key=lambda k: phases[k]["ms_per_launch"], default=None)
    if not dom:
        return None
    ach = alg[dom] / (phases[dom]["ms_per_launch"] * 1e-3) / 1e9
    estep_ms = sum(phases[k]["ms_per_launch"] for k in ("bw_forward", "bw_backward") if k in phases)
    kname = {"n4_left_to_right": "k_bw_%s4<true>", "n4_dense": "k_bw_%s4<false>", "left_to_right": "k_bw_%sL",
             "generic": "k_bw_%sG"}.get(family, "k_bw_%s") % ("bwd" if dom == "bw_backward" else "fwd")
    traffic, traffic_src = measured_traffic(workload, dom, frames_rank)
    est = frames_rank * (2 * sym_b + 16 * N) / (estep_ms * 1e-3) / 1e9
    return {"bound": "hbm", "kernel": kname, "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
            "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": alg[dom],
            "estep": {"algorithmic_bytes_per_frame": 2 * sym_b + 16 * N, "achieved": est, "frac": est / hbm_peak},
            "phases": phases}


def make_bw(env: Env, cfg, seed: int, S=None, hook="native"):
    """Resident Baum-Welch problem of shape cfg on this rank (S sequences per word), default parameters."""
    engine, synthetic = env.engine, env.synthetic
    W, T, N, M = cfg["W"], cfg["T"], cfg["N"], cfg["M"]
    S = cfg["S"] if S is None else S
    obs, offsets, wos = synthetic.fixed_length_codewords(seed, W, S, T, N, M)
    pi0, A0, B0 = engine.default_init(N, M)
    init = (np.tile(pi0, (W, 1)), np.tile(A0, (W, 1, 1)), np.tile(B0, (W, 1, 1)))
    bw = engine.BaumWelch(obs, offsets, wos, W, N, M)
    bw.set_params(*init)
    if env.world > 1:
        bw.set_dist(env.rank, env.world, env.allreduce_hook(hook))
    return bw, (obs, offsets, wos), init


def block_config4(env: Env, args, hbm_peak, peak_src):
    """BASELINE config 4 (the multi-GPU configuration north_star names): 1000 words, 16 states, 1024 codewords,
    500 sequences per word PER GPU (weak scaling), one 133 MB fp64 all-reduce per iteration."""
    cfg = dict(WORKLOADS["bw_c4"])
    cfg["S"] = max(1, int(round(cfg["S"] * args.scale)))
    bw, (obs, offsets, wos), init = make_bw(env, cfg, 3000 + env.rank)
    frames_rank = int(offsets[-1])
    steps = max(3, min(args.steps, 6))
    ms, launches, phases = time_baum_welch(env, bw, steps, 3)
    family = bw.kernel_family()
    exact, handover = bw.diagnostics()
    bw.close()
    W, N, M = cfg["W"], cfg["N"], cfg["M"]
    accum_doubles = W * (((N + N * N + M * N) + 1 + 15) // 16 * 16) + env.world * W * 2
    # end to end through engine.bw_fit, one EM iteration per call; codewords, the 131 MB of initial parameters and the
    # 133 MB of results all in pinned host memory, so that every copy is one direct DMA
    e2e = None
    try:
        torch = env.torch

        def pin(a):  # copy into pinned host memory (torch has no uint16 tensors on every version: go through int16)
            a = np.ascontiguousarray(a)
            src = a.view(np.int16) if a.dtype == np.uint16 else a
            return torch.from_numpy(src).pin_memory().numpy().view(a.dtype)

        obs_h, off_h, wos_h = pin(obs), pin(offsets), pin(wos)
        init_h = tuple(pin(x) for x in init)
        out_h = tuple(pin(np.zeros_like(x)) for x in init)
        ar = env.allreduce_hook("native")
        call = lambda: env.engine.bw_fit(obs_h, off_h, wos_h, W, N, M, *init_h, -1.0, 1, allreduce=ar, rank=env.rank,
                                         world=env.world, out=out_h)
        call()
        env.barrier()
        t0 = time.perf_counter()
        for _ in range(2):
            res = call()
        env.barrier()
        dt = env.max_over_ranks((time.perf_counter() - t0) / 2)
        e2e = {"value": frames_rank * env.world / dt, "unit": "frames/s/iter", "ms_per_step": dt * 1e3,
               "h2d_bytes_per_step": int(obs_h.nbytes + off_h.nbytes + wos_h.nbytes + sum(x.nbytes for x in init_h)),
               "d2h_bytes_per_step": int(sum(x.nbytes for x in res)), "buffers": "pinned (inputs and outputs)"}
    except Exception as exc:  # pragma: no cover
        e2e = {"error": repr(exc)}
    out = {"workload": cfg["desc"], "scaling": "weak", "frames_per_gpu_per_iter": frames_rank, "ms_per_step": ms,
           "value": frames_rank * env.world / (ms * 1e-3), "unit": "frames/s/iter", "steps": steps,
           "kernel_family": family, "gpu_launches": launches,
           "allreduce_bytes": accum_doubles * 8,
           "allreduce_ms": phases.get("bw_allreduce", {}).get("ms_per_launch"),
           "roofline": bw_roofline("bw_c4", family, phases, frames_rank, N, M, hbm_peak, peak_src),
           "e2e": e2e, "precision_guard": {"exact_sequence_passes": exact, "backward_handovers": handover}}
    return out


def block_strong(env: Env, args, headline_ms):
    """Strong scaling: config 3's 200 M frames per iteration in TOTAL, split over the ranks (every rank generates
    its own 1/world of the sequences of every word)."""
    cfg = dict(WORKLOADS["bw_c3"])
    S_total = max(env.world, int(round(cfg["S"] * args.scale)))
    if env.world == 1:
        return {"workload": cfg["desc"], "scaling": "strong", "frames_total_per_iter": cfg["W"] * S_total * cfg["T"],
                "ms_per_step": headline_ms, "value": cfg["W"] * S_total * cfg["T"] / (headline_ms * 1e-3),
                "unit": "frames/s/iter", "note": "one rank: identical to the headline run"}
    S = S_total // env.world
    bw, (obs, offsets, wos), _ = make_bw(env, cfg, 2000 + env.rank, S=S)
    ms, launches, phases = time_baum_welch(env, bw, args.steps, 3)
    bw.close()
    frames_total = cfg["W"] * S * cfg["T"] * env.world
    return {"workload": cfg["desc"], "scaling": "strong", "frames_total_per_iter": frames_total,
            "seq_per_word_per_gpu": S, "ms_per_step": ms, "value": frames_total / (ms * 1e-3), "unit": "frames/s/iter",
            "allreduce_ms": phases.get("bw_allreduce", {}).get("ms_per_launch"),
            "phases": {k: v["ms_per_launch"] for k, v in phases.items()}}


def _rel_err(x, ref):
    x, ref = np.asarray(x, float), np.asarray(ref, float)
    both_inf = np.isinf(ref) & (x == ref)
    d = np.abs(x - ref) / np.maximum(np.abs(ref), 1e-300)
    d[both_inf] = 0.0
    d[(ref == 0) & (x == 0)] = 0.0
    d[np.isnan(ref) & np.isnan(x)] = 0.0
    return float(np.nanmax(d)) if d.size else 0.0


def block_parity(env: Env):
    """SURVEY.md 8e "Determinism": world-rank training must agree with a single-rank run on the same sequences to
    1e-12 relative (NCCL's summation order differs, nothing else may).  Every rank first trains the whole
    sub-sample alone (no collective), then its round-robin shard with the all-reduce; the models and the
    log-likelihood histories are compared on every rank and the worst error over ranks is reported.  Same for the
    LBG codebook: iteration counts per generation equal, centroids to 1e-12."""
    engine, synthetic, hdist = env.engine, env.synthetic, env.hdist
    tol = 1e-12
    out = {"ranks": env.world, "tolerance": tol, "cases": {}}
    if env.world == 1:
        out["note"] = "one rank: nothing to compare (the 2-rank comparison runs in tests/test_gpu_multi.py and at --gpus >= 2)"
        out["pass"] = True
        return out
    ok = True
    for name, (W, S, T, N, M, iters) in {"config3_shape": (10, 4096, 200, 4, 256, 3),
                                         "config4_shape": (24, 96, 200, 16, 1024, 3)}.items():
        obs, offsets, wos = synthetic.fixed_length_codewords(4242, W, S, T, N, M)
        pi0, A0, B0 = engine.default_init(N, M)
        init = (np.tile(pi0, (W, 1)), np.tile(A0, (W, 1, 1)), np.tile(B0, (W, 1, 1)))
        single = engine.bw_fit(obs, offsets, wos, W, N, M, *init, -1.0, iters)
        mine = hdist.shard_sequences_round_robin(wos, env.rank, env.world)
        rows = obs.reshape(W * S, T)[mine]
        off = np.arange(len(mine) + 1, dtype=np.int64) * T
        errs = {}
        for kind in ("native", "torch"):
            if kind == "native" and not env.native:
                continue
            multi = engine.bw_fit(np.ascontiguousarray(rows.reshape(-1)), off, wos[mine], W, N, M, *init, -1.0, iters,
                                  allreduce=env.allreduce_hook(kind), rank=env.rank, world=env.world)
            e = max(_rel_err(a, b) for a, b in zip(multi[:4], single[:4]))
            same_iters = bool(np.array_equal(multi[4], single[4]))
            errs[kind] = env.max_over_ranks(e)
            ok = ok and errs[kind] <= tol and same_iters
        out["cases"][name] = {"max_rel_err": errs, "frames": int(W * S * T), "iterations": iters}
    # LBG: frames sharded contiguously, centroid sums / counts / distance all-reduced once per Lloyd pass
    X = synthetic.mfcc_mixture(7, 65536, 64)
    C1, _, _, it1, gd1 = engine.lbg_fit(X, 64, 25, 1e-3)
    lo, hi = hdist.shard_range(len(X), env.rank, env.world)
    Cn, _, _, itn, gdn = engine.lbg_fit(X[lo:hi], 64, 25, 1e-3, allreduce=env.allreduce_hook("native"))
    e = env.max_over_ranks(max(_rel_err(Cn, C1), _rel_err(gdn, gd1)))
    same = bool(np.array_equal(it1, itn))
    out["cases"]["lbg_65536x64"] = {"max_rel_err": e, "iters_per_generation_equal": same,
                                    "iters_per_generation": [int(i) for i in itn]}
    ok = ok and e <= 1e-9 and same  # (centroid means are sums of ~1e3 frames: 1e-12 of the sum, looser on the mean of a small cluster)
    out["pass"] = bool(env.max_over_ranks(0.0 if ok else 1.0) == 0.0)
    return out


def block_shards(env: Env):
    """BASELINE config 5 ("1-8 B200") and VQ encode as pure shards: the utterances / frames are split over the
    ranks, no collective on the data path; every rank times its own host-API call (pinned host buffers, H2D and
    D2H inside) between two barriers and the aggregate is total units / slowest rank."""
    torch, engine, synthetic = env.torch, env.engine, env.synthetic
    out = {}
    U_total, Wm, T = 1_000_000, 10, 100
    U = U_total // env.world
    rng = np.random.default_rng(5)
    obs, offsets, _ = synthetic.fixed_length_codewords(77 + env.rank, Wm, U // Wm, T, 4, 256)
    U = len(offsets) - 1
    pi, A, _ = engine.default_init(4, 256)
    Bm = rng.dirichlet(np.ones(256) * 0.3, size=(Wm, 4))
    pim, Am = np.tile(pi, (Wm, 1)), np.tile(A, (Wm, 1, 1))
    obs_p = torch.empty(obs.shape, dtype=torch.uint8, pin_memory=True).numpy()
    obs_p[:] = obs
    ll_p = torch.empty((U, Wm), dtype=torch.float64, pin_memory=True).numpy()
    engine.score(obs_p, offsets, 4, 256, pim, Am, Bm, out_ll=ll_p)
    res = {}
    for label, kw in (("ll_and_argmax", dict(out_ll=ll_p)), ("argmax_only", dict(want_ll=False))):
        reps = 3
        env.barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            engine.score(obs_p, offsets, 4, 256, pim, Am, Bm, **kw)
        dt = env.max_over_ranks((time.perf_counter() - t0) / reps)
        res[label] = {"value": U * env.world / dt, "seconds": dt}
    out["score_sharded"] = {"metric": "recognition_utterances_per_s", "unit": "utterances/s (host API per rank, pinned buffers)",
                            "utterances_total": U * env.world, "models": Wm, "T": T, "ranks": env.world,
                            "parallelism": "utterance ranges per rank, no collective", **res}
    F_total, K = 1_000_000, 256
    F = F_total // env.world
    X = synthetic.mfcc_mixture(100 + env.rank, F, K)
    C = synthetic.random_codebook(1, K)
    Xp = torch.from_numpy(X).pin_memory().numpy()
    engine.vq_encode(Xp, C)
    env.barrier()
    t0 = time.perf_counter()
    for _ in range(3):
        engine.vq_encode(Xp, C)
    dt = env.max_over_ranks((time.perf_counter() - t0) / 3)
    out["vq_encode_sharded"] = {"metric": "vq_encode_frames_per_s", "value": F * env.world / dt, "unit": "frames/s (host API per rank, pinned buffers)",
                                "frames_total": F * env.world, "K": K, "ranks": env.world, "seconds": dt,
                                "parallelism": "frame ranges per rank, no collective"}
    # BASELINE config 2's codebook build with the frames split over the ranks: every Lloyd pass ends in one
    # sum-all-reduce of the centroid sums, counts and the global distance (<= 28.7 KB; SURVEY 8e)
    try:
        ar = env.allreduce_hook("native") if env.world > 1 else None
        engine.lbg_fit(Xp, K, 100, 1e-3, allreduce=ar)
        env.barrier()
        t0 = time.perf_counter()
        _, _, _, iters, _ = engine.lbg_fit(Xp, K, 100, 1e-3, allreduce=ar)
        dt = env.max_over_ranks(time.perf_counter() - t0)
        out["lbg_sharded"] = {"metric": "lbg_codebook_build_s", "value": dt, "unit": "s", "higher_is_better": False,
                              "frames_total": F * env.world, "K": K, "ranks": env.world, "lloyd_passes": int(np.sum(iters)),
                              "allreduce": "one per Lloyd pass (centroid sums + counts + distance)",
                              "parallelism": "frame ranges per rank"}
    except Exception as exc:  # pragma: no cover
        out["lbg_sharded"] = {"error": repr(exc)}
    return out


def block_h2d_probe(env: Env):
    """Pinned host -> device copy ceiling with every rank copying at once (what bounds `e2e` at N > 1)."""
    torch = env.torch
    nbytes = 256 << 20
    src = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    src.fill_(1)
    dst = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    dst.copy_(src, non_blocking=True)
    env.barrier()
    t0 = time.perf_counter()
    for _ in range(4):
        dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / 4
    mine = nbytes / dt / 1e9
    slow = nbytes / env.max_over_ranks(dt) / 1e9
    return {"bytes_per_copy": nbytes, "concurrent_ranks": env.world, "gbs_this_rank": mine, "gbs_slowest_rank": slow,
            "gbs_aggregate": env.sum_over_ranks(mine)}


def main():
    real_stdout = _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="bw_c3", choices=list(WORKLOADS))
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the workload's sequences (debug)")
    ap.add_argument("--no-extras", action="store_true", help="headline + e2e only (no config 4 / strong / parity / shard / VQ / LBG / scoring / CPU blocks)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    cfg = dict(WORKLOADS[args.workload])
    cfg["S"] = max(1, int(round(cfg["S"] * args.scale)))
    if args.impl == "reference":
        run_reference(args, cfg, real_stdout)
        return
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        # torchrun exports OMP_NUM_THREADS=1; give every rank its share of the host cores for the library's
        # host-side blocking (hmmb_init reads HMMB_HOST_THREADS)
        local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
        os.environ.setdefault("HMMB_HOST_THREADS", str(max(1, min(8, (os.cpu_count() or 1) // max(local_world, 1)))))
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from hmm_training_b200 import _lib, engine, synthetic
    from hmm_training_b200 import dist as hdist
    affinity = hdist.cpu_affinity_info(local_rank)
    bound_cpus = hdist.bind_to_gpu_cpus(local_rank) if world > 1 else 0  # NUMA-local pinned buffers and host threads
    lib = _lib.load()
    _lib.init(local_rank)
    hdist.bind_torch_stream()
    env = Env(torch, dist, lib, _lib, engine, synthetic, hdist, rank, world, local_rank)
    if world > 1:
        try:
            hdist.native_comm_init(rank, world)
            env.native = True
        except Exception as exc:  # pragma: no cover
            print(f"[bench] native communicator unavailable ({exc!r}); using the torch hook", file=sys.stderr)
    hbm_peak, peak_src = measured_peaks()
    fp64_peak, fp32_peak = ctypes_double(lib, _lib, 0), ctypes_double(lib, _lib, 1)

    W, S, T, N, M = cfg["W"], cfg["S"], cfg["T"], cfg["N"], cfg["M"]
    bw, (obs, offsets, wos), (pi0, A0, B0) = make_bw(env, cfg, 1000 + rank)
    frames_rank = int(offsets[-1])
    smi = SmiLoopSampler(local_rank).start() if (world > 1 and rank == 0) else None
    if smi:
        time.sleep(1.0)  # nvidia-smi needs about a second to start printing
    # single GPU: NVML thread every ~2 ms during the timed region; several ranks: an nvidia-smi child of rank 0
    clk = ClockSampler(local_rank) if world == 1 else None
    on_timed = None
    if args.dump_outputs and rank == 0:
        on_timed = lambda b: dump_outputs(args.dump_outputs, bw_outputs(b, args.warmup + args.steps))
    ms_per_step, gpu_launches, phases = time_baum_welch(env, bw, args.steps, args.warmup, sampler=clk, on_timed=on_timed)
    if smi:
        time.sleep(0.05)
        smi.stop()
        clk = smi
    exact_passes, bwd_handover = bw.diagnostics()
    bw_family = bw.kernel_family()
    allreduce_info = None
    if world > 1:
        # the same loop once more through the other plumbing: torch.distributed from a Python callback
        bw.set_dist(rank, world, env.allreduce_hook("torch"))
        ms_torch, _, ph_torch = time_baum_welch(env, bw, args.steps, 2)
        allreduce_info = {"default": "native (hmmb_comm_allreduce: ncclAllReduce called from C on the library's stream)" if env.native
                          else "torch hook (native communicator unavailable)",
                          "ms_per_step_default": ms_per_step, "ms_per_step_torch_hook": ms_torch,
                          "allreduce_ms": phases.get("bw_allreduce", {}).get("ms_per_launch"),
                          "allreduce_ms_torch_hook": ph_torch.get("bw_allreduce", {}).get("ms_per_launch"),
                          "bytes": (W * (((N + N * N + M * N) + 1 + 15) // 16 * 16) + world * W * 2) * 8}
    frames_total = frames_rank * world
    value = frames_total / (ms_per_step * 1e-3)
    bw.close()
    roofline = bw_roofline(args.workload, bw_family, phases, frames_rank, N, M, hbm_peak, peak_src)

    # ---- e2e: public packed-array API from pinned host buffers, one EM iteration per call
    e2e = None
    try:
        obs_p = torch.empty(obs.shape, dtype=torch.uint8 if obs.dtype == np.uint8 else torch.int16, pin_memory=True)
        obs_h = obs_p.numpy().view(obs.dtype)
        obs_h[:] = obs
        off_h = torch.from_numpy(offsets).pin_memory().numpy()
        wos_h = torch.from_numpy(wos).pin_memory().numpy()
        ar = env.allreduce_hook("native")
        k_e2e = max(2, min(args.steps, 5))
        engine.bw_fit(obs_h, off_h, wos_h, W, N, M, pi0, A0, B0, -1.0, 1, allreduce=ar, rank=rank, world=world)
        env.barrier()
        t0 = time.perf_counter()
        for _ in range(k_e2e):
            out = engine.bw_fit(obs_h, off_h, wos_h, W, N, M, pi0, A0, B0, -1.0, 1, allreduce=ar, rank=rank, world=world)
        env.barrier()
        dt = env.max_over_ranks((time.perf_counter() - t0) / k_e2e)
        h2d = obs_h.nbytes + off_h.nbytes + wos_h.nbytes + pi0.nbytes + A0.nbytes + B0.nbytes
        d2h = sum(x.nbytes for x in out)
        e2e = {"value": frames_total / dt, "unit": "frames/s/iter", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "ms_per_step": dt * 1e3, "steps": k_e2e,
               "api": "engine.bw_fit (hmmb_bw_create/set_params/iterate/get_params) with pinned host buffers, 1 EM iteration per call"}
        del obs_p, obs_h
    except Exception as exc:  # pragma: no cover
        e2e = {"error": repr(exc)}
    del obs

    blocks = {}
    if not args.no_extras:
        for name, fn in (("h2d_probe", lambda: block_h2d_probe(env)),
                         ("config4", lambda: block_config4(env, args, hbm_peak, peak_src)),
                         ("strong", lambda: block_strong(env, args, ms_per_step)),
                         ("parity", lambda: block_parity(env)),
                         ("shards", lambda: block_shards(env))):
            try:
                t0 = time.perf_counter()
                res = fn()
                if name == "shards":
                    blocks.update(res)
                else:
                    blocks[name] = res
                print(f"[bench] block {name}: {time.perf_counter() - t0:.1f} s", file=sys.stderr)
            except Exception as exc:  # pragma: no cover - a failing secondary block must not lose the headline
                import traceback
                traceback.print_exc()
                blocks[name] = {"error": repr(exc)}
        if e2e and "ms_per_step" in e2e and "h2d_probe" in blocks and "gbs_slowest_rank" in blocks["h2d_probe"]:
            e2e["h2d_floor_ms"] = e2e["h2d_bytes_per_step"] / (blocks["h2d_probe"]["gbs_slowest_rank"] * 1e9) * 1e3
            e2e["note"] = "h2d_floor_ms = this call's upload at the pinned-copy rate measured with all ranks copying at once"
        if rank == 0 and world == 1:
            blocks.update(run_extras(torch, lib, _lib, engine, synthetic, hbm_peak, True, fp64_peak, fp32_peak))

    cpu_baseline = None
    if world == 1 and not args.no_extras:
        cores = os.cpu_count() or 1
        # bounded sample of the same workload: ~10-20 s of CPU work on all host cores
        spw = int(os.environ.get("HMMB_CPU_SEQ_PER_WORD", "6000" if N <= 4 else "300"))
        v, dt, sample = cpu_baum_welch(cfg, spw, 1, cores)
        v1, dt1, sample1 = cpu_baum_welch(cfg, max(min(spw // 8, 500), 1), 1, 1, max_words=1)
        cpu_baseline = {"value": v, "unit": "frames/s/iter", "cores": cores, "kind": "port", "sample": sample,
                        "seconds": dt, "one_core": {"value": v1, "sample": sample1, "seconds": dt1},
                        "literal_reference_survey": LITERAL_REFERENCE_SURVEY}

    if rank == 0:
        line = {
            "metric": "baum_welch_frames_per_s_per_iter", "value": value, "unit": "frames/s/iter", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": cfg["desc"], "frames_per_gpu_per_iter": frames_rank, "W": W, "seq_per_word_per_gpu": S,
                       "T": T, "N": N, "M": M, "parallelism": f"sequences sharded over {world} GPU(s), 1 allreduce/iter",
                       "l2": "inputs larger than L2 (codewords + alpha spill >> 126 MB)",
                       "timing": "value: CUDA events around the K iterations with the library's per-launch events OFF; roofline.phases: a second pass of K iterations with them on",
                       "cpus_bound_per_rank": bound_cpus, "cpu_affinity": affinity},
            "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "gpu_launches": gpu_launches,
            "clocks": clk.summary(), "precision_guard": {"exact_sequence_passes": exact_passes,
                                                         "backward_handovers": bwd_handover},
            "peaks": {"hbm_gbs": hbm_peak, "hbm_source": peak_src, "fp64_tflops": fp64_peak, "fp32_tflops": fp32_peak,
                      "fp_source": "hmmb_peak_probe: FMA-only kernel, eight independent chains per thread, best of three, measured in this run"},
            "allreduce": allreduce_info,
        }
        line.update(blocks)
        _emit(real_stdout, line)
    # orderly teardown: free device memory and the library's events before NCCL goes away
    torch.cuda.synchronize()
    if env.native:
        hdist.native_comm_destroy()
    lib.hmmb_set_stream(None)
    lib.hmmb_shutdown()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def ctypes_double(lib, _lib, what: int) -> float:
    import ctypes
    v = ctypes.c_double(0.0)
    _lib.check(lib.hmmb_peak_probe(what, ctypes.byref(v)))
    return float(v.value)


def run_extras(torch, lib, _lib, engine, synthetic, hbm_peak, with_cpu, fp64_peak=None, fp32_peak=None):
    """Secondary blocks for BASELINE configs 2 (VQ / LBG, 1M frames) and 5 (recognition)."""
    out = {}
    F, K = 1_000_000, 256
    X = synthetic.mfcc_mixture(0, F, K)
    C = synthetic.random_codebook(1, K)
    dX = torch.from_numpy(X).cuda()
    dC = torch.from_numpy(C).cuda()
    dI = torch.empty(F, dtype=torch.int32, device="cuda")
    call = lambda: _lib.check(lib.hmmb_vq_encode_dev(dX.data_ptr(), F, dC.data_ptr(), K, dI.data_ptr(), None))
    for _ in range(3):
        call()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 10
    ev0.record()
    for _ in range(reps):
        call()
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / reps
    Xp = torch.from_numpy(X).pin_memory().numpy()
    engine.vq_encode(Xp, C)
    t0 = time.perf_counter()
    for _ in range(3):
        engine.vq_encode(Xp, C)
    dt = (time.perf_counter() - t0) / 3
    # two-stage search (DESIGN.md §6): fp32 prefilter ||c||^2 - 2 x.c = 12 FFMA per frame-centroid pair (24 flop), then
    # the winner's exact fp64 distance (24 DP operations per FRAME).  The kernel is bound by the fp32 / issue rate.
    pre_flops = F * K * 24.0
    out["vq_encode"] = {"metric": "vq_encode_frames_per_s", "value": F / (ms * 1e-3), "unit": "frames/s",
                        "frames": F, "K": K, "ms": ms,
                        "roofline": {"bound": "fp32 FMA / issue", "kernel": "k_vq_assign<0>",
                                     "achieved_tflops": pre_flops / (ms * 1e-3) / 1e12, "peak_tflops": fp32_peak,
                                     "frac": (pre_flops / (ms * 1e-3) / 1e12 / fp32_peak) if fp32_peak else None,
                                     "peak_source": "hmmb_peak_probe(fp32), this run",
                                     "direct_form_equivalent_fp64_tflops": F * K * 36.0 / (ms * 1e-3) / 1e12,
                                     "fp64_peak_tflops": fp64_peak,
                                     "hbm_achieved_gbs": F * 108 / (ms * 1e-3) / 1e9,
                                     "hbm_frac": F * 108 / (ms * 1e-3) / 1e9 / hbm_peak,
                                     "note": "12 FFMA + 5 min/max/select per frame-centroid pair on the fp32 / ALU pipes; the round-1 direct form "
                                             "(12 DADD + 12 DFMA per pair) ran at 83 % of the fp64 pipe (profiles/r2a_vq_assign_direct_form_ncu.md)"},
                        "e2e": {"value": F / dt, "unit": "frames/s", "h2d_bytes_per_step": int(X.nbytes + C.nbytes),
                                "d2h_bytes_per_step": 4 * F}}
    t0 = time.perf_counter()
    Cb, gens, assign, iters, gd = engine.lbg_fit(None, K, 100, 1e-3, x_dev_ptr=dX.data_ptr(), F=F)
    dt = time.perf_counter() - t0
    passes = int(iters.sum())
    out["lbg"] = {"metric": "lbg_codebook_build_s", "value": dt, "unit": "s", "frames": F, "K": K,
                  "lloyd_passes": passes, "iters_per_generation": [int(i) for i in iters],
                  "frame_passes_per_s": F * passes / dt}
    if with_cpu:
        from oracle import vq_oracle
        n = 20000
        vq_oracle.encode(X[:1000], C)
        t0 = time.perf_counter()
        vq_oracle.encode(X[:n], C)
        dtc = time.perf_counter() - t0
        out["vq_encode"]["cpu_baseline"] = {"value": n / dtc, "unit": "frames/s", "cores": os.cpu_count(), "kind": "port",
                                            "sample": f"{n} frames x K={K} (C oracle, OpenMP)",
                                            "literal_reference_survey": {"value": LITERAL_REFERENCE_SURVEY["vq_encode_frames_per_s"],
                                                                         "cores": 1, "source": LITERAL_REFERENCE_SURVEY["source"]}}
    del dX, dI
    # recognition (BASELINE config 5): U utterances x 10 models, pinned host buffers, warm
    U, Wm = 1_000_000, 10
    rng = np.random.default_rng(5)
    obs, offsets, _ = synthetic.fixed_length_codewords(77, Wm, U // Wm, 100, 4, 256)
    pi, A, B = engine.default_init(4, 256)
    Bm = rng.dirichlet(np.ones(256) * 0.3, size=(Wm, 4))
    pim, Am = np.tile(pi, (Wm, 1)), np.tile(A, (Wm, 1, 1))
    obs_p = torch.empty(obs.shape, dtype=torch.uint8, pin_memory=True).numpy()
    obs_p[:] = obs
    ll_p = torch.empty((U, Wm), dtype=torch.float64, pin_memory=True).numpy()
    engine.score(obs_p, offsets, 4, 256, pim, Am, Bm, out_ll=ll_p)
    reps = 3
    t0 = time.perf_counter()
    for _ in range(reps):
        ll, arg = engine.score(obs_p, offsets, 4, 256, pim, Am, Bm, out_ll=ll_p)
    dt = (time.perf_counter() - t0) / reps
    # kernel time from a separate pass with the library's per-launch CUDA events on (they cost ~0.4 ms per call)
    _lib.check(lib.hmmb_set_profiling(1))
    _lib.check(lib.hmmb_phase_reset())
    for _ in range(reps):
        engine.score(obs_p, offsets, 4, 256, pim, Am, Bm, out_ll=ll_p)
    kms, kn = _lib.phase_ms("score")
    _lib.check(lib.hmmb_set_profiling(0))
    t0 = time.perf_counter()
    for _ in range(reps):
        engine.score(obs_p, offsets, 4, 256, pim, Am, Bm, want_ll=False)
    dt_arg = (time.perf_counter() - t0) / reps
    kernel_ms = kms / reps  # all k_score4 launches of one call (the pipelined scorer launches it once per stage)
    fm = U * 100 * Wm  # frame x model pairs
    out["score"] = {"metric": "recognition_utterances_per_s", "value": U / dt,
                    "unit": "utterances/s (host API end to end, [U,W] log-likelihoods + argmax back on the host)",
                    "utterances": U, "models": Wm, "T": 100, "seconds": dt,
                    "argmax_only": {"value": U / dt_arg, "seconds": dt_arg},
                    "kernel": {"name": "k_score4r", "ms": kernel_ms, "frame_models_per_s": fm / (kernel_ms * 1e-3),
                               "fp64_tflops": fm * 45.0 / (kernel_ms * 1e-3) / 1e12, "fp64_peak_tflops": fp64_peak,
                               "frac": (fm * 45.0 / (kernel_ms * 1e-3) / 1e12 / fp64_peak) if fp64_peak else None,
                               "note": "45 flop per frame x model by SURVEY 8d's 2N^2 + 3N count (the bidiagonal kernel issues 11 DP "
                                       "instructions = 18 flop per step); issue-bound, no HBM stream to speak of"},
                    "h2d_bytes_per_step": int(obs_p.nbytes + offsets.nbytes), "d2h_bytes_per_step": int(ll_p.nbytes + 4 * U)}
    if with_cpu:
        from oracle import hmm_oracle as O
        nu = 400
        seqs = [obs[u * 100:(u + 1) * 100].astype(np.int64) for u in range(nu)]
        models = [(Am[w], Bm[w], pim[w]) for w in range(Wm)]
        O.score_batch(seqs[:20], models)
        t0 = time.perf_counter()
        O.score_batch(seqs, models)
        dtc = time.perf_counter() - t0
        out["score"]["cpu_baseline"] = {"value": nu / dtc, "unit": "utterances/s", "cores": 1, "kind": "port",
                                        "sample": f"{nu} utterances x {Wm} models, T=100 (numpy oracle, 1 core)"}
    # MFCC front-end (SURVEY 8f row 3; parity unpinned): 100k frames of 320 samples
    Ym = np.random.default_rng(9).normal(size=(100_000, 320)) * 1000.0
    Ymp = torch.from_numpy(Ym).pin_memory().numpy()
    engine.mfcc_frames(Ymp)  # warm: device blocks of this size enter the library's caching allocator
    _lib.check(lib.hmmb_set_profiling(1))
    _lib.check(lib.hmmb_phase_reset())
    t0 = time.perf_counter()
    engine.mfcc_frames(Ymp)
    dtm = time.perf_counter() - t0
    mms, _ = _lib.phase_ms("mfcc")
    _lib.check(lib.hmmb_set_profiling(0))
    out["mfcc"] = {"metric": "mfcc_frames_per_s", "value": len(Ym) / dtm, "unit": "frames/s (host API end to end)",
                   "frames": len(Ym), "frame_len": 320, "kernel_ms": mms, "kernel_frames_per_s": len(Ym) / (mms * 1e-3),
                   "h2d_bytes_per_step": int(Ym.nbytes), "d2h_bytes_per_step": len(Ym) * 13 * 8,
                   "note": "parity with librosa unpinned (oracle/mfcc_oracle.py)"}
    # config 5 stress variant: 1000 left-to-right models with 16 states and 1024 codewords (k_scoreL)
    Us, Ws, Ns, Ms, Ts = 100_000, 1000, 16, 1024, 100
    obs, offsets, _ = synthetic.fixed_length_codewords(78, 10, Us // 10, Ts, Ns, Ms)
    pi, A, B = engine.default_init(Ns, Ms)
    Bs = np.empty((Ws, Ns, Ms))
    base = rng.dirichlet(np.ones(Ms) * 0.3, size=(8, Ns))
    for w in range(Ws):
        Bs[w] = np.roll(base[w % 8], 7 * w, axis=1)
    pis, As = np.tile(pi, (Ws, 1)), np.tile(A, (Ws, 1, 1))
    obs_p = torch.empty(obs.shape, dtype=torch.int16, pin_memory=True).numpy().view(np.uint16)
    obs_p[:] = obs
    engine.score(obs_p[:Ts * 1000], offsets[:1001], Ns, Ms, pis, As, Bs, want_ll=False)
    _lib.check(lib.hmmb_set_profiling(1))
    _lib.check(lib.hmmb_phase_reset())
    t0 = time.perf_counter()
    engine.score(obs_p, offsets, Ns, Ms, pis, As, Bs, want_ll=False)
    dt = time.perf_counter() - t0
    kms, kn = _lib.phase_ms("score")
    _lib.check(lib.hmmb_set_profiling(0))
    fm = Us * Ts * Ws
    out["score_n16"] = {"metric": "recognition_utterances_per_s", "value": Us / dt, "unit": "utterances/s (host API, argmax only)",
                        "utterances": Us, "models": Ws, "N": Ns, "M": Ms, "T": Ts, "seconds": dt,
                        "kernel": {"name": "k_scoreL<16>", "ms": kms / max(kn, 1),
                                   "frame_models_per_s": fm / (kms / max(kn, 1) * 1e-3)}}
    return out


if __name__ == "__main__":
    main()

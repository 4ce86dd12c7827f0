"""End-to-end breakdown of one engine.bw_fit-style call (create / set / iterate / get / close), config 3 by default,
config 4 with C4=1; PINP=1 also pins the initial parameters and the result arrays."""
import sys, time, os
sys.path.insert(0, os.getcwd())
import numpy as np, torch
from hmm_training_b200 import _lib, engine, synthetic
_lib.init(0)
W,S,T,N,M=(1000,500,200,16,1024) if os.environ.get('C4') else (10,100000,200,4,256)
obs, off, wos = synthetic.fixed_length_codewords(1000, W,S,T,N,M)
def pin(a):
    a = np.ascontiguousarray(a)
    src = a.view(np.int16) if a.dtype == np.uint16 else a
    return torch.from_numpy(src).pin_memory().numpy().view(a.dtype)
obs_h = pin(obs)
pi0,A0,B0 = engine.default_init(N,M); pi0,A0,B0 = np.tile(pi0,(W,1)),np.tile(A0,(W,1,1)),np.tile(B0,(W,1,1))
out = None
if os.environ.get("PINP"):
    pi0, A0, B0 = pin(pi0), pin(A0), pin(B0)
    out = (pin(np.zeros_like(pi0)), pin(np.zeros_like(A0)), pin(np.zeros_like(B0)))
PIPE = os.environ.get("PIPE","1")=="1"
for rep in range(4):
    t=time.perf_counter(); bw = engine.BaumWelch(obs_h, off, wos, W,N,M, pipeline_upload=PIPE, init=(pi0,A0,B0) if PIPE else None); t1=time.perf_counter()
    if not PIPE: bw.set_params(pi0,A0,B0)
    t2=time.perf_counter()
    bw.iterate(1,-1.0,1,True); t3=time.perf_counter()
    res=bw.params(True, out=out); h=bw.history(1); t4=time.perf_counter(); bw.close(); t5=time.perf_counter()
    print('create %.2f set %.2f iterate %.2f get %.2f close %.2f total %.2f ms'%tuple(1e3*x for x in (t1-t,t2-t1,t3-t2,t4-t3,t5-t4,t5-t)), flush=True)
# phase timing of the pipelined first iteration (CUDA events around every launch)
lib = _lib.load()
_lib.check(lib.hmmb_set_profiling(1)); _lib.check(lib.hmmb_phase_reset())
bw = engine.BaumWelch(obs_h, off, wos, W, N, M, pipeline_upload=PIPE, init=(pi0, A0, B0) if PIPE else None)
if not PIPE: bw.set_params(pi0, A0, B0)
bw.iterate(1, -1.0, 1, True); bw.close()
print({k: (round(_lib.phase_ms(k)[0], 3), _lib.phase_ms(k)[1]) for k in ("prepare", "bw_load", "bw_forward", "bw_backward", "bw_exact", "bw_reduce", "bw_mstep", "bw_finalize")})
_lib.check(lib.hmmb_set_profiling(0))

import os, sys, ctypes as C
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from abrsimulator_b200 import synth, _lib
from abrsimulator_b200.env import BatchedABREnv
V=48
bitrates,sizes=synth.make_video(V)
bw,tl,ti=synth.make_traces(1024,2048)
N=131072
env=BatchedABREnv(bw,sizes,bitrates,N,trace_len=tl,trace_interval=ti,track_history=1,track_acc=1)
tid,off=synth.make_sessions(N,1024,2048,group=64)
env.reset(tid,off)
lib=_lib.load()
cnt=(C.c_ulonglong*4)()
act=torch.empty(N,dtype=torch.int32,device="cuda")
for t in range(48):
    lib.abr_debug_mpc_counters(cnt,1)
    env.mpc_decide(5,"robust",out=act)
    lib.abr_debug_mpc_counters(cnt,0)
    if t in (0,1,2,5,10,20,30,47):
        seen,ev,rows,rounds=[int(x) for x in cnt]
        print(f"chunk {t:2d}: prefixes evaluated {ev/max(seen,1):.3f}  rows/(6*prefixes seen) {rows/max(6*seen,1):.3f}  warp rounds executed per decision {rounds/N:.2f} of 7")
    env._lib.abr_env_step(env._h, C.c_void_p(act.data_ptr()), None,None,None,None,None,None,None,None, C.c_void_p(torch.cuda.current_stream().cuda_stream))

"""Development aid: wall time of one hm_match_host call from Python over small square problems (the single-launch path of
csrc/hm_small.cu)."""
import os
import sys, time, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from slam_experiments_b200 import _native as nat
ctx=nat.HostContext()
rng=np.random.default_rng(0)
for n in (8,64,200,400,512):
    q=rng.integers(0,256,(n,32),dtype=np.uint8); t=rng.integers(0,256,(n,32),dtype=np.uint8)
    for _ in range(50): ctx.match(q,t)
    t0=time.perf_counter()
    for _ in range(3000): ctx.match(q,t)
    print(n,'x',n, round((time.perf_counter()-t0)/3000*1e6,1),'us per hm_match_host call')

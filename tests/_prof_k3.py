import os, sys, time, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from yacht_b200 import _lib, synth
n=int(sys.argv[1]) if len(sys.argv)>1 else 85205
db=synth.make_reference_db(n,3)
ctx=_lib.GpuContext(0)
ctx.load_sketches(db.hashes,db.offsets)
st=ctx.build_index(); print(st)
for ck in (1,2,1,2):
    ctx.set_option("count_kernel",ck); ctx.reset_timers()
    p=ctx.pairwise_flag(0.95**31); print(ck,len(p),ctx.timings()['ms_count'])

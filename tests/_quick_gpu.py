import os, sys, time, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from yacht_b200 import _lib, synth
from oracle import train_oracle as to
ctx=_lib.GpuContext(0)
for n in (2000,10000):
    t=time.time(); db=synth.make_reference_db(n,2); print('gen',n,time.time()-t, 'T',int(db.offsets[-1]))
    for rep in range(3):
        ctx.reset_timers()
        t=time.time(); ctx.load_sketches(db.hashes,db.offsets); t1=time.time(); st=ctx.build_index(); t2=time.time(); p=ctx.pairwise_flag(0.95**31); t3=time.time()
        print(n,'load',t1-t,'index',t2-t1,'pairs',t3-t2,len(p),st, ctx.timings())
    if n==2000:
        ref=to.oracle_train(db.hashes,db.offsets,0.95**31)
        print('match', [(int(a),int(b),int(c)) for a,b,c in zip(p['i'],p['j'],p['count'])]==[(int(a),int(b),int(c)) for a,b,c in zip(ref.pairs['i'],ref.pairs['j'],ref.pairs['count'])])

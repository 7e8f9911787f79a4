"""A/B of the grouping kernel's occupancy variants at full size (run manually on the GPU box)."""
import os, sys, time, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from yacht_b200 import _lib, synth
n = int(sys.argv[1]) if len(sys.argv) > 1 else 85205
db = synth.make_reference_db(n, 3)
ctx = _lib.GpuContext(0)
ctx.load_sketches(db.hashes, db.offsets)
for ctas in (4, 5, 4, 5):
    ctx.set_option("group_ctas", ctas)
    for rep in range(3):
        ctx.reset_timers()
        st = ctx.build_index()
        tm = ctx.timings()
    print(f"group_ctas {ctas}: k2_group2 {tm['ms_group']:.3f} ms, partition {tm['ms_sort']:.3f} ms, index total {tm['ms_index']:.3f} ms, W {st['n_increments']}", flush=True)

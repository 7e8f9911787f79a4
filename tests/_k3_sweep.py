"""K3 accumulator-tile sweep at full size (run manually on the GPU box): narrower column tiles put several (row, tile)
units in flight per SM at the price of re-reading a row's work list once per tile."""
import os, sys, time, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from yacht_b200 import _lib, synth
n = int(sys.argv[1]) if len(sys.argv) > 1 else 85205
db = synth.make_reference_db(n, 3)
ctx = _lib.GpuContext(0)
ctx.load_sketches(db.hashes, db.offsets)
st = ctx.build_index()
ref = None
for tile_w in (0, 43000, 28500, 21500, 14300):
    ctx.set_option("force_tile_w", tile_w)
    for rep in range(3):
        ctx.reset_timers()
        F = ctx.pairwise_flag_device(0.95 ** 31, 0, n)
        ms = ctx.timings()["ms_count"]
    p = ctx.pairs_host(F)
    if ref is None:
        ref = p.tobytes()
    print(f"tile_w {tile_w}: F {F} count kernel {ms:.3f} ms same={p.tobytes() == ref}", flush=True)

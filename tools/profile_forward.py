"""Runs a few forwards of the synthetic checkpoint (for ncu launch lists / captures)."""
import os
import sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ctd_b200
from oracle import synth

bs = int(sys.argv[1]) if len(sys.argv) > 1 else 16
iters = int(sys.argv[2]) if len(sys.argv) > 2 else 2
prec = int(sys.argv[3]) if len(sys.argv) > 3 else 0
ck = synth.make_checkpoint(0, smooth=True)
prog = ctd_b200.compiler.compile_checkpoint(ck, fuse=ctd_b200.compiler.fuse_default(prec == 0))
pages = np.stack([synth.structured_page(1000 + i) for i in range(bs)])
eng = ctd_b200.Engine(prog, precision=prec, max_batch=bs, max_h=1024, max_w=1024)
for it in range(iters):
    eng.forward(pages)
    print("forward ms", eng.last_forward_ms(), flush=True)
# op table for mapping launches to layers
for i, o in enumerate(prog.ops):
    print("op", i, "kind", o["kind"], "k", o["ksize"], "s", o["stride"], "cin", sum(o["src_c"]), "cout", o["cout"], "down", prog.bufs[o["src_buf"][0]][1] if o["n_src"] else 1)
eng.close()

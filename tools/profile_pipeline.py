"""Runs a few FULL-pipeline batches (ctd_submit_full / ctd_collect: network + post-processing + group_output +
refine_mask) of the synthetic checkpoint, one batch at a time (for ncu launch lists / captures)."""
import os
import sys
import numpy as np
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ctd_b200
from oracle import synth

bs = int(sys.argv[1]) if len(sys.argv) > 1 else 16
iters = int(sys.argv[2]) if len(sys.argv) > 2 else 2
ck = synth.make_checkpoint(0, smooth=True)
prog = ctd_b200.compiler.compile_checkpoint(ck, fuse=ctd_b200.compiler.fuse_default(True))
pages = torch.from_numpy(np.stack([synth.structured_page(1000 + i) for i in range(bs)])).pin_memory()
eng = ctd_b200.Engine(prog, max_batch=bs, max_h=1024, max_w=1024)
out = torch.empty((eng.results_layout()["total_bytes"],), dtype=torch.uint8).pin_memory()
import time
for it in range(iters):
    t0 = time.perf_counter()
    eng.submit_full(0, pages.data_ptr(), bs, 1024, 1024, out.data_ptr())
    eng.collect(0)
    print("batch ms", 1e3 * (time.perf_counter() - t0), flush=True)
eng.close()

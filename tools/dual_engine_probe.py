"""Probe: does running two engines (two CUDA graphs on two streams) back to back raise whole-GPU throughput?"""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ctd_b200
from oracle import synth

B = int(sys.argv[1]) if len(sys.argv) > 1 else 16
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 20
ck = synth.make_checkpoint(0, smooth=True)
prog = ctd_b200.compiler.compile_checkpoint(ck)
pages = torch.from_numpy(np.stack([synth.structured_page(1000 + i) for i in range(B)])).cuda()
for n_eng in (1, 2, 3):
    engs = [ctd_b200.Engine(prog, max_batch=B, max_h=1024, max_w=1024) for _ in range(n_eng)]
    for e in engs:
        for _ in range(3):
            e.forward_device(pages.data_ptr(), B, 1024, 1024)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(steps):
        engs[i % n_eng].forward_device(pages.data_ptr(), B, 1024, 1024)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    print("engines %d: %.3f ms/step, %.1f pages/s" % (n_eng, dt / steps * 1e3, B * steps / dt), flush=True)
    for e in engs:
        e.close()

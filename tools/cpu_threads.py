"""How does the reference's CPU forward scale with torch threads on this host? (for bench.py --cpu-threads)"""
import os, sys, time
ROOT =os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch
from oracle import synth
from oracle.net_ref import RefNet
ck = synth.make_checkpoint(0, smooth=True)
net = RefNet(ck)
x = torch.from_numpy(synth.structured_page(1000).transpose(2, 0, 1)[None].astype(np.float32) / 255)
import os
print("cpu_count", os.cpu_count())
for t in (8, 16, 32, 64, 128):
    torch.set_num_threads(t)
    net(x)
    t0 = time.perf_counter(); net(x); dt = time.perf_counter() - t0
    print("threads", t, "forward s", round(dt, 2), flush=True)

"""Net-level error of each engine precision against the fp32 oracle at several page sizes (GPU box)."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import ctd_b200
from oracle import synth
from oracle.net_ref import RefNet
from util import get_checkpoint, page_to_net_input

ck = get_checkpoint(0, True)
prog = ctd_b200.compiler.compile_checkpoint(ck)
ref = RefNet(ck)
for (n, h, w) in [(2, 256, 320), (2, 512, 512), (2, 1024, 1024)]:
    pages = np.stack([synth.structured_page(1000 + i, h, w) if i % 2 == 0 else synth.noise_page(1000 + i, h, w) for i in range(n)])
    with torch.no_grad():
        outs = [ref(page_to_net_input(pages[i:i + 1])) for i in range(n)]
    rb, rm, rl = (torch.cat([o[k] for o in outs]).numpy() for k in range(3))
    for prec, name in ((1, "fp32_simt"), (3, "split_tc")):
        eng = ctd_b200.Engine(prog, precision=prec, max_batch=n, max_h=h, max_w=w)
        try:
            eng.forward(pages)
            blks, mask, lines = eng.net_outputs()
        finally:
            eng.close()
        dm, dl = np.abs(mask - rm), np.abs(lines - rl)
        print("%dx%dx%d %-10s mask max %.3g mean %.3g p99.99 %.3g | lines max %.3g mean %.3g p99.99 %.3g | flips %d"
              % (n, h, w, name, dm.max(), dm.mean(), np.quantile(dm, 0.9999), dl.max(), dl.mean(), np.quantile(dl, 0.9999),
                 int(((lines[:, 0] > 0.3) != (rl[:, 0] > 0.3)).sum())))

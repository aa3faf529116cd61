"""tiny split-fp16 forward (for compute-sanitizer runs)"""
import os
import sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import ctd_b200
from oracle import synth
from util import get_checkpoint
prec = int(sys.argv[1]) if len(sys.argv) > 1 else 3
ck = get_checkpoint(0, True)
prog = ctd_b200.compiler.compile_checkpoint(ck)
size = int(sys.argv[2]) if len(sys.argv) > 2 else 128
n, h, w = 1, size, size
pages = np.stack([synth.structured_page(1000 + i, h, w) for i in range(n)])
eng = ctd_b200.Engine(prog, precision=prec, max_batch=n, max_h=h, max_w=w)
eng.forward(pages)
b, m, l = eng.net_outputs()
print("ok", float(m.mean()), float(l.mean()))
eng.close()

"""cProfile of the drop-in TextDetector.__call__ on synthetic pages (where does the per-page host time go)."""
import cProfile
import pstats
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ctd_b200
from oracle import synth

ck = synth.make_checkpoint(0, smooth=True)
det = ctd_b200.TextDetector(ck, input_size=1024, act="leaky")
pages = [synth.structured_page(1000 + i) for i in range(4)]
det(pages[0].copy())
t0 = time.perf_counter()
for p in pages:
    det(p.copy())
print("s/page", (time.perf_counter() - t0) / len(pages))
pr = cProfile.Profile()
pr.enable()
for p in pages:
    det(p.copy())
pr.disable()
pstats.Stats(pr).sort_stats("cumulative").print_stats(22)
det.close()

"""refine_mask of ONE synthetic page's windows, twice (for ncu captures of refine_kernel)."""
import os
import sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ctd_b200
from ctd_b200.inference import expand_textwindow
from oracle import synth
seed = int(sys.argv[1]) if len(sys.argv) > 1 else 1004
ck = synth.make_checkpoint(0, smooth=True)
det = ctd_b200.TextDetector(ck, input_size=1024, act="leaky")
page = synth.structured_page(seed)
mask, mask_refined, blks = det(page.copy())
wins = np.array([expand_textwindow(page.shape, b.xyxy, 16) for b in blks], np.int32).reshape(-1, 4)
for _ in range(2):
    det.net.refine_mask(page, mask, wins, 0)
print("windows", len(wins))
det.close()

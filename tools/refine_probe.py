"""How long does refine_mask take on the synthetic 1024x1024 pages, and how are the window sizes distributed?
(sizing input for the batched device pipeline; run on the GPU box)"""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ctd_b200
from ctd_b200.inference import expand_textwindow
from oracle import synth

ck = synth.make_checkpoint(0, smooth=True)
det = ctd_b200.TextDetector(ck, input_size=1024, act="leaky")
for seed in range(1000, 1006):
    page = synth.structured_page(seed)
    t0 = time.perf_counter()
    mask, mask_refined, blks = det(page.copy())
    t_call = time.perf_counter() - t0
    wins = np.array([expand_textwindow(page.shape, b.xyxy, 16) for b in blks], np.int32).reshape(-1, 4)
    area = np.maximum(wins[:, 2] - wins[:, 0], 0) * np.maximum(wins[:, 3] - wins[:, 1], 0)
    det.net.refine_mask(page, mask, wins, 0)
    t0 = time.perf_counter()
    for _ in range(5):
        det.net.refine_mask(page, mask, wins, 0)
    t_ref = (time.perf_counter() - t0) / 5
    # the biggest window alone, and everything but the 5 biggest
    order = np.argsort(-area)
    t0 = time.perf_counter()
    det.net.refine_mask(page, mask, wins[order[:1]], 0)
    t_big = time.perf_counter() - t0
    t0 = time.perf_counter()
    det.net.refine_mask(page, mask, wins[order[5:]], 0)
    t_rest = time.perf_counter() - t0
    t0 = time.perf_counter()
    from ctd_b200 import textblock as tb
    print("page %d: call %.1f ms; %d windows, sum area %.2f pages, max %.3f pages, median %d px; refine %.2f ms "
          "(largest alone %.2f ms, all but 5 largest %.2f ms)" % (seed, t_call * 1e3, len(wins), area.sum() / 1024 ** 2,
                                                                  area.max(initial=0) / 1024 ** 2, int(np.median(area)) if len(area) else 0,
                                                                  t_ref * 1e3, t_big * 1e3, t_rest * 1e3))
det.close()

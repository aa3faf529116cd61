"""Per-op device time of the forward with the yolo activations as compiled (SiLU) vs replaced by LeakyReLU (no MUFU):
how much of each layer's time is the SiLU epilogue.  (Experiment only: the LeakyReLU program is not a valid model.)"""
import os
import sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ctd_b200
from ctd_b200 import compiler as cc
from oracle import synth

bs = 16
ck = synth.make_checkpoint(0, smooth=True)
pages = np.stack([synth.structured_page(1000 + i) for i in range(bs)])
res = {}
for name in ("silu", "leaky"):
    prog = cc.compile_checkpoint(ck, fuse=True)
    if name == "leaky":
        for o in prog.ops:
            if o["act"] == cc.ACT_SILU:
                o["act"] = cc.ACT_LEAKY
    eng = ctd_b200.Engine(prog, max_batch=bs, max_h=1024, max_w=1024)
    eng.forward(pages)
    t = None
    for _ in range(3):
        op_ms, _, _ = eng.profile_forward(pages=pages)
        t = op_ms if t is None else np.minimum(t, op_ms)
    res[name] = t
    eng.close()
prog = cc.compile_checkpoint(ck, fuse=True)
tot_s = tot_l = 0.0
for i, o in enumerate(prog.ops):
    if o["act"] == cc.ACT_SILU:
        s, l = 1e3 * res["silu"][i], 1e3 * res["leaky"][i]
        tot_s += s; tot_l += l
        print("op%-3d kind %2d k%d s%d cin %4d cout %4d /%-2d  silu %7.1f us  leaky %7.1f us  diff %6.1f" % (
            i, o["kind"], o["ksize"], o["stride"], sum(o["src_c"]), o["cout"], prog.bufs[o["src_buf"][0]][1], s, l, s - l))
print("SiLU layers: %.1f us with SiLU, %.1f us with LeakyReLU" % (tot_s, tot_l))

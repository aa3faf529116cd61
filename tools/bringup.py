"""GPU bring-up diagnostics (not a test): per-stage error report + timings.  Run under gpurun."""
import os, sys, time
import numpy as np
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ctd_b200
from ctd_b200.binding import PREC_FP16_TC, PREC_FP32_SIMT, PREC_FP16_SIMT
from oracle import synth
from oracle.net_ref import RefNet

def main():
    ck = synth.make_checkpoint(0, smooth=True)
    prog = ctd_b200.compiler.compile_checkpoint(ck)
    n, h, w = 1, 256, 256
    pages = np.stack([synth.structured_page(1000, h, w)])
    ref = RefNet(ck)
    x = torch.from_numpy(np.ascontiguousarray(pages.transpose(0, 3, 1, 2)).astype(np.float32) / 255)
    rb, rm, rl = ref(x)
    feats = {k: v for k, v in zip(("f256", "f128", "f64", "f32", "f3"), ref.last_feats)}
    for prec, name in ((PREC_FP32_SIMT, "fp32_simt"), (PREC_FP16_SIMT, "fp16_simt"), (PREC_FP16_TC, "fp16_tc")):
        try:
            eng = ctd_b200.Engine(prog, precision=prec, max_batch=n, max_h=h, max_w=w)
            eng.forward(pages)
            blks, mask, lines = eng.net_outputs()
            print(name, "mask err %.3g lines err %.3g blks err %.3g" % (np.abs(mask - rm.numpy()).max(), np.abs(lines - rl.numpy()).max(), np.abs(blks - rb.numpy()).max()), flush=True)
            for k, v in feats.items():
                got = eng.debug_read(prog.names[k])
                r = v.permute(0, 2, 3, 1).numpy()
                print("   ", k, "err %.3g (ref max %.3g)" % (np.abs(got - r).max(), np.abs(r).max()), flush=True)
            eng.close()
        except Exception as e:
            print(name, "FAILED:", repr(e), flush=True)
    # timing at 1024
    for prec, name, bs in ((PREC_FP16_TC, "fp16_tc", 1), (PREC_FP16_TC, "fp16_tc", 16), (PREC_FP16_TC, "fp16_tc_graph", 16), (PREC_FP16_SIMT, "fp16_simt", 1), (PREC_FP32_SIMT, "fp32_simt", 1)):
        try:
            pages = np.stack([synth.structured_page(1000 + i) for i in range(bs)])
            eng = ctd_b200.Engine(prog, precision=prec, max_batch=bs, max_h=1024, max_w=1024, use_graph=name.endswith("graph"))
            ts = []
            for it in range(5):
                eng.forward(pages)
                ts.append(eng.last_forward_ms())
            print(name, "bs", bs, "forward ms (incl H2D):", ["%.2f" % t for t in ts], "launches", eng.last_launch_count(), flush=True)
            eng.close()
        except Exception as e:
            print(name, "timing FAILED:", repr(e), flush=True)

if __name__ == "__main__":
    main()

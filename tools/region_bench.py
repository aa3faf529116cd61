"""OCR line crops (`TextDetector.get_transformed_regions` / ctd_transform_regions) against the reference's per-line cv2 loop
(oracle/regions_ref.py: findHomography + warpPerspective per line, as utils/textblock.py:162-194 does).

Synthetic 1024x1024 pages go through a real TextDetector first; every line of every block is then cropped at
textheight 48.  Prints one JSON line:
  gpu_host      lines/s and ms per page of the call with a HOST page in and HOST crops out (upload, two kernels, download)
  gpu_device    the same with the page already in HBM and the crops left there
  cv2_loop      the reference's loop on the host cores (cv2 thread count stated)
  k_region_warp kernel time from torch.profiler (CUDA activities, separate pass) and GB/s over the bytes the algorithm must
                move: the crops written plus the page read once (an upper bound on the page bytes a crop set needs)
Usage: python tools/region_bench.py [--pages 8] [--reps 20] [--out FILE]"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pages", type=int, default=8)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--textheight", type=float, default=48)
    ap.add_argument("--cv2-threads", type=int, default=-1, help="cv2.setNumThreads value (-1: OpenCV's default)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import cv2
    import torch
    import ctd_b200
    from ctd_b200 import binding
    from oracle import regions_ref, synth

    if not torch.cuda.is_available():
        raise SystemExit("region_bench needs a GPU")
    det = ctd_b200.TextDetector(synth.make_checkpoint(0, smooth=True), input_size=1024, act="leaky")
    pages, blks = [], []
    for i in range(a.pages):
        p = synth.structured_page(2000 + i, 1024, 1024)
        pages.append(p)
        blks.append(det(p.copy())[2])
    n_lines = sum(len(b.lines) for bl in blks for b in bl)
    th = a.textheight

    def args_of(bl):
        items = [(b, i) for b in bl for i in range(len(b.lines))]
        q = np.array([np.asarray(b.lines[i], np.float64) for b, i in items]).reshape(-1, 4, 2)
        f = np.array([(binding.REGION_EXPAND if regions_ref.expands(b.language, b.vertical) else 0)
                      | (binding.REGION_VERTICAL if b.vertical else 0) for b, _ in items], np.int32)
        fs = np.array([b.font_size for b, _ in items], np.float64)
        return q, f, fs
    args = [args_of(bl) for bl in blks]

    # (a) host page in, host crops out: the public method
    for p, bl in zip(pages, blks):
        det.get_transformed_regions(p, bl, th)
    t0 = time.perf_counter()
    for _ in range(a.reps):
        for p, bl in zip(pages, blks):
            det.get_transformed_regions(p, bl, th)
    t_host = (time.perf_counter() - t0) / a.reps

    # (b) page resident in HBM, crops kept there
    dev_pages = [torch.from_numpy(p).cuda() for p in pages]
    totals = [binding.plan_regions(q, f, fs, 1024, 1024, 3, th)[1] for q, f, fs in args]
    dev_out = torch.empty(max(totals) + 1, dtype=torch.uint8, device="cuda")

    def dev_call(k):
        q, f, fs = args[k]
        det.net.transform_regions(None, q, f, fs, th, img_dev=(dev_pages[k].data_ptr(), 1024, 1024, 3),
                                  out_dev=dev_out.data_ptr(), out_bytes=dev_out.numel())
    for k in range(a.pages):
        dev_call(k)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(a.reps):
        for k in range(a.pages):
            dev_call(k)       # blocking: the call synchronises the engine stream
    t_dev = (time.perf_counter() - t0) / a.reps

    # the reference's loop with cv2 on the host cores
    if a.cv2_threads >= 0:
        cv2.setNumThreads(a.cv2_threads)
    cv_reps = max(1, a.reps // 10)
    t0 = time.perf_counter()
    for _ in range(cv_reps):
        for p, bl in zip(pages, blks):
            regions_ref.transformed_regions(p, bl, th)
    t_cv = (time.perf_counter() - t0) / cv_reps

    # kernel time of k_region_warp / k_region_homography (profiled pass, not part of the timings above)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for k in range(a.pages):
            dev_call(k)
        torch.cuda.synchronize()
    kern = {}
    for k in prof.key_averages():
        for name in ("k_region_warp", "k_region_homography"):
            if name in k.key:
                kern[name] = kern.get(name, 0.0) + k.device_time_total
    crop_bytes = int(sum(totals))
    warp_bytes = crop_bytes + a.pages * 1024 * 1024 * 3
    warp_us = kern.get("k_region_warp", 0.0)
    props = torch.cuda.get_device_properties(0)
    try:
        import subprocess
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                               text=True, timeout=30).stdout.strip()
    except Exception:
        power = "unknown"
    res = {
        "what": "TextBlock.get_transformed_region for every line of %d synthetic 1024x1024 pages (TextDetector output), "
                "textheight %g" % (a.pages, th),
        "gpu": props.name, "power_limit": power, "pages": a.pages, "lines": n_lines,
        "lines_per_page": n_lines / a.pages,
        "gpu_host": {"lines_per_s": n_lines / t_host, "ms_per_page": 1e3 * t_host / a.pages},
        "gpu_device": {"lines_per_s": n_lines / t_dev, "ms_per_page": 1e3 * t_dev / a.pages},
        "cv2_loop": {"lines_per_s": n_lines / t_cv, "ms_per_page": 1e3 * t_cv / a.pages, "cv2_threads": cv2.getNumThreads(),
                     "host_cpus": os.cpu_count()},
        "k_region_warp": {"launches": a.pages, "us_total": warp_us, "crop_bytes": crop_bytes, "bytes": warp_bytes,
                          "GBps": warp_bytes / (warp_us * 1e-6) / 1e9 if warp_us else None},
        "k_region_homography_us_total": kern.get("k_region_homography"),
    }
    det.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py -- pages/sec of the comic-text-detector hot path on N B200s (driver contract).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--batch B]

A "step" = one pass of the WHOLE hot path -- everything `TextDetector.__call__` does (reference
inference.py:141-178): backbone + seg head + DB head + Detect decode + NMS + mask u8 + DB threshold + connected
components + text-line boxes/scores (device, one CUDA graph), postprocess_yolo casts + box_thresh + group_output
(host C++, the engine's worker thread), refine_mask (device, on the resident pages) -- over one batch of B
synthetic 1024x1024 pages per GPU (BASELINE.json configs[2]/[3]: batch 16 per GPU, fp16 tcgen05 path).

* value      : whole-job pages/s with the pages already resident in HBM (ctd_submit_full with pages_on_device);
               --engines E (default 2) workspaces per GPU x two batches in flight each; timed with CUDA events on
               engine 0's stream around a host-drained region, max over ranks.
* e2e        : the same call with HOST (pinned) page buffers: H2D of the pages and D2H of the complete results
               (mask u8, detections, line boxes/scores, counts, mask_refined, block records) of EVERY step inside the
               timed region; at N > 1 also the NCCL gather of every rank's result arena to rank 0 and rank 0's D2H of
               the gathered arenas.
* net_only   : the round-1 step (network + NMS + CCL + line boxes, no group_output / refine_mask), for comparison.
* roofline   : tensor roofline of the tcgen05 convolution kernels: algorithmic conv FLOPs / summed device time of
               the conv launches (per-op CUDA events, serial order, each kernel timed ALONE at boost clocks ->
               MEASURED_PEAKS.json bf16_tflops, the burst figure); `whole_step_frac` divides the algorithmic FLOPs
               by the whole timed net_only step against the same peak.
* config2 / config5 / api_e2e : BASELINE configs[1] (batch 1, fp32-accurate engines) and configs[4] (mixed
               640/1024/1536 stream) and the drop-in Python class, measured on rank 0 at N = 1.
* cpu_baseline / --impl reference: the oracle restatement of the reference's CPU path for the SAME stages
               (oracle/net_ref.py + oracle/postproc_ref.py + oracle/textblock_ref.py + oracle/pipeline_ref.py: torch
               CPU fp32 + torchvision + cv2 + numpy, i.e. the reference's own library calls) on this box's host cores.

--dump-outputs DIR writes what the last timed step of `value` returned for rank 0's batch as DIR/<name>.npy (see
step_outputs), so that two builds run with the same arguments, hence the same pages and checkpoint, can be compared
output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GFLOP_PER_PAGE_1024 = 191.414  # BASELINE.md section 2 (2*MAC over the 115 conv/deconv layers)


def conv_flops(prog, n, h, w):
    """Algorithmic FLOPs of each op of the program at batch n (0 for non-conv ops)."""
    out = []
    for o in prog.ops:
        kind = o["kind"]
        if kind == 0:  # stem: 6x6 s2 conv 3 -> cout (algorithmic FLOPs, not the zero-padded tensor-core K)
            out.append(2.0 * (h // 2) * (w // 2) * n * 108 * o["cout"])
            continue
        if kind == 10:  # fused Bottleneck: 1x1 c -> c plus 3x3 c -> c on the same pixels
            down = prog.bufs[o["src_buf"][0]][1]
            out.append(2.0 * (h // down) * (w // down) * n * 10 * o["cout"] * o["cout"])
            continue
        if kind not in (1, 2, 6, 7):
            out.append(0.0)
            continue
        down = prog.bufs[o["src_buf"][0]][1]
        px = (h // down) * (w // down) * n
        cin = sum(o["src_c"][: o["n_src"]])
        if kind == 7:   # seg tail: ConvT 4x4 s2, C -> 1 (16 taps per input pixel)
            out.append(2.0 * px * 16 * cin)
        elif kind == 2:
            out.append(2.0 * px * 16 * cin * o["cout"])
        else:
            k, s = o["ksize"], o["stride"]
            out.append(2.0 * (px // (s * s)) * k * k * cin * o["cout"])
    return out


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._halt = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for nm, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(nm)
            except Exception:
                pass
            self._halt.wait(0.1)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def cpu_pipeline_factory():
    """The reference's CPU path for the same stages (network .. refine_mask), via the oracle restatement."""
    import torch
    from oracle import synth, pipeline_ref, textblock_ref
    from oracle.net_ref import RefNet
    ck = synth.make_checkpoint(0, smooth=True)
    net = RefNet(ck)

    def run(page_u8):
        x = torch.from_numpy(np.ascontiguousarray(page_u8.transpose(2, 0, 1))[None].astype(np.float32) / 255)
        with torch.no_grad():
            blks, mask, lines = net(x)
        return pipeline_ref.postprocess_page(page_u8, blks[0].numpy(), mask[0, 0].numpy(), lines[0].numpy(),
                                             textblock_ref.group_output, refine_mode=0)
    return run


CPU_WORKLOAD = ("reference CPU path, same stages as the GPU step (oracle port: torch CPU fp32 forward + torchvision NMS + "
                "cv2 CC / findContours / minAreaRect + group_output + refine_mask)")


def run_reference(args):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import synth
    cores = min(os.cpu_count(), args.cpu_threads)
    torch.set_num_threads(cores)
    run = cpu_pipeline_factory()
    pages = [synth.structured_page(1000 + i) for i in range(max(1, args.cpu_pages))]
    for _ in range(min(args.warmup, 2)):
        run(pages[0])
    t0 = time.perf_counter()
    for k in range(args.steps):
        for p in pages:
            run(p)
    dt = time.perf_counter() - t0
    npages = args.steps * len(pages)
    val = npages / dt
    print(json.dumps({
        "impl": "reference", "metric": "pages/sec @1024x1024 synthetic", "value": val, "unit": "pages/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": CPU_WORKLOAD + ", %d page(s) of 1024x1024 per step, %d host threads" % (len(pages), cores)},
        "cpu_baseline": {"value": val, "unit": "pages/s", "cores": cores, "kind": "port",
                         "sample": "%d steps x %d structured synthetic 1024x1024 page(s)" % (args.steps, len(pages))},
        "e2e": {"value": val, "unit": "pages/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


DUMP_MASK_PIXELS = 1 << 22   # pixels kept of each batch-sized mask: 16 MB as float32 (a quarter of 16 pages of 1024^2)


def step_outputs(arena, lay, n, h, w):
    """The results a caller of the full-pipeline step receives for its batch of n pages (unpacked from the result
    arena) as float32 / float64 arrays, one row per item, column 0 the page index:
      mask_sample, mask_refined_sample  u8 masks at the same DUMP_MASK_PIXELS flat positions of the [n][h][w] batch,
                                        np.random.default_rng(0).choice(n*h*w, DUMP_MASK_PIXELS, replace=False), sorted
      det          page, x1, y1, x2, y2, conf, cls                  line_boxes   page, x1, y1, .. x4, y4
      line_scores  one per line_boxes row                           n_labels / block_flags   one per page
      blocks       page, x1, y1, x2, y2, language (LANGCLS2IDX), vertical, font_size, angle, vec x, vec y, norm,
                   merged, weight, number of lines
      block_lines  page, block, x1, y1, .. x4, y4
      block_distances  page, block, distance, is_nan: a distance is NaN where the block's reading direction is degenerate
                   (examine_textblk's arccos of 0/0, as in the reference); such rows hold distance 0 and is_nan 1 so that
                   every value written is finite"""
    from ctd_b200 import multigpu
    from ctd_b200.textblock import LANGCLS2IDX
    r = multigpu.unpack_arena(arena, lay, n, h, w, full=True)
    px = np.sort(np.random.default_rng(0).choice(n * h * w, min(DUMP_MASK_PIXELS, n * h * w), replace=False))

    def per_page(arrays, width, dtype):
        return np.concatenate([np.concatenate([np.full((len(a), 1), i), np.reshape(a, (len(a), width - 1))], 1).astype(dtype)
                               for i, a in enumerate(arrays)])

    blocks, lines, dists = [], [], []
    for i, page in enumerate(r["blocks"]):
        for j, b in enumerate(page):
            blocks.append([i, *b.xyxy, LANGCLS2IDX[b.language], b.vertical, b.font_size, b.angle, *b.vec, b.norm, b.merged,
                           b.weight, len(b.lines)])
            lines += [[i, j, *np.ravel(q)] for q in b.lines]
            dists += [[i, j, 0.0, 1.0] if np.isnan(d) else [i, j, d, 0.0] for d in np.ravel(b.distance)]
    return {"mask_sample": r["mask"].reshape(-1)[px].astype(np.float32),
            "mask_refined_sample": r["mask_refined"].reshape(-1)[px].astype(np.float32),
            "det": per_page(r["det"], 7, np.float32),
            "line_boxes": per_page(r["line_boxes"], 9, np.float32),
            "line_scores": np.concatenate(r["line_scores"]).astype(np.float32),
            "n_labels": r["n_labels"].astype(np.float64),
            "block_flags": np.array(r["block_flags"], np.float64),
            "blocks": np.array(blocks, np.float64).reshape(-1, 15),
            "block_lines": np.array(lines, np.float64).reshape(-1, 10),
            "block_distances": np.array(dists, np.float64).reshape(-1, 4)}


class _DevArr:
    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--batch", type=int, default=16, help="pages per GPU per step")
    ap.add_argument("--cpu-pages", type=int, default=1, help="pages per step of the CPU arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip config2 / config5 / api_e2e")
    ap.add_argument("--engines", type=int, default=2, help="workspaces per GPU; consecutive batches alternate between them")
    ap.add_argument("--sustain-steps", type=int, default=150, help="steps of the seconds-long sustained measurement (0 = skip)")
    ap.add_argument("--api-pages", type=int, default=8, help="pages timed through the TextDetector Python API (0 = skip)")
    ap.add_argument("--cpu-threads", type=int, default=16,
                    help="torch intra-op threads of the CPU arm (measured on the B200 host: 16 threads 0.25 s/forward, "
                         "64 threads 0.48 s, 128 threads 33 s -- more threads only hurt)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed for rank 0's pages as DIR/<name>.npy (see step_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import ctd_b200
    from ctd_b200 import multigpu
    from oracle import synth  # synthetic checkpoint + pages only (no oracle compute on this path)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    B, H, W = args.batch, 1024, 1024
    warm = max(3, args.warmup)

    ck = synth.make_checkpoint(0, smooth=True)
    prog = ctd_b200.compiler.compile_checkpoint(ck, fuse=ctd_b200.compiler.fuse_default(True))
    n_eng = max(1, args.engines)
    engs = [ctd_b200.Engine(prog, device=local, max_batch=B, max_h=H, max_w=W, use_graph=True) for _ in range(n_eng)]
    eng = engs[0]
    lay = eng.results_layout()
    res_bytes = lay["total_bytes"]

    def make_pages(r):
        return np.stack([synth.structured_page(1000 + r * B + i) for i in range(B)])
    pages = make_pages(rank)
    host_pages = torch.from_numpy(pages).pin_memory()
    dev_pages = host_pages.cuda()
    torch.cuda.synchronize()
    out_arena = [[torch.empty((res_bytes,), dtype=torch.uint8).pin_memory() for _ in range(2)] for _ in range(n_eng)]
    used_bytes = lay["phase_a_bytes"] + B * H * W + B * lay["blocks_stride"]   # what a step really moves D2H

    # ---- the step: full pipeline, n_eng engines x 2 slots in flight -------------------------------------------
    state = {"k": 0, "on_device": True}
    pending = []
    gathered = {}
    if world > 1:
        # one NCCL gather of each rank's COMPLETE device result arena (mask u8 | detections | lines | mask_refined |
        # block records) to rank 0 per step, then rank 0's D2H of the gathered arenas
        for ei, e in enumerate(engs):
            for slot in range(2):
                e.submit_full(slot, dev_pages.data_ptr(), B, H, W, out_arena[ei][slot].data_ptr(), pages_on_device=True)
                e.collect(slot)
                base, _st = e.device_arena(slot)
                res_t = torch.as_tensor(_DevArr(base, res_bytes), device="cuda")
                glist = [torch.empty_like(res_t) for _ in range(world)] if rank == 0 else None
                ghost = [torch.empty((res_bytes,), dtype=torch.uint8).pin_memory() for _ in range(world)] if rank == 0 else None
                gathered[(ei, slot)] = (res_t, glist, ghost)
    gstream = torch.cuda.Stream() if world > 1 else None
    gather_done = {}

    def finish(ei, slot):
        engs[ei].collect(slot)
        if world > 1:
            res_t, glist, ghost = gathered[(ei, slot)]
            with torch.cuda.stream(gstream):
                dist.gather(res_t, gather_list=glist, dst=0)
                ev = torch.cuda.Event()
                ev.record(gstream)          # the slot's device arena may be overwritten once the gather has read it
                gather_done[(ei, slot)] = ev
                if rank == 0 and not state["on_device"]:
                    for g, hbuf in zip(glist, ghost):
                        hbuf.copy_(g, non_blocking=True)

    def step_full():
        k = state["k"]
        state["k"] += 1
        ei, slot = k % n_eng, (k // n_eng) & 1
        if len(pending) == 2 * n_eng:
            finish(*pending.pop(0))
        if (ei, slot) in gather_done:
            gather_done.pop((ei, slot)).synchronize()
        src = dev_pages.data_ptr() if state["on_device"] else host_pages.data_ptr()
        engs[ei].submit_full(slot, src, B, H, W, out_arena[ei][slot].data_ptr(), pages_on_device=state["on_device"])
        pending.append((ei, slot))

    def drain_full():
        while pending:
            finish(*pending.pop(0))
        if gstream is not None:
            gstream.synchronize()

    ctr = {"res": 0}

    def step_net_only():
        e = engs[ctr["res"] % n_eng]
        ctr["res"] += 1
        e.forward_device(dev_pages.data_ptr(), B, H, W)

    def join_all():
        for e in engs[1:]:
            eng.join(e)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, drain=None):
        barrier()
        eng.timer_start()
        for _ in range(steps):
            fn()
        if drain is not None:
            drain()  # host-blocks until the last results landed, so the stop event is recorded after them
        join_all()   # the other engines' streams become dependencies of the timer stream
        ms = eng.timer_stop()
        barrier()
        if dist is not None:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    state["on_device"] = True
    for _ in range(warm * n_eng):
        step_full()
    drain_full()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms = timed(step_full, args.steps, drain_full)
    clocks = sampler.stop() if sampler else None
    dump = None
    if args.dump_outputs and rank == 0:
        k = state["k"] - 1   # the last timed step; its host arena is reused by the steps below
        dump = step_outputs(out_arena[k % n_eng][(k // n_eng) & 1].numpy(), lay, B, H, W)
    state["on_device"] = False
    for _ in range(2 * n_eng):
        step_full()
    drain_full()
    ms_e2e = timed(step_full, args.steps, drain_full)
    for _ in range(warm * n_eng):
        step_net_only()
    ms_net = timed(step_net_only, args.steps)
    # the same full-pipeline step over a seconds-long region (VERDICT r1 #11: the headline region is ~0.2 s at boost clocks)
    sustained = None
    if world == 1 and args.sustain_steps > 0:
        state["on_device"] = True
        for _ in range(2 * n_eng):
            step_full()
        drain_full()
        s2 = ClockSampler(local)
        s2.start()
        ms_sus = timed(step_full, args.sustain_steps, drain_full)
        c2 = s2.stop()
        sustained = {"steps": args.sustain_steps, "seconds": ms_sus * 1e-3, "value": B * args.sustain_steps / (ms_sus * 1e-3),
                     "unit": "pages/s", "clocks": c2,
                     "what": "the headline step (pages resident) repeated over a seconds-long timed region"}

    # ---- multi-GPU correctness: rank 0 re-runs every rank's pages locally and compares the gathered arenas ------
    mg_check = None
    if world > 1:
        state["on_device"] = False
        step_full()
        drain_full()
        barrier()
        if rank == 0:
            ei, slot = (state["k"] - 1) % n_eng, ((state["k"] - 1) // n_eng) & 1
            _res_t, _glist, ghost = gathered[(ei, slot)]
            same, npages_checked = True, 0
            chk = torch.empty((res_bytes,), dtype=torch.uint8).pin_memory()
            for r in range(world):
                pr = torch.from_numpy(make_pages(r)).pin_memory()
                eng.submit_full(0, pr.data_ptr(), B, H, W, chk.data_ptr())
                eng.collect(0)
                a = multigpu.unpack_arena(chk.numpy(), lay, B, H, W, full=True)
                g = multigpu.unpack_arena(ghost[r].numpy(), lay, B, H, W, full=True)
                ok = np.array_equal(a["mask"], g["mask"]) and np.array_equal(a["mask_refined"], g["mask_refined"])
                for i in range(B):
                    ok = ok and np.array_equal(a["det"][i], g["det"][i]) and np.array_equal(a["line_boxes"][i], g["line_boxes"][i])
                    ok = ok and np.array_equal(a["line_scores"][i], g["line_scores"][i])
                    ok = ok and [(b.xyxy, b.lines, b.language, b.vertical, b.angle) for b in a["blocks"][i]] == \
                        [(b.xyxy, b.lines, b.language, b.vertical, b.angle) for b in g["blocks"][i]]
                same = same and bool(ok)
                npages_checked += B
            mg_check = {"ranks": world, "pages": npages_checked, "identical_to_single_gpu": same,
                        "what": "rank 0 re-ran every rank's pages on its own GPU and compared the gathered result arenas "
                                "(mask u8, mask_refined, detections, line boxes/scores, blocks) byte for byte"}
        barrier()

    # per-op device times of one forward -> roofline of the tensor-core conv kernels
    op_ms, nms_ms, ccl_ms = eng.profile_forward(dev_ptr=dev_pages.data_ptr(), shape=(B, H, W))
    op_ms2, _, _ = eng.profile_forward(dev_ptr=dev_pages.data_ptr(), shape=(B, H, W))
    op_ms = np.minimum(op_ms, op_ms2)
    fl = conv_flops(prog, B, H, W)
    tc_idx = [i for i, o in enumerate(prog.ops) if o["kind"] in (0, 1, 2, 6, 7, 10)]
    tc_ms = float(sum(op_ms[i] for i in tc_idx))
    tc_flops = float(sum(fl[i] for i in tc_idx))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    # each conv kernel is timed ALONE between events (sub-millisecond bursts at boost clock) -> burst peak
    peak_tf = float(peaks.get("bf16_tflops", 1676.8))
    peak_src = ("MEASURED_PEAKS.json bf16_tflops (burst: kernels timed in isolation)" if peaks
                else "fallback 1676.8 TFLOP/s burst (B200_PROFILING.md)")
    achieved = tc_flops / (tc_ms * 1e-3) / 1e12 if tc_ms > 0 else 0.0
    traffic, traffic_src = None, None
    for name in ("r02_conv_traffic.json", "r01_conv_traffic.json"):
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", name)))
            if int(tj.get("batch", 0)) == B:
                traffic = float(tj["dram_bytes"])
                traffic_src = "profiles/%s (ncu dram__bytes_read.sum + dram__bytes_write.sum over the %d conv launches of one step)" % (name, int(tj["launches"]))
                break
        except Exception:
            pass

    if rank == 0:
        total_pages = B * world * args.steps
        value = total_pages / (ms * 1e-3)
        e2e_val = total_pages / (ms_e2e * 1e-3)
        net_val = total_pages / (ms_net * 1e-3)
        d2h = int(used_bytes) + (int(world * res_bytes) if world > 1 else 0)
        line = {
            "metric": "pages/sec @1024x1024 synthetic", "value": value, "unit": "pages/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp16",
            "data": "synthetic",
            "config": {"workload": "BASELINE configs[2]: 1024x1024 pages, batch %d per GPU, fp16 tcgen05 path, FULL pipeline of "
                                   "TextDetector.__call__ (backbone + seg head + DB head + Detect/NMS + mask u8 + DB threshold + CCL + "
                                   "contour boxes/scores on the device, group_output in host C++, refine_mask on the device)" % B,
                       "pages_per_gpu_per_step": B, "page": [H, W], "checkpoint": "synthetic seed 0 (oracle/synth.py)",
                       "l2": "activations per step (~%.1f GB) exceed the 126 MB L2; no explicit flush" % (
                           sum(c * (H // d) * (W // d) for c, d in prog.bufs) * 2 * B / 1e9),
                       "cuda_graph": True, "engines_per_gpu": n_eng,
                       "fused_ops": "5 fused Bottleneck kernels + seg tail as GEMM + col2im (bit-identical / fp32-rounding-equal to the unfused program)",
                       "in_flight": "%d batches per GPU (%d workspaces x 2 slots)" % (2 * n_eng, n_eng),
                       "multi_gpu": ("pages sharded B per rank; one NCCL gather of each rank's complete result arena to rank 0 per step"
                                     if world > 1 else "single GPU")},
            # forward graph (convs + thin ops + NMS / CCL / contour kernels) + copies + the 29 refine_mask launches of a batch
            "gpu_launches": (eng.last_launch_count() + 6 + 29) * args.steps,
            "clocks": clocks,
            "conv_roofline_frac_of_nominal": net_val / world * GFLOP_PER_PAGE_1024 * 1e9 / 2.25e15,
            "e2e": {"value": e2e_val, "unit": "pages/s", "h2d_bytes_per_step": int(B * H * W * 3), "d2h_bytes_per_step": d2h,
                    "mode": "ctd_submit_full/ctd_collect on %d engine(s) per GPU, two batches in flight per engine, pinned host buffers%s"
                            % (n_eng, "; + NCCL gather of all ranks' arenas and rank 0's D2H of them" if world > 1 else "")},
            "net_only": {"value": net_val, "unit": "pages/s", "ms_per_step": ms_net / args.steps,
                         "what": "round-1 step: network + NMS + CCL + line boxes only (ctd_forward on resident pages), no group_output / refine_mask"},
            "roofline": {"bound": "tensor", "kernel": "conv_tc / conv_halo / conv_hs / conv_sw / conv_bneck kernels, the tcgen05 implicit-GEMM convolutions (%d launches per step)" % len(tc_idx),
                         "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                         "traffic": traffic, "traffic_unit": "bytes/step", "traffic_source": traffic_src,
                         "peak_source": peak_src, "flops_per_step": tc_flops, "ms_per_step": tc_ms,
                         "share_of_step": tc_ms / float(op_ms.sum() + nms_ms + ccl_ms),
                         "whole_step_frac": (GFLOP_PER_PAGE_1024 * 1e9 * B) / (ms_net / args.steps * 1e-3) / 1e12 / peak_tf,
                         "whole_step_what": "algorithmic conv FLOPs of a batch / the net_only step time (all kernels, 2 workspaces overlapped), same peak"},
            "stage_ms": {"conv_tc": tc_ms, "other_ops": float(op_ms.sum()) - tc_ms, "nms": nms_ms, "ccl_and_line_boxes": ccl_ms,
                         "group_output_and_refine_mask_per_step": ms / args.steps - ms_net / args.steps},
        }
        if sustained is not None:
            line["sustained"] = sustained
        if mg_check is not None:
            line["multi_gpu_check"] = mg_check
        if world == 1 and not args.no_extras:
            extras(line, args, ck, prog, pages, local)
        if not args.no_cpu_baseline and world == 1:
            cores = min(os.cpu_count(), args.cpu_threads)
            torch.set_num_threads(cores)
            run = cpu_pipeline_factory()
            run(pages[0])
            t0 = time.perf_counter()
            ncpu = 4
            for i in range(ncpu):
                run(pages[i % B])
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": ncpu / dt, "unit": "pages/s", "cores": cores, "kind": "port",
                                    "sample": "%d structured synthetic 1024x1024 pages; %s" % (ncpu, CPU_WORKLOAD)}
        print(json.dumps(line))
    if dump is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    for e in engs:
        e.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def extras(line, args, ck, prog, pages, local):
    """BASELINE configs[1] (batch 1, vs reference fp32), configs[4] (mixed-resolution stream) and the drop-in class."""
    import torch
    import ctd_b200
    from ctd_b200.binding import PREC_FP16_TC, PREC_FP32_SIMT, PREC_SPLIT_TC
    B = pages.shape[0]
    # config 2: single page, full pipeline through the drop-in call, per precision
    c2 = {}
    for name, prec in (("split_tc", PREC_SPLIT_TC), ("fp32_simt", PREC_FP32_SIMT), ("fp16_tc", PREC_FP16_TC)):
        try:
            det = ctd_b200.TextDetector(ck, input_size=1024, act="leaky", precision=prec, device_index=local)
            det(pages[0].copy())
            n = max(1, args.api_pages)
            t0 = time.perf_counter()
            nblk = 0
            for i in range(n):
                _m, _r, bl = det(pages[i % B])
                nblk += len(bl)
            dt = time.perf_counter() - t0
            fwd = []
            for _ in range(3):
                det.net.forward(pages[:1])
                fwd.append(det.net.last_forward_ms())
            fwd_ms = min(fwd)
            det.close()
            c2[name] = {"pages_per_s": n / dt, "ms_per_page": 1e3 * dt / n, "forward_ms": fwd_ms, "blocks_per_page": nblk / n}
        except Exception as ex:   # a precision mode that fails must not take the headline down with it
            c2[name] = {"error": str(ex)[:200]}
    line["config2"] = {"workload": "BASELINE configs[1]: one 1024x1024 page per call, full pipeline (TextDetector.__call__), "
                                   "per engine precision; split_tc / fp32_simt meet the 1e-3 tolerance vs the fp32 reference",
                       **c2}
    if "fp16_tc" in c2 and "pages_per_s" in c2["fp16_tc"]:
        line["api_e2e"] = {"value": c2["fp16_tc"]["pages_per_s"], "unit": "pages/s", "pages": max(1, args.api_pages),
                           "blocks_per_page": c2["fp16_tc"]["blocks_per_page"],
                           "what": "TextDetector.__call__ per page (one native ctd_detect_page call), single stream, blocking"}
    # config 5: mixed-resolution stream, batch 8 per GPU, per-shape plans + CUDA graphs (built on first use)
    try:
        from oracle import synth
        Bm = 8
        sizes = [640, 1024, 1536]
        e5 = ctd_b200.Engine(prog, device=local, max_batch=Bm, max_h=1536, max_w=1536, use_graph=True)
        lay5 = e5.results_layout()
        bufs = {s: torch.from_numpy(np.stack([synth.structured_page(500 + i, s, s) for i in range(Bm)])).pin_memory() for s in sizes}
        outs = [torch.empty((lay5["total_bytes"],), dtype=torch.uint8).pin_memory() for _ in range(2)]
        order = [sizes[i % 3] for i in range(12)]
        for s in sizes:   # builds plans + graphs
            e5.submit_full(0, bufs[s].data_ptr(), Bm, s, s, outs[0].data_ptr())
            e5.collect(0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pend = []
        for k, s in enumerate(order):
            if len(pend) == 2:
                e5.collect(pend.pop(0))
            e5.submit_full(k & 1, bufs[s].data_ptr(), Bm, s, s, outs[k & 1].data_ptr())
            pend.append(k & 1)
        while pend:
            e5.collect(pend.pop(0))
        dt = time.perf_counter() - t0
        e5.close()
        mpix = sum(Bm * s * s for s in order) / 1e6
        line["config5"] = {"workload": "BASELINE configs[4]: mixed-resolution stream %s, batch %d per GPU, one engine sized for 1536x1536, "
                                       "per-shape launch plans (tensor maps / tile counts) and CUDA graphs cached" % (sizes, Bm),
                           "pages_per_s": len(order) * Bm / dt, "megapixels_per_s": mpix / dt, "batches": len(order)}
    except Exception as ex:
        line["config5"] = {"error": str(ex)[:200]}


if __name__ == "__main__":
    main()

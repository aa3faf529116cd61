"""not-gpu: the driver-facing contract of bench.py that can be exercised without a GPU -- the reference arm
(`--impl reference`: oracle port of the reference's CPU path) prints ONE JSON line with the agreed keys."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1",
                          "--warmup", "0", "--cpu-threads", "8"], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"].startswith("pages/sec") and d["unit"] == "pages/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["value"] > 0 and abs(d["value"] - 1000.0 / d["ms_per_step"]) / d["value"] < 0.05
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "pages/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def _synthetic_arena(n, h, w):
    """a complete result arena (ctd_submit_full layout, offsets chosen here) of n pages: page i has i + 1 detections,
    one text line, and one block with two lines and three distances, the second NaN"""
    import numpy as np
    from ctd_b200 import multigpu
    from ctd_b200.binding import BLOCK_DTYPE, MAX_BLOCKS, MAX_BLOCK_DIST
    lay = dict(multigpu.arena_layout(n, h, w), blk_records_off=256)
    lay["mask_refined"] = lay["phase_a_bytes"]
    lay["blocks"] = lay["mask_refined"] + n * h * w
    lay["blk_lines_off"] = lay["blk_records_off"] + MAX_BLOCKS * BLOCK_DTYPE.itemsize
    lay["blk_dist_off"] = lay["blk_lines_off"] + MAX_BLOCKS * 32
    lay["blocks_stride"] = lay["blk_dist_off"] + MAX_BLOCK_DIST * 8
    a = np.zeros(lay["blocks"] + n * lay["blocks_stride"], np.uint8)
    a[:n * h * w] = np.arange(n * h * w) % 251
    a[lay["mask_refined"]:lay["mask_refined"] + n * h * w] = np.arange(n * h * w) % 7
    for i in range(n):
        a[lay["det"]:lay["det"] + n * 300 * 24].view(np.float32).reshape(n, 300, 6)[i, :i + 1] = i + 0.5
        a[lay["det_count"]:lay["det_count"] + 4 * n].view(np.int32)[i] = i + 1
        a[lay["line_boxes"]:lay["line_boxes"] + n * 16000].view(np.int16).reshape(n, 1000, 8)[i, 0] = np.arange(8) + i
        a[lay["line_scores"]:lay["line_scores"] + n * 4000].view(np.float32).reshape(n, 1000)[i, 0] = 0.75
        a[lay["line_count"]:lay["line_count"] + 4 * n].view(np.int32)[i] = 1
        sec = a[lay["blocks"] + i * lay["blocks_stride"]:lay["blocks"] + (i + 1) * lay["blocks_stride"]]
        sec[:16].view(np.int32)[:] = [1, 0, 0, 0]
        rec = sec[lay["blk_records_off"]:lay["blk_records_off"] + BLOCK_DTYPE.itemsize].view(BLOCK_DTYPE)
        rec["xyxy"], rec["language"], rec["n_lines"], rec["n_dist"], rec["vec"] = [1, 2, 30, 40], 1, 2, 3, [0.5, -0.5]
        sec[lay["blk_lines_off"]:lay["blk_lines_off"] + 64].view(np.int32)[:] = np.arange(16)
        sec[lay["blk_dist_off"]:lay["blk_dist_off"] + 24].view(np.float64)[:] = [1.5, np.nan, 3.5]
    return a, lay


def test_step_outputs_of_a_result_arena():
    """bench.py --dump-outputs: every item of the arena, as float32 / float64 rows tagged with their page"""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    n, h, w = 3, 64, 128
    arena, lay = _synthetic_arena(n, h, w)
    out = bench.step_outputs(arena, lay, n, h, w)
    assert all(a.dtype in (np.float32, np.float64) and np.all(np.isfinite(a)) for a in out.values())
    px = np.sort(np.random.default_rng(0).choice(n * h * w, min(bench.DUMP_MASK_PIXELS, n * h * w), replace=False))
    assert np.array_equal(out["mask_sample"], px % 251) and np.array_equal(out["mask_refined_sample"], px % 7)
    assert out["det"].shape == (6, 7) and out["det"][:, 0].tolist() == [0, 1, 1, 2, 2, 2]
    assert np.all(out["det"][:, 1:] == out["det"][:, :1] + 0.5)
    assert out["line_boxes"].tolist() == [[i, *range(i, i + 8)] for i in range(n)] and out["line_scores"].tolist() == [0.75] * n
    assert out["blocks"].shape == (n, 15) and out["blocks"][:, 0].tolist() == list(range(n))
    assert out["blocks"][0, 1:7].tolist() == [1, 2, 30, 40, 1, 0] and out["blocks"][0, 9:11].tolist() == [0.5, -0.5]
    assert out["blocks"][0, 14] == 2 and out["block_lines"].shape == (2 * n, 10)
    assert out["block_lines"][:2, 2:].ravel().tolist() == list(range(16))
    assert out["block_distances"][:3].tolist() == [[0, 0, 1.5, 0], [0, 0, 0, 1], [0, 0, 3.5, 0]]   # NaN -> is_nan

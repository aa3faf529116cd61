#!/bin/bash
# compute-sanitizer evidence (SURVEY section 5 / VERDICT r1 #8): memcheck over the per-kernel GPU tests and the refine /
# full-pipeline tests at small shapes, racecheck + synccheck over one small forward per engine precision and one
# full-pipeline call.  Writes gpurun_out/sanitizer_*.log (copied to profiles/ after the run).
cd "$(dirname "$0")/.."
OUT=gpurun_out
mkdir -p $OUT
CS="compute-sanitizer --print-limit 5 --launch-timeout 120"
timeout 900 $CS --tool memcheck python -m pytest tests/test_gpu_kernels.py -q -m gpu -x 2>&1 | tail -25 > $OUT/sanitizer_memcheck_kernels.log
timeout 600 $CS --tool memcheck python -m pytest tests/test_gpu_refine.py -q -m gpu -x 2>&1 | tail -25 > $OUT/sanitizer_memcheck_refine.log
cat > /tmp/fullpipe_small.py <<'PY'
import os
import sys
import numpy as np
sys.path.insert(0, os.getcwd()); sys.path.insert(0, os.path.join(os.getcwd(), "tests"))
import ctd_b200
from oracle import synth
from util import get_checkpoint
det = ctd_b200.TextDetector(get_checkpoint(0, True), input_size=256, act="leaky")
page = synth.structured_page(1000, 300, 220)
m, r, b = det(page.copy(), keep_undetected_mask=True)
print("ok", len(b), int(r.sum()))
det.close()
PY
for tool in memcheck racecheck synccheck; do
  timeout 400 $CS --tool $tool python /tmp/fullpipe_small.py 2>&1 | tail -25 > $OUT/sanitizer_${tool}_fullpipe.log
  for prec in 0 3; do
    timeout 400 $CS --tool $tool python tools/split_smoke.py $prec 128 2>&1 | tail -25 > $OUT/sanitizer_${tool}_forward_prec$prec.log
  done
done
grep -H "ERROR SUMMARY\|^ok\|passed\|failed" $OUT/sanitizer_*.log

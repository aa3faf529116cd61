#!/bin/bash
# compute-sanitizer over the kernels added / rewritten in round 2 (fused Bottleneck, seg tail GEMM + col2im, refine_mask on bit
# masks): memcheck + racecheck + synccheck of one full drop-in call on a 300x220 page (input size 256, keep_undetected) and
# memcheck of the refine tests.  Writes gpurun_out/sanitizer2_*.log
cd "$(dirname "$0")/.."
OUT=gpurun_out
mkdir -p $OUT
CS="compute-sanitizer --print-limit 5 --launch-timeout 120"
cat > /tmp/fullpipe_small.py <<'PY'
import os
import sys
import numpy as np
sys.path.insert(0, os.getcwd()); sys.path.insert(0, os.path.join(os.getcwd(), "tests"))
import ctd_b200
from oracle import synth
from util import get_checkpoint
det = ctd_b200.TextDetector(get_checkpoint(0, True), input_size=256, act="leaky")
assert any(o["kind"] == 10 for o in det.program.ops), "fused ops expected"
page = synth.structured_page(1000, 300, 220)
m, r, b = det(page.copy(), keep_undetected_mask=True)
print("ok", len(b), int(r.sum()))
det.close()
PY
for tool in memcheck racecheck synccheck; do
  timeout 420 $CS --tool $tool python /tmp/fullpipe_small.py 2>&1 | tail -12 > $OUT/sanitizer2_${tool}_fullpipe.log
done
timeout 600 $CS --tool memcheck python -m pytest tests/test_gpu_refine.py -q -m gpu -x 2>&1 | tail -12 > $OUT/sanitizer2_memcheck_refine.log
grep -H "ERROR SUMMARY\|^ok\|passed\|failed" $OUT/sanitizer2_*.log

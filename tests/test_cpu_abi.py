"""not-gpu: the C-ABI shared library loads, exports every symbol include/ctd_b200.h declares, and
refuses to run without a GPU (no CPU fallback)."""
import ctypes
import os
import re
import subprocess
import sys

import ctd_b200

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "ctd_b200.h")).read()
    return sorted(set(re.findall(r"CTD_API\s+[\w\s\*]+?\b(ctd_\w+)\s*\(", src)))


def test_header_symbols_exported():
    names = _declared()
    assert len(names) >= 16, names
    lib = ctypes.CDLL(ctd_b200.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), "libctd_b200.so does not export %s" % n
    assert sorted(ctd_b200.binding.EXPORTS) == names


def test_struct_layouts_match_header():
    # field counts / sizes the ctypes mirrors must agree with (ctd_op: 20 int32 + 4 int64)
    from ctd_b200.binding import CtdOp, CtdBufDesc, CtdConfig
    assert ctypes.sizeof(CtdOp) == 20 * 4 + 4 * 8
    assert ctypes.sizeof(CtdBufDesc) == 8
    assert ctypes.sizeof(CtdConfig) == 12 * 4


_CREATE_ENGINE = """
import ctd_b200
from ctd_b200 import compiler as cc
P = cc.Program()
P.nc = 2
P.newbuf(8, 1)
P._op(cc.OP_AVGPOOL2, [P.tensor(0, 0, 8)], P.tensor(P.newbuf(8, 2), 0, 8))
try:
    ctd_b200.Engine(P, max_batch=1, max_h=64, max_w=64)
    print("engine created")
except ctd_b200.CtdError as e:
    print("CtdError:", e)
"""


def test_no_cpu_fallback():
    # in a child process with every GPU hidden, so that this also holds on a machine that has one
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, "-c", _CREATE_ENGINE], cwd=ROOT, env=env, capture_output=True, text=True,
                         timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert out.stdout.startswith("CtdError:"), out.stdout
    assert "no CPU fallback" in out.stdout or "not sm_100" in out.stdout

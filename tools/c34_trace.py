"""Diagnostic: where the roles of the fused conv3 + conv4 kernel (tc_conv34.cuh) wait.

    python tools/c34_trace.py --build     # here (no GPU): trace build of the library next to the normal one
    python tools/c34_trace.py             # on the GPU box
"""
import ctypes as C
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
TRACE_LIB = ROOT / "hardnetnas_b200" / "csrc" / "_build" / "libhardnet_b200_c34trace.so"

if "--build" in sys.argv:
    from hardnetnas_b200 import build as B
    B.build()
    obj = B.OBJ / "hardnet_forward_c34trace.o"
    subprocess.run([B._nvcc(), *B.NVCC_FLAGS, "-DHN_C34_TRACE", "-DHN_FF_TRACE", "-c", str(B.CSRC / "hardnet_forward.cu"), "-o", str(obj)], check=True,
                   capture_output=True)
    objs = [str(o) for o in B.OBJ.glob("*.o") if o.name not in ("hardnet_forward.o", obj.name)] + [str(obj)]
    subprocess.run([B._nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(TRACE_LIB), *objs], check=True)
    print("built", TRACE_LIB)
    sys.exit(0)

import torch  # noqa: E402
from hardnetnas_b200 import _lib  # noqa: E402

_lib.LIB_PATH = TRACE_LIB
from hardnetnas_b200.hardnet import HardNet  # noqa: E402

lib = _lib.load()
lib.hn_debug_c34_trace.restype = C.c_int
lib.hn_debug_c34_trace.argtypes = [C.c_void_p, C.c_int]
x = torch.randn(18944 * 4, 1, 32, 32, device="cuda")
out = torch.empty(x.size(0), 128, device="cuda")
names = {0: "issuer: full (loads)", 1: "issuer: mid ready", 2: "issuer: t3empty", 10: "issuer: t4empty", 11: "shifter: mma4",
         5: "epi warp 4: t3full", 6: "epi warp 4: t4full", 7: "epi warp 4: conv3 epilogue", 8: "epi warp 4: conv3 + conv4 epilogue",
         9: "producer: empty", 12: "producer 0: issue section"}
m = HardNet().cuda().eval()
for _ in range(2):
    m(x, out=out)
buf = (C.c_ulonglong * 16)()
lib.hn_debug_c34_trace(buf, 1)
m(x, out=out)
lib.hn_debug_c34_trace(buf, 0)
v = list(buf)
n = max(v[4], 1)
print(f"CTA 0: {v[3] / n:.0f} cycles per patch over {n} patches")
for k, nm in names.items():
    print(f"  {nm:40s} {v[k] / n:9.0f} cycles/patch")

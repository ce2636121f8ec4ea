import os, sys, json, torch
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from tools.nas_tail_check import timing
for env in ({}, {"HN_NAS_DW_F32":"1"}):
    for arch in ("wang2","wang3","wang4"):
        for k in ("HN_NAS_DW_F32",): os.environ.pop(k,None)
        os.environ.update(env)
        r=timing(arch, {}); print("TIMING", arch, env, "%.3f ms %.2f M/s"%(r["ms"], r["patches_per_sec"]/1e6))

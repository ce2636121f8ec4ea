"""Radius matching (match_radius, match_radius_pairs) against match_topk(k=1) and a chunked torch.mm baseline on the same GPU,
in one process.

    python tools/match_radius_time.py [--out profiles/r10_match_radius.json] [--calls 3] [--reps 7]

Workloads (seeded, resident on the device before timing):
- bench: make_match_set(65536, 65536, seed=11) (the bench.py matching set) as fp32, fp16 and e4m3 rows, r = 0.5, 1.0, 1.2.
  Per (dtype, r): nnz, match_radius (count, one host read of the total, fill), the GEMM and re-rank stage times of its call
  (hn_match_profile_*: the re-rank stage is the count re-rank with its scan plus the fill re-rank), match_topk(k=1) on the same
  rows and the baseline (fp32 only: torch.mm of 4096-row query chunks against the gallery in the FDLNet form, then
  .lt(r).nonzero()).
- hpatches / exhaustive: the pair tables of tools/match_pairs_time.py (fp32), r = 1.0, against match_topk_pairs(k=1).
Every workload reports the fraction of query rows whose count re-rank scanned a whole list (hn_match_topk_fallback_*).
Timing: each form warmed up, then timed alternately with CUDA events (`calls` calls per window, `reps` windows); reported as
median ms and spread (max - min over the windows, relative to the median). The card's name, power limit and SM clock are read
in the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import sys
from pathlib import Path

import torch

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))
sys.path.insert(0, str(REPO / "tools"))
from hardnetnas_b200 import _lib  # noqa: E402
from hardnetnas_b200.matching import match_radius, match_radius_pairs, match_topk, match_topk_pairs, pair_table  # noqa: E402
from match_batched_time import gpu_info  # noqa: E402
from match_pairs_time import exhaustive_set, hpatches_set  # noqa: E402
from match_topk_time import fallback_fraction, timed  # noqa: E402
from oracle import synth  # noqa: E402


def stage_ms(lib, fn, n):
    """(GEMM ms, re-rank ms) per call, the re-rank stage summed over the call's count and fill launches."""
    ms, cnt = (C.c_double * 3)(), (C.c_longlong * 3)()
    _lib.check(lib.hn_match_profile_enable(1), "hn_match_profile_enable")
    for _ in range(n):
        fn()
    _lib.check(lib.hn_match_profile_read(ms, cnt), "hn_match_profile_read")
    lib.hn_match_profile_enable(0)
    return round(ms[1] / n, 4), round(ms[2] / n, 4)


def torch_radius(q, g, r, chunk=4096):
    for s in range(0, q.size(0), chunk):
        d = torch.sqrt((2 - 2 * torch.mm(q[s:s + chunk], g.t())).clamp(1e-8, 4.0))
        d.lt(r).nonzero()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(REPO / "profiles" / "r10_match_radius.json"))
    ap.add_argument("--calls", type=int, default=3)
    ap.add_argument("--reps", type=int, default=7)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("match_radius_time.py measures on the GPU: no CUDA device")
    lib = _lib.load()
    res = {"gpu": gpu_info(), "calls": a.calls, "reps": a.reps, "bench": [], "pairs": []}
    q32, g32, _ = synth.make_match_set(65536, 65536, seed=11)
    q32, g32 = q32.cuda(), g32.cuda()
    for dt in (torch.float32, torch.float16, torch.float8_e4m3fn):
        q, g = q32.to(dt), g32.to(dt)
        for r in (0.5, 1.0, 1.2):
            forms = {"radius": lambda: match_radius(q, g, r), "topk1": lambda: match_topk(q, g, 1)}
            if dt == torch.float32:
                forms["torch_mm_lt_nonzero"] = lambda: torch_radius(q, g, r)
            e = {"dtype": str(dt).replace("torch.", ""), "r": r, "nnz": int(match_radius(q, g, r)[0][-1]),
                 "times": timed(forms, a.calls, a.reps)}
            e["radius_stage_ms"] = dict(zip(("gemm", "rerank"), stage_ms(lib, lambda: match_radius(q, g, r), a.calls)))
            e["topk1_stage_ms"] = dict(zip(("gemm", "rerank"), stage_ms(lib, lambda: match_topk(q, g, 1), a.calls)))
            e["fallback_rows"] = fallback_fraction(lib, lambda: match_radius(q, g, r), q.size(0))
            print(json.dumps(e), flush=True)
            res["bench"].append(e)
        del q, g
    for name, make in (("hpatches", hpatches_set), ("exhaustive", exhaustive_set)):
        X, counts, i1, i2 = make(5)
        T = pair_table(counts.cuda(), i1.cuda(), i2.cuda())
        tl = T.cpu().tolist()
        max_q, max_g = max(t[1] for t in tl), max(t[3] for t in tl)
        rows = sum(t[1] for t in tl)
        r = 1.0
        forms = {"radius_pairs": lambda: match_radius_pairs(X, X, T, r, max_q, max_g),
                 "topk1_pairs": lambda: match_topk_pairs(X, X, T, 1, max_q, max_g)}
        e = {"workload": name, "pairs": len(tl), "r": r, "nnz": int(match_radius_pairs(X, X, T, r, max_q, max_g)[0][-1]),
             "times": timed(forms, a.calls, a.reps)}
        e["radius_stage_ms"] = dict(zip(("gemm", "rerank"), stage_ms(lib, lambda: match_radius_pairs(X, X, T, r, max_q, max_g), a.calls)))
        e["topk1_stage_ms"] = dict(zip(("gemm", "rerank"), stage_ms(lib, lambda: match_topk_pairs(X, X, T, 1, max_q, max_g), a.calls)))
        e["fallback_rows"] = fallback_fraction(lib, lambda: match_radius_pairs(X, X, T, r, max_q, max_g), rows)
        print(json.dumps(e), flush=True)
        res["pairs"].append(e)
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()

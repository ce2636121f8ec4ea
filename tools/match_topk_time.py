"""k-nearest-neighbour matching (match_topk, match_topk_pairs) against the top-2 calls and a chunked torch.mm + torch.topk
baseline on the same GPU, in one process.

    python tools/match_topk_time.py [--out profiles/r9_match_topk.json] [--calls 3] [--reps 7]

Workloads (seeded, resident on the device before timing):
- bench: make_match_set(65536, 65536, seed=11) (the bench.py matching set) as fp32, fp16 and e4m3 rows, k = 1, 2, 4, 8.
  Per (dtype, k): match_topk, the GEMM and re-rank stage times of its call (hn_match_profile_*), match_top2 on the same rows
  and the baseline (fp32 only: torch.mm of 4096-row query chunks against the gallery in the FDLNet form, then torch.topk).
- hpatches / exhaustive: the pair tables of tools/match_pairs_time.py (fp32), k = 2 and 8, against match_top2_pairs.
Every workload reports the fraction of query rows whose re-rank scanned a whole list (hn_match_topk_fallback_*).
Timing: each form warmed up, then timed alternately with CUDA events (`calls` calls per window, `reps` windows); reported as
median ms and spread (max - min over the windows, relative to the median). The card's name, power limit and SM clock are read
in the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import statistics
import sys
from pathlib import Path

import torch

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))
sys.path.insert(0, str(REPO / "tools"))
from hardnetnas_b200 import _lib  # noqa: E402
from hardnetnas_b200.matching import match_top2, match_top2_pairs, match_topk, match_topk_pairs, pair_table  # noqa: E402
from match_batched_time import gpu_info, window  # noqa: E402
from match_pairs_time import exhaustive_set, gemm_ms, hpatches_set  # noqa: E402
from oracle import synth  # noqa: E402


def timed(forms, calls, reps):
    """{name: (median ms, relative spread)} of the forms, timed in alternating windows after a warm-up."""
    for f in forms.values():
        f()
    torch.cuda.synchronize()
    t = {n: [] for n in forms}
    for _ in range(reps):
        for n, f in forms.items():
            t[n].append(window(f, calls))
    out = {}
    for n, v in t.items():
        med = statistics.median(v)
        out[n] = {"ms": round(med, 4), "spread": round((max(v) - min(v)) / med, 4)}
    return out


def fallback_fraction(lib, fn, rows):
    _lib.check(lib.hn_match_topk_fallback_enable(1), "hn_match_topk_fallback_enable")
    fn()
    n = C.c_longlong(0)
    _lib.check(lib.hn_match_topk_fallback_read(C.byref(n)), "hn_match_topk_fallback_read")
    lib.hn_match_topk_fallback_enable(0)
    return n.value / rows


def torch_topk(q, g, k, chunk=4096):
    for s in range(0, q.size(0), chunk):
        d = torch.sqrt((2 - 2 * torch.mm(q[s:s + chunk], g.t())).clamp(1e-8, 4.0))
        torch.topk(d, k, dim=1, largest=False, sorted=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(REPO / "profiles" / "r9_match_topk.json"))
    ap.add_argument("--calls", type=int, default=3)
    ap.add_argument("--reps", type=int, default=7)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("match_topk_time.py measures on the GPU: no CUDA device")
    lib = _lib.load()
    res = {"gpu": gpu_info(), "calls": a.calls, "reps": a.reps, "bench": [], "pairs": []}
    q32, g32, _ = synth.make_match_set(65536, 65536, seed=11)
    q32, g32 = q32.cuda(), g32.cuda()
    for dt in (torch.float32, torch.float16, torch.float8_e4m3fn):
        q, g = q32.to(dt), g32.to(dt)
        for k in (1, 2, 4, 8):
            forms = {"topk": lambda: match_topk(q, g, k), "top2": lambda: match_top2(q, g)}
            if dt == torch.float32:
                forms["torch_mm_topk"] = lambda: torch_topk(q, g, k)
            e = {"dtype": str(dt).replace("torch.", ""), "k": k, "times": timed(forms, a.calls, a.reps)}
            gm, rr = gemm_ms(lib, lambda: match_topk(q, g, k), a.calls)
            e["topk_stage_ms"] = {"gemm": round(gm, 4), "rerank": round(rr, 4)}
            gm, rr = gemm_ms(lib, lambda: match_top2(q, g), a.calls)
            e["top2_stage_ms"] = {"gemm": round(gm, 4), "rerank": round(rr, 4)}
            e["fallback_rows"] = fallback_fraction(lib, lambda: match_topk(q, g, k), q.size(0))
            print(json.dumps(e), flush=True)
            res["bench"].append(e)
        del q, g
    for name, make in (("hpatches", hpatches_set), ("exhaustive", exhaustive_set)):
        X, counts, i1, i2 = make(5)
        T = pair_table(counts.cuda(), i1.cuda(), i2.cuda())
        tl = T.cpu().tolist()
        max_q, max_g = max(r[1] for r in tl), max(r[3] for r in tl)
        rows = sum(r[1] for r in tl)
        for k in (2, 8):
            forms = {"topk_pairs": lambda: match_topk_pairs(X, X, T, k, max_q, max_g),
                     "top2_pairs": lambda: match_top2_pairs(X, X, T, max_q, max_g)}
            e = {"workload": name, "pairs": len(tl), "k": k, "times": timed(forms, a.calls, a.reps)}
            gm, rr = gemm_ms(lib, lambda: match_topk_pairs(X, X, T, k, max_q, max_g), a.calls)
            e["topk_stage_ms"] = {"gemm": round(gm, 4), "rerank": round(rr, 4)}
            gm, rr = gemm_ms(lib, lambda: match_top2_pairs(X, X, T, max_q, max_g), a.calls)
            e["top2_stage_ms"] = {"gemm": round(gm, 4), "rerank": round(rr, 4)}
            e["fallback_rows"] = fallback_fraction(lib, lambda: match_topk_pairs(X, X, T, k, max_q, max_g), rows)
            print(json.dumps(e), flush=True)
            res["pairs"].append(e)
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()

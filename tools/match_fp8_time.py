"""Matching on fp8 e4m3 descriptor rows (HN_F8E4M3: e4m3 operands, kind::f8f6f4 GEMM) against fp32 and fp16 rows, in one
process.

    python tools/match_fp8_time.py [--out profiles/r7_match_fp8.json] [--calls 3] [--reps 7]

Workloads: those of tools/match_16bit_time.py (r5 / r6): the padded batches 256 x 1024, 64 x 4096, 256 x [512, 1024] and
1 x 8192, the HPatches-shaped and exhaustive pair tables, and one 64k x 64k problem, each as top-2 and as mutual NN + ratio.
The fp32 rows are generated as there; the fp16 and e4m3 rows are their conversions. The three row types are warmed up, then
timed alternately within one process (`calls` calls per window, `reps` windows; medians and spreads = (max - min) / median).
Reported per row type: ms per call, stage times of hn_match_profile_* (pack, GEMM + shortlist, re-rank), peak allocation
during one call, and whether the outputs equal the fp32 call on the rows' .float() bit for bit. For information only: the
fraction of valid query rows whose nearest gallery row (i1) on e4m3 rows equals i1 on the original fp32 rows.
"""
from __future__ import annotations

import argparse
import json
import statistics
import sys
from pathlib import Path

import torch

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))
sys.path.insert(0, str(REPO / "tools"))
from hardnetnas_b200 import _lib  # noqa: E402
from match_16bit_time import identical, peak_bytes, python_call, rows_of, stage_ms, with_rows, workloads  # noqa: E402
from match_batched_time import gpu_info, window  # noqa: E402

DTYPES = {"fp32": torch.float32, "fp16": torch.float16, "e4m3": torch.float8_e4m3fn}


def _ia_agreement(kind, data, i1_8, i1_32):
    """Fraction of valid query rows whose i1 on e4m3 rows equals i1 on the original fp32 rows."""
    if kind == "single":
        return (i1_8 == i1_32).float().mean().item()
    if kind == "batched":
        lq = data[2]
        valid = torch.arange(i1_8.size(1), device=i1_8.device)[None, :] < lq[:, None]
    else:
        T = data[1]
        valid = torch.arange(i1_8.size(1), device=i1_8.device)[None, :] < T[:, 1:2]
    return ((i1_8 == i1_32) & valid).sum().item() / max(valid.sum().item(), 1)


def run_workload(name, kind, data32, a, lib):
    inputs = {dt: with_rows(kind, data32, [r.to(t) for r in rows_of(kind, data32)]) for dt, t in DTYPES.items()}
    entry = {"workload": name, "kind": kind,
             "rows": sum(r.shape[0] * (r.shape[1] if r.dim() == 3 else 1) for r in rows_of(kind, data32)),
             "input_bytes": {dt: sum(r.numel() * r.element_size() for r in rows_of(kind, d)) for dt, d in inputs.items()}}
    for form in ("top2", "mutual_ratio"):
        fns = {dt: python_call(kind, form, d) for dt, d in inputs.items()}
        for _ in range(2):
            for fn in fns.values():
                fn()
        torch.cuda.synchronize()
        times = {k: [] for k in fns}
        for _ in range(a.reps):          # alternate the row types
            for k, fn in fns.items():
                times[k].append(window(fn, a.calls))
        med = {k: statistics.median(v) for k, v in times.items()}
        res = {}
        for k, fn in fns.items():
            res[k] = {"ms": med[k], "ms_all": times[k], "spread": (max(times[k]) - min(times[k])) / med[k],
                      "peak_alloc_bytes": peak_bytes(fn), "stage_ms": stage_ms(lib, fn, a.calls)}
        for dt in ("fp16", "e4m3"):
            d = inputs[dt]
            res[dt]["equal_to_fp32_call_on_float"] = identical(fns[dt](), python_call(
                kind, form, with_rows(kind, d, [r.float() for r in rows_of(kind, d)]))())
        if form == "top2":
            res["e4m3"]["ia_equal_to_fp32_rows_fraction"] = _ia_agreement(kind, data32, fns["e4m3"]()[2], fns["fp32"]()[2])
        res["e4m3_over_fp16"] = med["e4m3"] / med["fp16"]
        res["e4m3_over_fp32"] = med["e4m3"] / med["fp32"]
        res["gemm_e4m3_over_fp16"] = res["e4m3"]["stage_ms"]["gemm"] / res["fp16"]["stage_ms"]["gemm"]
        entry[form] = res
    del inputs
    print(json.dumps({"workload": name, **{f: {k: (round(v["ms"], 4) if isinstance(v, dict) else round(v, 4))
                                                for k, v in entry[f].items()} for f in ("top2", "mutual_ratio")},
                      "gemm_ms": {f: {k: round(entry[f][k]["stage_ms"]["gemm"], 4) for k in DTYPES} for f in ("top2", "mutual_ratio")}}),
          flush=True)
    return entry


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(REPO / "profiles" / "r7_match_fp8.json"))
    ap.add_argument("--calls", type=int, default=3)
    ap.add_argument("--reps", type=int, default=7)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("match_fp8_time.py measures on the GPU: no CUDA device")
    lib = _lib.load()
    result = {"gpu": gpu_info(), "calls_per_window": a.calls, "windows": a.reps, "workloads": []}
    for name, kind, data in workloads():
        result["workloads"].append(run_workload(name, kind, data, a, lib))
        del data
        torch.cuda.empty_cache()
    result["gpu_after"] = gpu_info()
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    # one line per workload: the file stays readable in a diff
    body = ",\n".join(f"  {json.dumps(w)}" for w in result.pop("workloads"))
    head = ",\n".join(f" {json.dumps(k)}: {json.dumps(v)}" for k, v in result.items())
    Path(a.out).write_text("{\n" + head + ',\n "workloads": [\n' + body + "\n ]\n}\n")
    print("wrote", a.out)


if __name__ == "__main__":
    main()

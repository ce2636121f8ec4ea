"""Batched matching (hn_match_batched) against a Python loop of per-pair calls over the same slices, in one process.

    python tools/match_batched_time.py [--out profiles/r3_match_batched.json] [--calls 5] [--reps 7]

Workloads: 256 pairs x 1024 keypoints, 64 x 4096, 256 pairs with ragged lengths uniform in [512, 1024] (padded to 1024),
1 x 8192. Each pair is an oracle/synth.make_match_set set, resident on the device before timing. For every workload and for
top-2 (match_top2) and mutual NN + ratio (mutual_nn_ratio, return_pairs=False) the two forms are warmed up, then timed
alternately with CUDA events (`calls` calls per window, `reps` windows each, median reported). The working sets of the
256-pair workloads (256 MB of fp32 descriptors) exceed the 126 MB L2; the others are partly L2-resident across calls.
Reported per form: ms per call, descriptor pairs per second (sum of q_len * g_len / time) and the fraction of the B200's
dense bf16 data-sheet peak (2.25 PFLOP/s at 1000 W) that 256 FLOP per descriptor pair represents; for the batched top-2 call
also the GEMM kernel's own time (CUDA events around it, hn_match_profile_*) and its fraction of that peak.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import statistics
import subprocess
import sys
from pathlib import Path

import torch

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))
from hardnetnas_b200 import _lib  # noqa: E402
from hardnetnas_b200.matching import (match_top2, match_top2_batched, mutual_nn_ratio,  # noqa: E402
                                      mutual_nn_ratio_batched)
from oracle import synth  # noqa: E402

PEAK_BF16 = 2.25e15          # dense bf16 FLOP/s of one B200 (data sheet, 1000 W)
FLOP_PER_PAIR = 2 * 128      # one 128-term dot product per (query, gallery) descriptor pair


def gpu_info() -> dict:
    info = {"torch_name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        info["nvidia_smi"] = r.stdout.strip().splitlines()[0] if r.stdout.strip() else r.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


def make_workload(B, n, ragged, seed):
    gen = torch.Generator().manual_seed(seed)
    if ragged:
        lq = torch.randint(512, 1025, (B,), generator=gen).tolist()
        lg = torch.randint(512, 1025, (B,), generator=gen).tolist()
    else:
        lq, lg = [n] * B, [n] * B
    Q = torch.zeros(B, n, 128, device="cuda")
    G = torch.zeros(B, n, 128, device="cuda")
    for b in range(B):
        q, g, _ = synth.make_match_set(lq[b], lg[b], seed=seed + b)
        Q[b, :lq[b]] = q.cuda()
        G[b, :lg[b]] = g.cuda()
    return Q, G, lq, lg


def window(fn, calls):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / calls


def launches(fn, lib):
    torch.cuda.synchronize()
    n0 = lib.hn_launch_count()
    fn()
    torch.cuda.synchronize()
    return lib.hn_launch_count() - n0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(REPO / "profiles" / "r3_match_batched.json"))
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--reps", type=int, default=7)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("match_batched_time.py measures on the GPU: no CUDA device")
    lib = _lib.load()
    result = {"gpu": gpu_info(), "calls_per_window": a.calls, "windows": a.reps, "workloads": []}
    for name, B, n, ragged in [("256x1024", 256, 1024, False), ("64x4096", 64, 4096, False),
                               ("256x[512,1024]", 256, 1024, True), ("1x8192", 1, 8192, False)]:
        Q, G, lq, lg = make_workload(B, n, ragged, seed=100)
        L1 = torch.tensor(lq, dtype=torch.int32, device="cuda")
        L2 = torch.tensor(lg, dtype=torch.int32, device="cuda")
        slices = [(Q[b, :lq[b]], G[b, :lg[b]]) for b in range(B)]
        dpairs = sum(x * y for x, y in zip(lq, lg))
        forms = {
            "top2": (lambda: match_top2_batched(Q, G, L1, L2), lambda: [match_top2(q, g) for q, g in slices]),
            "mutual_ratio": (lambda: mutual_nn_ratio_batched(Q, G, L1, L2),
                             lambda: [mutual_nn_ratio(q, g, return_pairs=False) for q, g in slices]),
        }
        entry = {"workload": name, "pairs": B, "padded_rows": n, "descriptor_pairs": dpairs}
        for form, (batched, loop) in forms.items():
            for _ in range(3):
                batched()
                loop()
            torch.cuda.synchronize()
            tb, tl = [], []
            for _ in range(a.reps):      # alternate the two forms
                tb.append(window(batched, a.calls))
                tl.append(window(loop, a.calls))
            mb, ml = statistics.median(tb), statistics.median(tl)
            # same outputs: the batched call equals the loop pair by pair
            if form == "top2":
                got, want = batched(), loop()
                equal = all(torch.equal(got[k][b, :lq[b]], want[b][k]) for b in range(B) for k in range(4))
            else:
                got, want = batched(), loop()
                equal = all(torch.equal(got[0][b, :lq[b]], want[b][1]) and torch.equal(got[2][b, :lq[b]], want[b][3])
                            for b in range(B))
            entry[form] = {
                "batched_ms": mb, "loop_ms": ml, "speedup": ml / mb,
                "batched_ms_all": tb, "loop_ms_all": tl,
                "batched_desc_pairs_per_s": dpairs / (mb * 1e-3), "loop_desc_pairs_per_s": dpairs / (ml * 1e-3),
                "batched_frac_bf16_peak": dpairs * FLOP_PER_PAIR / (mb * 1e-3) / PEAK_BF16,
                "loop_frac_bf16_peak": dpairs * FLOP_PER_PAIR / (ml * 1e-3) / PEAK_BF16,
                "batched_launches": launches(batched, lib), "loop_launches": launches(loop, lib),
                "equal_to_loop": bool(equal),
            }
        # the GEMM kernel's own time inside the batched top-2 call
        ms, cnt = (C.c_double * 3)(), (C.c_longlong * 3)()
        _lib.check(lib.hn_match_profile_enable(1), "hn_match_profile_enable")
        for _ in range(a.calls * a.reps):
            match_top2_batched(Q, G, L1, L2)
        _lib.check(lib.hn_match_profile_read(ms, cnt), "hn_match_profile_read")
        lib.hn_match_profile_enable(0)
        stage = [ms[i] / max(cnt[i], 1) for i in range(3)]
        entry["top2"]["batched_stage_ms"] = {"pack": stage[0], "gemm": stage[1], "rerank": stage[2]}
        entry["top2"]["gemm_frac_bf16_peak"] = dpairs * FLOP_PER_PAIR / (stage[1] * 1e-3) / PEAK_BF16
        result["workloads"].append(entry)
        print(json.dumps({k: entry[k] for k in ("workload", "descriptor_pairs")}),
              {f: {k: round(v, 4) if isinstance(v, float) else v for k, v in entry[f].items() if not k.endswith("_all")}
               for f in forms}, flush=True)
        del Q, G, slices
        torch.cuda.empty_cache()
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(result, indent=1) + "\n")
    print("wrote", a.out)


if __name__ == "__main__":
    main()

"""Pair-table matching (hn_match_pairs) against the padded batched call and a loop of per-pair calls, plus an A/B of
hn_match_batched against another build of the library, in one process.

    python tools/match_pairs_time.py [--out profiles/r4_match_pairs.json] [--calls 3] [--reps 7] [--parent-lib PATH]

Workloads (descriptor sets resident on the device before timing, seeded):
- hpatches: 116 sequences x 6 images, keypoints per image uniform in [1024, 4096]; 580 (reference, other) pairs. One
  concatenated set; each image other than the reference holds noisy copies (sigma 0.04) of 80 % of the reference's rows.
- exhaustive: 64 images x 2048 keypoints (unit random rows), all 2016 unordered pairs (i < j).
Forms, each for top-2 (match_top2*) and mutual NN + ratio (mutual_nn_ratio*):
- pairs: match_top2_pairs / mutual_nn_ratio_pairs on the concatenated set, packing included (one pack, g is q);
- padded: building the padded copies [P, max_len, 128] of both sides (gather; its time reported as build_ms and included in
  padded_ms) + match_top2_batched / mutual_nn_ratio_batched;
- loop: the per-pair call on each pair's slices.
Timing: every form warmed up, then timed alternately with CUDA events (`calls` calls per window, `reps` windows, medians).
Reported per form: ms per call, device memory held by its inputs, descriptor pairs per second (sum of q_len * g_len / time)
and, for the pair-table top-2 call, the GEMM kernel's own time (hn_match_profile_*) and its share of the B200's dense bf16
data-sheet rate (2.25 PFLOP/s at 1000 W) at 256 FLOP per descriptor pair.
A/B (--parent-lib): the four workloads of tools/match_batched_time.py through hn_match_batched of this build and of the other
library, alternating windows; reports both medians, each build's spread (max - min over the windows, relative to its median)
and whether the outputs are bit-identical.
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
from hardnetnas_b200._ops import pack_descriptors  # noqa: E402
from hardnetnas_b200.matching import (match_top2, match_top2_batched, match_top2_pairs, mutual_nn_ratio,  # noqa: E402
                                      mutual_nn_ratio_batched, mutual_nn_ratio_pairs, pair_table)
from match_batched_time import gpu_info, launches, make_workload, window  # noqa: E402

PEAK_BF16 = 2.25e15          # dense bf16 FLOP/s of one B200 (data sheet, 1000 W)
FLOP_PER_PAIR = 2 * 128      # one 128-term dot product per (query, gallery) descriptor pair


def _unit(x):
    return x / x.norm(dim=1, keepdim=True)


def hpatches_set(seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    cpu = torch.Generator().manual_seed(seed)
    counts = torch.randint(1024, 4097, (116 * 6,), generator=cpu)
    blocks = []
    for s in range(116):
        ref = _unit(torch.randn(int(counts[6 * s]), 128, device="cuda", generator=gen))
        blocks.append(ref)
        for k in range(1, 6):
            n = int(counts[6 * s + k])
            x = _unit(torch.randn(n, 128, device="cuda", generator=gen))
            m = int(0.8 * min(n, ref.size(0)))
            src = torch.randperm(ref.size(0), device="cuda", generator=gen)[:m]
            x[:m] = _unit(ref[src] + 0.04 * torch.randn(m, 128, device="cuda", generator=gen))
            blocks.append(x[torch.randperm(n, device="cuda", generator=gen)])
    X = torch.cat(blocks)
    ref_idx = torch.arange(116).repeat_interleave(5) * 6
    other = ref_idx + torch.arange(1, 6).repeat(116)
    return X, counts, ref_idx, other


def exhaustive_set(seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    X = _unit(torch.randn(64 * 2048, 128, device="cuda", generator=gen))
    i, j = torch.triu_indices(64, 64, offset=1)
    return X, torch.full((64,), 2048), i, j


def padded_copies(X, table, max_len, side):
    """[P, max_len, 128] copies of one side's row ranges (zero rows past each length) and the lengths as device int32."""
    start, length = table[:, 2 * side].long(), table[:, 2 * side + 1].long()
    r = torch.arange(max_len, device=X.device)
    rows = (start.unsqueeze(1) + r).clamp(max=X.size(0) - 1)
    out = X[rows]
    out[r.unsqueeze(0) >= length.unsqueeze(1)] = 0
    return out, length.to(torch.int32)


def gemm_ms(lib, fn, n):
    ms, cnt = (C.c_double * 3)(), (C.c_longlong * 3)()
    _lib.check(lib.hn_match_profile_enable(1), "hn_match_profile_enable")
    for _ in range(n):
        fn()
    _lib.check(lib.hn_match_profile_read(ms, cnt), "hn_match_profile_read")
    lib.hn_match_profile_enable(0)
    return ms[1] / max(cnt[1], 1), ms[2] / max(cnt[2], 1)


def run_workload(name, X, counts, idx1, idx2, a, lib):
    T = pair_table(counts.cuda(), idx1.cuda(), idx2.cuda())
    tl = T.cpu().tolist()
    max_q, max_g = max(r[1] for r in tl), max(r[3] for r in tl)
    dpairs = sum(r[1] * r[3] for r in tl)
    slices = [(X[r[0]:r[0] + r[1]], X[r[2]:r[2] + r[3]]) for r in tl]
    holder = {}

    def build():
        holder["Q"], holder["L1"] = padded_copies(X, T, max_q, 0)
        holder["G"], holder["L2"] = padded_copies(X, T, max_g, 1)

    build()
    padded_bytes = holder["Q"].numel() * 4 + holder["G"].numel() * 4
    set_bytes = X.numel() * 4
    entry = {"workload": name, "pairs": len(tl), "images": int(counts.numel()), "set_rows": X.size(0), "max_q": max_q,
             "max_g": max_g, "descriptor_pairs": dpairs,
             "input_bytes": {"pairs": set_bytes + X.size(0) * 128 * 2 + T.numel() * 4, "padded": padded_bytes + 2 * len(tl) * 4,
                             "loop": set_bytes}}
    forms = {
        "top2": (lambda: match_top2_pairs(X, X, T, max_q, max_g),
                 lambda: match_top2_batched(holder["Q"], holder["G"], holder["L1"], holder["L2"]),
                 lambda: [match_top2(q, g) for q, g in slices]),
        "mutual_ratio": (lambda: mutual_nn_ratio_pairs(X, X, T, max_q, max_g),
                         lambda: mutual_nn_ratio_batched(holder["Q"], holder["G"], holder["L1"], holder["L2"]),
                         lambda: [mutual_nn_ratio(q, g, return_pairs=False) for q, g in slices]),
    }
    for form, (pairs_fn, padded_fn, loop_fn) in forms.items():
        for _ in range(2):
            pairs_fn(), build(), padded_fn(), loop_fn()
        torch.cuda.synchronize()
        tp, tb, tpad, tl_ = [], [], [], []
        for _ in range(a.reps):      # alternate the forms
            tp.append(window(pairs_fn, a.calls))
            tb.append(window(build, a.calls))
            tpad.append(window(padded_fn, a.calls))
            tl_.append(window(loop_fn, a.calls))
        mp, mb, mpad, ml = (statistics.median(v) for v in (tp, tb, tpad, tl_))
        got, pad, loop = pairs_fn(), padded_fn(), loop_fn()
        equal_padded = all(torch.equal(x, y) for x, y in zip(got, pad))
        if form == "top2":
            equal_loop = all(torch.equal(got[k][p, :tl[p][1]], loop[p][k].long() if k >= 2 else loop[p][k])
                             for p in range(len(tl)) for k in range(4))
        else:
            equal_loop = all(torch.equal(got[0][p, :tl[p][1]], loop[p][1]) and torch.equal(got[2][p, :tl[p][1]], loop[p][3])
                             for p in range(len(tl)))
        entry[form] = {
            "pairs_ms": mp, "padded_ms": mpad + mb, "padded_build_ms": mb, "padded_call_ms": mpad, "loop_ms": ml,
            "pairs_ms_all": tp, "padded_build_ms_all": tb, "padded_call_ms_all": tpad, "loop_ms_all": tl_,
            "speedup_vs_padded": (mpad + mb) / mp, "speedup_vs_loop": ml / mp,
            "pairs_desc_pairs_per_s": dpairs / (mp * 1e-3), "padded_desc_pairs_per_s": dpairs / ((mpad + mb) * 1e-3),
            "loop_desc_pairs_per_s": dpairs / (ml * 1e-3),
            "pairs_launches": launches(pairs_fn, lib), "padded_launches": launches(padded_fn, lib), "loop_launches": launches(loop_fn, lib),
            "equal_to_padded": bool(equal_padded), "equal_to_loop": bool(equal_loop),
        }
    g_ms, r_ms = gemm_ms(lib, forms["top2"][0], a.calls * a.reps)
    entry["top2"]["pairs_stage_ms"] = {"gemm": g_ms, "rerank": r_ms}
    entry["top2"]["gemm_frac_bf16_peak"] = dpairs * FLOP_PER_PAIR / (g_ms * 1e-3) / PEAK_BF16
    print(json.dumps({k: entry[k] for k in ("workload", "pairs", "descriptor_pairs", "input_bytes")}),
          {f: {k: round(v, 4) if isinstance(v, float) else v for k, v in entry[f].items() if not k.endswith("_all")} for f in forms},
          flush=True)
    return entry


def load_lib(path):
    lib = C.CDLL(str(path))
    for name in ("hn_match_batched_workspace_bytes", "hn_match_batched", "hn_launch_count", "hn_last_error"):
        res, args = _lib.SIGNATURES[name]
        getattr(lib, name).restype = res
        getattr(lib, name).argtypes = args
    return lib


def ab_batched(parent_path, a):
    """hn_match_batched of this build and of the library at parent_path on the r3 workloads, alternating windows."""
    libs = {"this": load_lib(_lib.LIB_PATH), "parent": load_lib(parent_path)}
    out = {"parent_lib": str(parent_path), "workloads": []}
    for name, B, n, ragged in [("256x1024", 256, 1024, False), ("64x4096", 64, 4096, False),
                               ("256x[512,1024]", 256, 1024, True), ("1x8192", 1, 8192, False)]:
        Q, G, lq, lg = make_workload(B, n, ragged, seed=100)
        L1 = torch.tensor(lq, dtype=torch.int32, device="cuda")
        L2 = torch.tensor(lg, dtype=torch.int32, device="cuda")
        entry = {"workload": name}
        for form, mutual in (("top2", False), ("mutual_ratio", True)):
            state = {}
            for key, lib in libs.items():
                ws = torch.empty(lib.hn_match_batched_workspace_bytes(B, n, n, int(mutual)) + 256, dtype=torch.uint8, device="cuda")
                outs = [torch.empty(B * n, dtype=t, device="cuda") for t in (torch.float32, torch.float32, torch.int32, torch.int32)]
                mu = torch.empty(B * n, dtype=torch.uint8, device="cuda") if mutual else None
                args = ([C.c_void_p(Q.data_ptr()), C.c_void_p(G.data_ptr()), B, n, n, C.c_void_p(L1.data_ptr()),
                         C.c_void_p(L2.data_ptr())] + [C.c_void_p(t.data_ptr()) for t in outs] +
                        [C.c_void_p(mu.data_ptr() if mu is not None else 0), C.c_void_p(ws.data_ptr()), ws.numel(), None])

                def call(lib=lib, args=args):
                    st = lib.hn_match_batched(*args)
                    if st != 0:
                        raise RuntimeError(lib.hn_last_error().decode())
                state[key] = (call, outs + ([mu] if mu is not None else []), ws)
            for _ in range(3):
                for call, _, _ in state.values():
                    call()
            torch.cuda.synchronize()
            times = {k: [] for k in state}
            for _ in range(a.reps):
                for k, (call, _, _) in state.items():
                    times[k].append(window(call, a.calls * 2))
            identical = all(torch.equal(x, y) for x, y in zip(state["this"][1], state["parent"][1]))
            med = {k: statistics.median(v) for k, v in times.items()}
            entry[form] = {f"{k}_ms": med[k] for k in med}
            entry[form].update({f"{k}_ms_all": v for k, v in times.items()})
            entry[form].update({f"{k}_spread": (max(v) - min(v)) / med[k] for k, v in times.items()})
            entry[form]["this_over_parent"] = med["this"] / med["parent"]
            entry[form]["outputs_identical"] = bool(identical)
        out["workloads"].append(entry)
        print(json.dumps({"ab": name, **{f: {k: round(v, 4) if isinstance(v, float) else v for k, v in entry[f].items()
                                              if not k.endswith("_all")} for f in ("top2", "mutual_ratio")}}), flush=True)
        del Q, G
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(REPO / "profiles" / "r4_match_pairs.json"))
    ap.add_argument("--calls", type=int, default=3)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--parent-lib", default=None, help="another build of libhardnet_b200.so for the hn_match_batched A/B")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("match_pairs_time.py measures on the GPU: no CUDA device")
    lib = _lib.load()
    result = {"gpu": gpu_info(), "calls_per_window": a.calls, "windows": a.reps, "workloads": []}
    for name, make in (("hpatches", hpatches_set), ("exhaustive", exhaustive_set)):
        X, counts, i1, i2 = make(200)
        result["workloads"].append(run_workload(name, X, counts, i1, i2, a, lib))
        del X
        torch.cuda.empty_cache()
    if a.parent_lib:
        result["ab_match_batched"] = ab_batched(Path(a.parent_lib), a)
    result["gpu_after"] = gpu_info()
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(result, indent=1) + "\n")
    print("wrote", a.out)


if __name__ == "__main__":
    main()

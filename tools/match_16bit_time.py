"""Matching on fp16 / bf16 descriptor rows (the *_typed entry points) against fp32 rows, plus an A/B of the fp32 path against
another build of the library, in one process.

    python tools/match_16bit_time.py [--out profiles/r5_match_16bit.json] [--calls 3] [--reps 7] [--parent-lib PATH]

Workloads (descriptor sets resident on the device before timing, seeded): the four padded batches of
tools/match_batched_time.py (256 x 1024, 64 x 4096, 256 x [512, 1024], 1 x 8192; match_*_batched), the hpatches and
exhaustive pair tables of tools/match_pairs_time.py (match_*_pairs, one set, packed once per call), and one 64k x 64k
problem (match_top2 / mutual_nn_ratio). The fp32 rows are generated as in those tools; the 16-bit rows are their conversions.
Forms, each for top-2 and for mutual NN + ratio: fp32 rows, fp16 rows, bf16 rows, and "fp16 + upcast": the fp32 call on
x16.float() including that conversion (what a caller holding fp16 descriptors paid before the typed entry points).
Timing: every form warmed up, then timed alternately with CUDA events (`calls` calls per window, `reps` windows, medians and
spreads = (max - min) / median over the windows). Reported per form: ms per call, the stage times of hn_match_profile_*
(pack, GEMM, re-rank; top-2 and mutual alike), device memory held by the inputs, the peak allocation during one call (above
what was allocated before it, workspace already grown), and whether the outputs equal those of the fp32 call on x16.float()
bit for bit.
A/B (--parent-lib): the fp32 entry points (hn_match_batched, hn_pack_descriptors + hn_match_pairs, hn_match_ex /
hn_match_mutual) of this build and of the library at PATH on the same workloads, alternating windows; both medians, each
build's spread and whether the outputs are bit-identical.
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
from hardnetnas_b200.matching import (match_top2, match_top2_batched, match_top2_pairs, mutual_nn_ratio,  # noqa: E402
                                      mutual_nn_ratio_batched, mutual_nn_ratio_pairs, pair_table)
from match_batched_time import gpu_info, make_workload, window  # noqa: E402
from match_pairs_time import exhaustive_set, hpatches_set  # noqa: E402

DTYPES = {"fp32": torch.float32, "fp16": torch.float16, "bf16": torch.bfloat16}


def workloads():
    """name -> (kind, fp32 data): kind 'batched' (Q, G, L1, L2), 'pairs' (X, T, max_q, max_g) or 'single' (q, g)."""
    for name, B, n, ragged in [("256x1024", 256, 1024, False), ("64x4096", 64, 4096, False),
                               ("256x[512,1024]", 256, 1024, True), ("1x8192", 1, 8192, False)]:
        Q, G, lq, lg = make_workload(B, n, ragged, seed=100)
        yield name, "batched", (Q, G, torch.tensor(lq, dtype=torch.int32, device="cuda"),
                                torch.tensor(lg, dtype=torch.int32, device="cuda"))
    for name, make in (("hpatches", hpatches_set), ("exhaustive", exhaustive_set)):
        X, counts, i1, i2 = make(200)
        T = pair_table(counts.cuda(), i1.cuda(), i2.cuda())
        tl = T.cpu().tolist()
        yield name, "pairs", (X, T, max(r[1] for r in tl), max(r[3] for r in tl))
    gen = torch.Generator(device="cuda").manual_seed(300)
    q = torch.nn.functional.normalize(torch.randn(65536, 128, device="cuda", generator=gen), dim=1)
    g = torch.nn.functional.normalize(torch.randn(65536, 128, device="cuda", generator=gen), dim=1)
    yield "64kx64k", "single", (q, g)


def rows_of(kind, data):
    return data[:2] if kind in ("batched", "single") else data[:1]


def with_rows(kind, data, rows):
    return (*rows, *data[2:]) if kind in ("batched", "single") else (rows[0], *data[1:])


def python_call(kind, form, data):
    """The public matching call on `data` for one form: 'top2' or 'mutual_ratio'."""
    if kind == "batched":
        Q, G, L1, L2 = data
        return (lambda: match_top2_batched(Q, G, L1, L2)) if form == "top2" else (lambda: mutual_nn_ratio_batched(Q, G, L1, L2))
    if kind == "pairs":
        X, T, mq, mg = data
        return (lambda: match_top2_pairs(X, X, T, mq, mg)) if form == "top2" else (lambda: mutual_nn_ratio_pairs(X, X, T, mq, mg))
    q, g = data
    return (lambda: match_top2(q, g)) if form == "top2" else (lambda: mutual_nn_ratio(q, g, return_pairs=False))


def stage_ms(lib, fn, n):
    ms, cnt = (C.c_double * 3)(), (C.c_longlong * 3)()
    _lib.check(lib.hn_match_profile_enable(1), "hn_match_profile_enable")
    for _ in range(n):
        fn()
    _lib.check(lib.hn_match_profile_read(ms, cnt), "hn_match_profile_read")
    lib.hn_match_profile_enable(0)
    # per call: a stage may run more than once per call (packing of q and g in separate brackets) or not at all
    return {k: ms[i] / n for i, k in enumerate(("pack", "gemm", "rerank"))}


def peak_bytes(fn):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    out = fn()
    torch.cuda.synchronize()
    del out
    return torch.cuda.max_memory_allocated() - base


def _flat(x):
    return [t for t in (x if isinstance(x, (tuple, list)) else [x]) if isinstance(t, torch.Tensor)]


def identical(a, b):
    return all(torch.equal(x, y) for x, y in zip(_flat(a), _flat(b)))


def run_workload(name, kind, data32, a, lib):
    inputs = {dt: with_rows(kind, data32, [r.to(t) for r in rows_of(kind, data32)]) for dt, t in DTYPES.items()}
    entry = {"workload": name, "kind": kind,
             "rows": sum(r.shape[0] * (r.shape[1] if r.dim() == 3 else 1) for r in rows_of(kind, data32)),
             "input_bytes": {dt: sum(r.numel() * r.element_size() for r in rows_of(kind, d)) for dt, d in inputs.items()}}
    for form in ("top2", "mutual_ratio"):
        fns = {dt: python_call(kind, form, d) for dt, d in inputs.items()}
        fp16_rows = rows_of(kind, inputs["fp16"])
        fns["fp16_upcast"] = lambda: python_call(kind, form, with_rows(kind, data32, [r.float() for r in fp16_rows]))()
        for _ in range(2):
            for fn in fns.values():
                fn()
        torch.cuda.synchronize()
        times = {k: [] for k in fns}
        for _ in range(a.reps):          # alternate the forms
            for k, fn in fns.items():
                times[k].append(window(fn, a.calls))
        med = {k: statistics.median(v) for k, v in times.items()}
        res = {}
        for k, fn in fns.items():
            res[k] = {"ms": med[k], "ms_all": times[k], "spread": (max(times[k]) - min(times[k])) / med[k],
                      "peak_alloc_bytes": peak_bytes(fn)}
            if k in DTYPES:
                res[k]["stage_ms"] = stage_ms(lib, fn, a.calls)
        for dt in ("fp16", "bf16"):      # the 16-bit call against the fp32 call on its rows converted to fp32
            d = inputs[dt]
            res[dt]["equal_to_fp32_call_on_float"] = identical(fns[dt](), python_call(
                kind, form, with_rows(kind, d, [r.float() for r in rows_of(kind, d)]))())
        res["fp16_over_fp32"] = med["fp16"] / med["fp32"]
        res["bf16_over_fp32"] = med["bf16"] / med["fp32"]
        res["fp16_over_fp16_upcast"] = med["fp16"] / med["fp16_upcast"]
        entry[form] = res
    del inputs
    print(json.dumps({"workload": name, **{f: {k: (round(v["ms"], 4) if isinstance(v, dict) else round(v, 4))
                                                for k, v in entry[f].items()} for f in ("top2", "mutual_ratio")}}), flush=True)
    return entry


def load_lib(path):
    lib = C.CDLL(str(path))
    for name in ("hn_match_batched_workspace_bytes", "hn_match_batched", "hn_match_pairs_workspace_bytes", "hn_match_pairs",
                 "hn_pack_descriptors", "hn_dist_workspace_bytes", "hn_mutual_workspace_bytes", "hn_match_ex", "hn_match_mutual",
                 "hn_last_error"):
        res, args = _lib.SIGNATURES[name]
        getattr(lib, name).restype = res
        getattr(lib, name).argtypes = args
    return lib


def raw_call(lib, kind, data, mutual):
    """(call, outputs, keep-alive) of the fp32 entry point of `lib` on `data`."""
    P = lambda t: C.c_void_p(t.data_ptr() if t is not None else 0)  # noqa: E731
    if kind == "batched":
        Q, G, L1, L2 = data
        B, n = Q.size(0), Q.size(1)
        rows, ws_bytes = B * n, lib.hn_match_batched_workspace_bytes(B, n, G.size(1), int(mutual))
    elif kind == "pairs":
        X, T, mq, mg = data
        rows, ws_bytes = T.size(0) * mq, lib.hn_match_pairs_workspace_bytes(T.size(0), mq, mg, int(mutual))
        x16 = torch.empty(X.size(0), 128, dtype=torch.float16, device="cuda")
    else:
        q, g = data
        rows = q.size(0)
        ws_bytes = lib.hn_mutual_workspace_bytes(q.size(0), g.size(0)) if mutual else lib.hn_dist_workspace_bytes(q.size(0), g.size(0), 0)
    ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device="cuda")
    outs = [torch.empty(rows, dtype=t, device="cuda") for t in (torch.float32, torch.float32, torch.int32, torch.int32)]
    mu = torch.empty(rows, dtype=torch.uint8, device="cuda") if mutual else None
    o = [P(t) for t in outs] + [P(mu)]

    def check(st):
        if st != 0:
            raise RuntimeError(lib.hn_last_error().decode())

    if kind == "batched":
        def call():
            check(lib.hn_match_batched(P(Q), P(G), B, n, G.size(1), P(L1), P(L2), *o, P(ws), ws.numel(), None))
    elif kind == "pairs":
        def call():
            check(lib.hn_pack_descriptors(P(X), X.size(0), P(x16), None))
            check(lib.hn_match_pairs(P(X), P(x16), X.size(0), P(X), P(x16), X.size(0), P(T), T.size(0), mq, mg, *o, P(ws), ws.numel(),
                                     None))
    elif mutual:
        def call():
            check(lib.hn_match_mutual(P(q), P(g), None, None, q.size(0), g.size(0), *o, P(ws), ws.numel(), None))
    else:
        def call():
            check(lib.hn_match_ex(P(q), P(g), None, None, q.size(0), g.size(0), 0, *o[:4], None, P(ws), ws.numel(), None, None))
    return call, outs + ([mu] if mu is not None else [])


def ab_fp32(name, kind, data, parent, a):
    libs = {"this": load_lib(_lib.LIB_PATH), "parent": parent}
    entry = {"workload": name}
    for form, mutual in (("top2", False), ("mutual_ratio", True)):
        state = {k: raw_call(lib, kind, data, mutual) for k, lib in libs.items()}
        for _ in range(3):
            for call, _ in state.values():
                call()
        torch.cuda.synchronize()
        times = {k: [] for k in state}
        for _ in range(a.reps):
            for k, (call, _) in state.items():
                times[k].append(window(call, a.calls * 2))
        med = {k: statistics.median(v) for k, v in times.items()}
        e = {f"{k}_ms": med[k] for k in med}
        e.update({f"{k}_ms_all": v for k, v in times.items()})
        e.update({f"{k}_spread": (max(v) - min(v)) / med[k] for k, v in times.items()})
        e["this_over_parent"] = med["this"] / med["parent"]
        e["outputs_identical"] = identical(state["this"][1], state["parent"][1])
        entry[form] = e
        del state
    print(json.dumps({"ab": name, **{f: {k: round(v, 4) if isinstance(v, float) else v for k, v in entry[f].items()
                                          if not k.endswith("_all")} for f in ("top2", "mutual_ratio")}}), flush=True)
    return entry


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(REPO / "profiles" / "r5_match_16bit.json"))
    ap.add_argument("--calls", type=int, default=3)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--parent-lib", default=None, help="another build of libhardnet_b200.so for the fp32 A/B")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("match_16bit_time.py measures on the GPU: no CUDA device")
    lib = _lib.load()
    parent = load_lib(Path(a.parent_lib)) if a.parent_lib else None
    result = {"gpu": gpu_info(), "calls_per_window": a.calls, "windows": a.reps, "workloads": []}
    if parent is not None:
        result["ab_fp32"] = {"parent_lib": str(a.parent_lib), "workloads": []}
    for name, kind, data in workloads():
        result["workloads"].append(run_workload(name, kind, data, a, lib))
        if parent is not None:
            result["ab_fp32"]["workloads"].append(ab_fp32(name, kind, data, parent, a))
        del data
        torch.cuda.empty_cache()
    result["gpu_after"] = gpu_info()
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(result, indent=1) + "\n")
    print("wrote", a.out)


if __name__ == "__main__":
    main()

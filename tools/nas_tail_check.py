"""GPU check of the warpgroup-per-patch NAS tail kernel (csrc/nas_tail.cuh): parity against the CPU oracle and throughput
at batch 65 536 (BASELINE config 5) for several launch plans.

    python tools/nas_tail_check.py [--fast] [--timing-only]
"""
import json
import os
import sys
from pathlib import Path

import torch

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))

from hardnetnas_b200.nas import SampledDescriptorNet  # noqa: E402
from hardnetnas_b200.nas.fbnet_modeldef import arch_ops  # noqa: E402
from oracle import nas_oracle, synth  # noqa: E402

MIXED = ["ir_k3_e3_se", "ir_k5_s4", "ir_k3_s2_se", "ir_k5_e3", "ir_k3_s4_se", "ir_k3_e1_se"]
ENV_KEYS = ("HN_NAS_TAIL", "HN_NAS_TAIL_CUT", "HN_NAS_TAIL_WG", "HN_NAS_FRONT_DW", "HN_NAS_TAIL_MINOPS", "HN_NAS_FOLD")


def build(arch, env, **kw):
    """The net `arch` built under `env` (the switches are read in hn_create); every other switch of ENV_KEYS unset."""
    for k in ENV_KEYS:
        os.environ.pop(k, None)
    os.environ.update(env)
    ops = MIXED if arch == "mixed_se" else arch_ops(arch)
    torch.manual_seed(0)
    net = SampledDescriptorNet(ops, **kw)
    net.load_state_dict(synth.randomize_nas_state(net.state_dict(), 4))
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    return net.cuda().eval(), ops, sd


def parity(arch, env):
    """Descriptors and every stage output against the CPU oracle."""
    net, ops, sd = build(arch, env, chunk_patches=64, head_rows=256)
    plan = net.resident_plan()
    out = {"arch": arch, "env": env, "plan": plan}
    x = synth.make_patches(203, 6, edge_cases=False)
    ref, feats = nas_oracle.nas_forward(x, ops, sd, return_features=True)
    got = net(x.cuda()).float().cpu()
    out["desc_max_abs"] = (got - ref).abs().max().item()
    out["desc_min_cos"] = torch.nn.functional.cosine_similarity(got, ref, dim=1).min().item()
    prog = net.compile_program()
    worst = 0.0
    for stage, op_index in enumerate(prog.stage_end):
        g = net.forward_op(x[:37].cuda(), op_index).float().cpu().permute(0, 3, 1, 2)
        r = feats[stage][:37]
        worst = max(worst, (g - r).abs().max().item() / max(r.abs().max().item(), 1e-9))
    out["stage_rel_err_max"] = worst
    out["ok"] = bool(out["desc_max_abs"] <= 1e-3 and out["desc_min_cos"] >= 0.9999 and worst <= 6e-3)
    return out


def timing(arch, env, batch=65536, iters=5):
    """Forward throughput at `batch` patches (BASELINE config 5)."""
    net, ops, sd = build(arch, env)
    g = torch.Generator(device="cuda").manual_seed(9)
    x = torch.nn.functional.avg_pool2d(torch.rand((batch, 1, 32, 32), generator=g, device="cuda"), 5, 1, 2)
    for _ in range(2):
        y = net(x)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        y = net(x)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    return {"arch": arch, "env": env, "plan": net.resident_plan(), "ms": ms, "patches_per_sec": batch / ms * 1e3,
            "finite": bool(torch.isfinite(y).all())}


def main():
    fast = "--fast" in sys.argv
    ok = True
    plans = [{}, {"HN_NAS_FOLD": "0"}, {"HN_NAS_TAIL_CUT": "0"}, {"HN_NAS_TAIL_WG": "2"}]
    if "--timing-only" not in sys.argv:
        for arch in ("wang2", "wang3", "wang4", "mixed_se"):
            for env in (plans[:2] if fast else plans):
                try:
                    r = parity(arch, env)
                except Exception as exc:  # keep going: one broken plan must not hide the others
                    r = {"arch": arch, "env": env, "error": repr(exc), "ok": False}
                ok = ok and r["ok"]
                print("PARITY", json.dumps(r), flush=True)
    tplans = [{}, {"HN_NAS_TAIL_CUT": "0"}, {"HN_NAS_FOLD": "0"}, {"HN_NAS_TAIL": "0"}] if fast else \
        [{}, {"HN_NAS_TAIL_CUT": "0"}, {"HN_NAS_TAIL_WG": "3"}, {"HN_NAS_TAIL_WG": "2"}, {"HN_NAS_TAIL": "0"}]
    for arch in ("wang2", "wang3", "wang4"):
        for env in tplans:
            try:
                print("TIMING", json.dumps(timing(arch, env)), flush=True)
            except Exception as exc:
                print("TIMING", json.dumps({"arch": arch, "env": env, "error": repr(exc)}), flush=True)
    print("ALL_OK" if ok else "FAILED", flush=True)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())

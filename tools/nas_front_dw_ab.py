"""A/B of the front kernel with / without the fused stride-2 depthwise conv / max-pool (HN_NAS_FRONT_DW), parity + throughput."""
import os, sys
from pathlib import Path
import torch
REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))
from tools.nas_tail_check import build, timing  # noqa: E402
from oracle import nas_oracle, synth  # noqa: E402

for arch in ("wang2", "wang3", "wang4", "mixed_se"):
    net, ops, sd = build(arch, {"HN_NAS_FRONT_DW": "1"}, chunk_patches=64, head_rows=256)
    x = synth.make_patches(203, 6, edge_cases=False)
    ref, feats = nas_oracle.nas_forward(x, ops, sd, return_features=True)
    got = net(x.cuda()).float().cpu()
    prog = net.compile_program()
    worst = 0.0
    for stage, op_index in enumerate(prog.stage_end):
        g = net.forward_op(x[:37].cuda(), op_index).float().cpu().permute(0, 3, 1, 2)
        r = feats[stage][:37]
        worst = max(worst, (g - r).abs().max().item() / max(r.abs().max().item(), 1e-9))
    x8 = (synth.make_patches(150, 8, edge_cases=False) * 255).round().to(torch.uint8)
    e8 = (net(x8.cuda()).float().cpu() - nas_oracle.nas_forward(x8.float(), ops, sd)).abs().max().item()
    print("PARITY", arch, "max_abs %.2e cos %.7f stage_rel %.2e u8 %.2e" % ((got - ref).abs().max().item(),
          torch.nn.functional.cosine_similarity(got, ref, dim=1).min().item(), worst, e8), flush=True)
for arch in ("wang2", "wang3", "wang4"):
    for v in ("1", "0"):
        r = timing(arch, {"HN_NAS_FRONT_DW": v})
        print(f"TIMING {arch} front_dw={v}: {r['ms']:.3f} ms {r['patches_per_sec'] / 1e6:.2f} M/s", flush=True)

"""A/B of the fused conv3 + conv4 kernel (tc_conv34.cuh, mode 1 = the default) against the two separate kernels (mode 0,
HN_FUSE34=0): stage outputs and descriptors to the last fp16 bit (another accumulation order), then throughput and
per-stage times of both engines. Run on the GPU box; diagnostic, not a test.

    python tools/fuse34_check.py [modes ...]       # default: 0 1
"""
import os
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from oracle import synth  # noqa: E402
from hardnetnas_b200.hardnet import HardNet  # noqa: E402


def make(mode, chunk=0):
    os.environ["HN_FUSE34"] = str(mode)
    w, m, v = synth.hardnet_weights_from_seed(0, 3)
    torch.manual_seed(0)
    model = HardNet(chunk_patches=chunk)
    sd = model.state_dict()
    for i, bi in enumerate(synth.BN_IDX):
        sd[f"features.{bi}.running_mean"] = m[i]
        sd[f"features.{bi}.running_var"] = v[i]
    model.load_state_dict(sd)
    return model.cuda().eval()


def main():
    modes = [int(a) for a in sys.argv[1:] if not a.startswith("-")] or [0, 1]
    print(torch.cuda.get_device_name(0), flush=True)
    for n, chunk in (() if "--time-only" in sys.argv else ((2, 0), (301, 0), (4097, 0), (1000, 256), (18945, 0), (30001, 9472))):
        x = synth.make_patches(n, 77 + n).cuda()
        ref = None
        for mode in modes:
            model = make(mode, chunk)
            outs = {layer: model.forward_stage(x, layer) for layer in (3, 4, 5, 6)} if n <= model._engine_chunk() else {}
            outs["desc"] = model(x)
            torch.cuda.synchronize()
            if ref is None:
                ref = outs
                continue
            for k, v in outs.items():
                r = ref[k].float()
                d = (v.float() - r).abs()
                nbad = int((d > 0).sum())
                print(f"n={n} chunk={chunk} mode {mode} vs {modes[0]} {k}: max|diff| {d.max().item():.3e} (ref max {r.abs().max().item():.3f}) "
                      f"differing {nbad}/{d.numel()}", flush=True)
                if d.max().item() > 2e-2 * max(1.0, r.abs().max().item()):
                    bad = (d > 2e-2 * max(1.0, r.abs().max().item())).nonzero()
                    print("    first bad:", bad[:6].tolist(), "count", len(bad), flush=True)
    # throughput
    B = 148 * 128 * 8
    x = torch.randn(B, 1, 32, 32, device="cuda")
    out = torch.empty(B, 128, device="cuda")
    for mode in modes:
        model = make(mode)
        for _ in range(3):
            model(x, out=out)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        reps = 5
        for _ in range(reps):
            model(x, out=out)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        model.profile_enable(0x7f)
        model(x, out=out)
        st, nl = model.profile_read()
        model.profile_enable(0)
        print(f"mode {mode}: {B / ms / 1e3:.3f} M patches/s ({ms:.2f} ms per {B}); stage ns/patch "
              + " ".join(f"{model.STAGE_NAMES[i][:8]}={st[i] * 1e6 / B:.1f}" for i in range(1, 7)), flush=True)


HardNet._engine_chunk = lambda self: 148 * 128 if self._chunk_patches == 0 else self._chunk_patches

if __name__ == "__main__":
    main()

"""GPU parity of the NAS-derived descriptor nets (BASELINE config 5) against the CPU oracle and reference goldens."""
import numpy as np
import pytest
import torch

from hardnetnas_b200.nas import SampledDescriptorNet
from hardnetnas_b200.nas.fbnet_modeldef import arch_ops
from oracle import nas_oracle, synth

pytestmark = pytest.mark.gpu

MIXED = ["ir_k3_e3_se", "ir_k5_s4", "ir_k3_s2_se", "ir_k5_e3", "ir_k3_s4_se", "ir_k3_e1_se"]
DESC_MAX_ABS = 1e-3
DESC_MIN_COS = 0.9999


def build(arch, **kw):
    ops = MIXED if arch == "mixed_se" else arch_ops(arch)
    torch.manual_seed(0)
    net = SampledDescriptorNet(ops, **kw)
    net.load_state_dict(synth.randomize_nas_state(net.state_dict(), 4))
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    return net.cuda().eval(), ops, sd


def _cmp(got, ref):
    got = got.float().cpu()
    return (got - ref).abs().max().item(), torch.nn.functional.cosine_similarity(got, ref, dim=1).min().item()


@pytest.mark.parametrize("arch", ["wang2", "wang3", "wang4", "mixed_se"])
def test_stage_outputs_match_oracle(arch):
    net, ops, sd = build(arch)
    x = synth.make_patches(32, 1234, edge_cases=False)
    _, feats = nas_oracle.nas_forward(x, ops, sd, return_features=True)
    prog = net.compile_program()
    for stage, op_index in enumerate(prog.stage_end):
        got = net.forward_op(x.cuda(), op_index).float().cpu().permute(0, 3, 1, 2)
        ref = feats[stage]
        scale = ref.abs().max().item()
        err = (got - ref).abs().max().item()
        assert err <= 6e-3 * scale + 1e-5, f"{arch} stage {stage} (op {op_index}): err {err:.3e} scale {scale:.3e}"


@pytest.mark.parametrize("arch", ["wang2", "wang3", "wang4", "mixed_se"])
def test_descriptors_match_oracle_and_golden(arch, golden_dir):
    net, ops, sd = build(arch)
    x = synth.make_patches(32, 1234, edge_cases=False)
    got = net(x.cuda())
    ref = nas_oracle.nas_forward(x, ops, sd)
    max_abs, cos = _cmp(got, ref)
    assert max_abs <= DESC_MAX_ABS and cos >= DESC_MIN_COS, (max_abs, cos)
    gold = torch.from_numpy(np.load(golden_dir / "nas_forward.npz")[f"{arch}_desc"])
    max_abs, cos = _cmp(got, gold)
    assert max_abs <= DESC_MAX_ABS and cos >= DESC_MIN_COS, (max_abs, cos)


@pytest.mark.parametrize("batch", [1, 3, 127, 700])
def test_ragged_batches(batch):
    net, ops, sd = build("wang2", chunk_patches=64, head_rows=256)
    x = synth.make_patches(batch, 5, edge_cases=False)
    max_abs, cos = _cmp(net(x.cuda()), nas_oracle.nas_forward(x, ops, sd))
    assert max_abs <= DESC_MAX_ABS and cos >= DESC_MIN_COS, (max_abs, cos)


@pytest.mark.parametrize("front,dw", [("0", "1"), ("1", "0"), ("0", "0")])
def test_unfused_kernels_agree(front, dw, monkeypatch):
    """HN_NAS_FRONT=0 runs stem and first pointwise conv as two kernels instead of the fused front kernel; HN_NAS_DW_SMEM=0
    runs the register-strip depthwise kernel instead of the shared-memory one. Every combination reproduces the oracle
    (the defaults are covered by the tests above), also for a uint8 input and a ragged tail."""
    monkeypatch.setenv("HN_NAS_FRONT", front)
    monkeypatch.setenv("HN_NAS_DW_SMEM", dw)
    for arch in ("wang2", "wang3"):
        net, ops, sd = build(arch, chunk_patches=64, head_rows=256)
        x = synth.make_patches(203, 6, edge_cases=False)
        max_abs, cos = _cmp(net(x.cuda()), nas_oracle.nas_forward(x, ops, sd))
        assert max_abs <= DESC_MAX_ABS and cos >= DESC_MIN_COS, (arch, max_abs, cos)


def test_uint8_patches_through_the_fused_front():
    net, ops, sd = build("wang2", chunk_patches=64, head_rows=256)
    x8 = (synth.make_patches(150, 8, edge_cases=False) * 255).round().to(torch.uint8)
    max_abs, cos = _cmp(net(x8.cuda()), nas_oracle.nas_forward(x8.float(), ops, sd))
    assert max_abs <= DESC_MAX_ABS and cos >= DESC_MIN_COS, (max_abs, cos)


@pytest.mark.parametrize("arch", ["wang2", "mixed_se"])
def test_bf16_activations_looser_bound(arch):
    """bf16 activations (8-bit mantissa) through every NAS kernel: stated bound max-abs <= 1e-2, cosine >= 0.999 (the
    nets are ~20 ops deep; fp16 is the default and holds 1e-3)."""
    net, ops, sd = build(arch, act_dtype="bf16", chunk_patches=64, head_rows=256)
    x = synth.make_patches(131, 12, edge_cases=False)
    max_abs, cos = _cmp(net(x.cuda()), nas_oracle.nas_forward(x, ops, sd))
    assert max_abs <= 1e-2 and cos >= 0.999, (arch, max_abs, cos)


def test_config5_batch_64k_properties():
    """BASELINE config 5: wang2 at batch 65 536 — finite, unit norm, deterministic, equal to small-batch results."""
    net, ops, sd = build("wang2")
    x = synth.make_patches(65536, 9, edge_cases=False).cuda()
    d1 = net(x)
    d2 = net(x)
    assert torch.equal(d1, d2) and torch.isfinite(d1).all()
    assert (d1.norm(dim=1) - 1).abs().max().item() < 1e-3
    ref = nas_oracle.nas_forward(x[:256].cpu(), ops, sd)
    max_abs, cos = _cmp(d1[:256], ref)
    assert max_abs <= DESC_MAX_ABS and cos >= DESC_MIN_COS, (max_abs, cos)


def test_train_mode_is_stock_torch_and_cpu_eval_fails():
    from hardnetnas_b200._lib import HardnetB200Error
    net, _, _ = build("wang3")
    with pytest.raises(HardnetB200Error):
        net(synth.make_patches(4, 1))
    net.train()
    out = net(synth.make_patches(8, 1, edge_cases=False).cuda())
    assert out.requires_grad and out.shape == (8, 128)


@pytest.mark.parametrize("arch", ["wang2", "wang3", "wang4"])
def test_front_kernel_with_and_without_the_fused_depthwise_stage(arch, monkeypatch):
    """Default: the stride-2 depthwise conv (wang2: 3x3, wang3: 5x5) or max-pool (wang4) behind the stem runs inside the front
    kernel (the 64 KB/patch pointwise output stays in shared memory). HN_NAS_FRONT_DW=0 runs it as its own kernel. Both must
    reproduce the oracle at every stage, for fp32 and uint8 input and a ragged batch; bf16 nets never fuse it."""
    outs = []
    for flag in ("1", "0"):
        monkeypatch.setenv("HN_NAS_FRONT_DW", flag)
        net, ops, sd = build(arch, chunk_patches=64, head_rows=256)
        x = synth.make_patches(203, 6, edge_cases=False)
        ref, feats = nas_oracle.nas_forward(x, ops, sd, return_features=True)
        got = net(x.cuda())
        max_abs, cos = _cmp(got, ref)
        assert max_abs <= DESC_MAX_ABS and cos >= DESC_MIN_COS, (arch, flag, max_abs, cos)
        prog = net.compile_program()
        for stage, op_index in enumerate(prog.stage_end[:3]):
            g = net.forward_op(x[:37].cuda(), op_index).float().cpu().permute(0, 3, 1, 2)
            r = feats[stage][:37]
            assert (g - r).abs().max().item() <= 6e-3 * r.abs().max().item() + 1e-5, (arch, flag, stage)
        x8 = (synth.make_patches(150, 8, edge_cases=False) * 255).round().to(torch.uint8)
        max_abs, cos = _cmp(net(x8.cuda()), nas_oracle.nas_forward(x8.float(), ops, sd))
        assert max_abs <= DESC_MAX_ABS and cos >= DESC_MIN_COS, (arch, flag, "u8", max_abs, cos)
        outs.append(got)
    assert (outs[0].float() - outs[1].float()).abs().max().item() <= 5e-4


def test_default_plan_is_front_tail_head():
    """fp16 nets of expansion-1 blocks (every recorded architecture) run as fused front kernel + warpgroup-per-patch tail
    launches (csrc/nas_tail.cuh) + head GEMM; HN_NAS_TAIL=0, bf16 activations and wider blocks keep one kernel per op."""
    net, _, _ = build("wang2")
    # (packed op that produces the launch's first / last output, patches in flight per CTA, 0); folded form: the linear
    # convs 3, 6, 9, 12, 15 are gone (absorbed by ops 4, 7, 10, 13 and the head)
    assert net.resident_plan() == [(4, 8, 4, 0), (10, 14, 6, 0)]
    assert build("wang3")[0].resident_plan() == [(4, 8, 3, 0)]
    assert build("mixed_se")[0].resident_plan() == []
    assert build("wang2", act_dtype="bf16")[0].resident_plan() == []


@pytest.mark.parametrize("arch,env", [("wang2", {}), ("wang2", {"HN_NAS_FOLD": "0"}), ("wang2", {"HN_NAS_TAIL_CUT": "0"}), ("wang2", {"HN_NAS_TAIL_WG": "1"}),
                                      ("wang2", {"HN_NAS_TAIL_MINOPS": "1", "HN_NAS_TAIL_CUT": "1"}),
                                      ("wang2", {"HN_NAS_TAIL_MINOPS": "1", "HN_NAS_TAIL_CUT": "1", "HN_NAS_FOLD": "0"}), ("wang3", {}),
                                      ("wang3", {"HN_NAS_TAIL_MINOPS": "1"}), ("wang3", {"HN_NAS_FOLD": "0"}), ("wang4", {}),
                                      ("wang4", {"HN_NAS_TAIL_WG": "3", "HN_NAS_TAIL_MINOPS": "1"}), ("wang4", {"HN_NAS_FOLD": "0"})])
def test_tail_kernel_plans(arch, env, monkeypatch):
    """The tail kernel (IRFBlock pw -> dw -> pwl [+x] and Identity pool / 1x1 conv, fbnet_builder.py:455-570, :202-228, with the
    patch resident in shared memory; bias and second input added by the tensor core; parity layout in front of stride-2
    readers) under several launch plans, with the linear 1x1 convs folded into their consumers (default) and op by op
    (HN_NAS_FOLD=0): descriptors against the oracle for a ragged batch that leaves warpgroups without a patch, and the output
    of EVERY packed op (the dump runs the unfolded form cut short behind that op, incl. behind a parity-layout producer)
    against the one-kernel-per-op path and, at the block boundaries, against the oracle."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    net, ops, sd = build(arch, chunk_patches=64, head_rows=256)
    plan = net.resident_plan()
    assert plan and all(minb == 0 and 1 <= nwg <= 6 and b >= a for a, b, nwg, minb in plan), plan
    x = synth.make_patches(203, 6, edge_cases=False)
    ref, feats = nas_oracle.nas_forward(x, ops, sd, return_features=True)
    max_abs, cos = _cmp(net(x.cuda()), ref)
    assert max_abs <= DESC_MAX_ABS and cos >= DESC_MIN_COS, (arch, plan, max_abs, cos)
    prog = net.compile_program()
    n_ops = len(prog.ops)
    xs = x[:37].cuda()
    outs = [net.forward_op(xs, i).float().cpu() for i in range(n_ops - 1)]
    for stage, op_index in enumerate(prog.stage_end):
        r = feats[stage][:37]
        assert (outs[op_index].permute(0, 3, 1, 2) - r).abs().max().item() <= 6e-3 * r.abs().max().item() + 1e-5, (arch, stage, op_index)
    monkeypatch.setenv("HN_NAS_TAIL", "0")
    base, _, _ = build(arch, chunk_patches=64, head_rows=256)
    assert base.resident_plan() == []
    for i in range(n_ops - 1):
        b = base.forward_op(xs, i).float().cpu()
        assert (outs[i] - b).abs().max().item() <= 6e-3 * b.abs().max().item() + 1e-5, (arch, plan, i)
    assert (net(x.cuda()).float() - base(x.cuda()).float()).abs().max().item() <= 5e-4


def test_tail_kernel_uint8_and_batch_one():
    net, ops, sd = build("wang2")
    x8 = (synth.make_patches(150, 8, edge_cases=False) * 255).round().to(torch.uint8)
    max_abs, cos = _cmp(net(x8.cuda()), nas_oracle.nas_forward(x8.float(), ops, sd))
    assert max_abs <= DESC_MAX_ABS and cos >= DESC_MIN_COS, (max_abs, cos)
    x = synth.make_patches(1, 3, edge_cases=False)
    max_abs, cos = _cmp(net(x.cuda()), nas_oracle.nas_forward(x, ops, sd))
    assert max_abs <= DESC_MAX_ABS and cos >= DESC_MIN_COS, (max_abs, cos)


def test_latency_table_on_the_engine(tmp_path):
    """lookup_table_builder.py:121-158 measured on this library's kernels (differential whole-net timing) and, as the reference
    does it, on the candidates' torch modules; the written file reads back."""
    from hardnetnas_b200.nas.lookup_table import LookUpTable
    cands = ["skip", "ir_k3_e1", "ir_k5_s2", "ir_k3_e3_se"]
    path = tmp_path / "lookup_table.txt"
    t = LookUpTable(candidate_blocks=cands, calulate_latency=True, path_to_file=path, cnt_of_runs=3, engine="b200")
    assert len(t.lookup_table_latency) == 6
    for row in t.lookup_table_latency:
        assert row["skip"] == 0.0 and all(np.isfinite(v) and 0.0 <= v < 50.0 for v in row.values()), row
    assert any(row["ir_k3_e3_se"] > 0.0 for row in t.lookup_table_latency)
    assert LookUpTable(candidate_blocks=cands, path_to_file=path).lookup_table_latency == t.lookup_table_latency
    tt = LookUpTable(candidate_blocks=cands[:2], calulate_latency=True, cnt_of_runs=2, engine="torch")
    assert all(v > 0.0 and np.isfinite(v) for row in tt.lookup_table_latency for v in row.values())

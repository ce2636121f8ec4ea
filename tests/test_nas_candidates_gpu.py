"""Every NAS candidate block at every searched layer on the B200 kernels, against the float64 oracle (oracle/nas_oracle.py).

The nets are the ones a search can produce: each block of CANDIDATE_BLOCKS (and the e6 blocks hn_pack_nas accepts) at each
layer with `skip` elsewhere, the all-`skip` net, and seeded full architectures (oracle/nas_cases.py). hn_pack_nas picks the
front-kernel variant, the depthwise kernel, the GEMM tiling, the pass size and the tail / fold plan from the net's shapes,
so these cases run every such choice; tests/test_nas_candidates_cpu.py checks the compiled programs on the CPU."""
import re

import pytest
import torch

from hardnetnas_b200._lib import HardnetB200Error
from hardnetnas_b200.nas.fbnet_builder import PRIMITIVES
from hardnetnas_b200.nas.lookup_table import CANDIDATE_BLOCKS, LookUpTable
from oracle import nas_cases, nas_oracle, synth

pytestmark = pytest.mark.gpu

FP16 = (1e-3, 0.9999)   # descriptor max-abs, min cosine (tests/test_nas_gpu.py)
BF16 = (1e-2, 0.999)
# Stage dumps: <= STAGE_REL max|ref| + 1e-5 (tests/test_nas_gpu.py). 6e-3 is ~12 unit roundoffs of fp16 (2^-11). A bf16 net
# rounds at the same places (16-bit operands and stored activations) with a 4x larger unit roundoff (2^-9), so its stages get
# the same 12 roundoffs: 2.4e-2. Measured: the bf16 stem output alone is off by 6.5e-3 of max|ref|, about 3 roundoffs
# (patch, folded weight, output).
STAGE_REL_FP16 = 6e-3
STAGE_REL_BF16 = STAGE_REL_FP16 * 2 ** -9 / 2 ** -11
SMALL = dict(chunk_patches=64, head_rows=256)   # 203 patches = 4 passes (the last one ragged) and 1 head launch

X = synth.make_patches(203, 6, edge_cases=False)
N_DUMP = 37
_ORACLE = {}


def _ids(cases):
    return [nas_cases.case_id(ops) for ops in cases]


def _oracle(ops, sd, x=X, key="x"):
    """float64 oracle (descriptors, stage features of the first N_DUMP patches), once per architecture and input."""
    k = (tuple(ops), key)
    if k not in _ORACLE:
        ref, feats = nas_oracle.nas_forward(x.double(), ops, nas_oracle.state_dict_f64(sd), return_features=True)
        _ORACLE[k] = (ref, [f[:N_DUMP] for f in feats])
    return _ORACLE[k]


def _cmp(got, ref):
    got = got.double().cpu()
    return (got - ref).abs().max().item(), torch.nn.functional.cosine_similarity(got, ref, dim=1).min().item()


def _check(net, ops, sd, gate, what="", stage_rel=STAGE_REL_FP16):
    """Descriptors of X against the oracle under `gate`, and the forward_op dump at every stage_end against the oracle's
    features (<= stage_rel max|ref| + 1e-5). Returns (descriptor max-abs, min cosine)."""
    ref, feats = _oracle(ops, sd)
    max_abs, cos = _cmp(net(X.cuda()), ref)
    prog = net.compile_program()
    xs = X[:N_DUMP].cuda()
    for stage, op_index in enumerate(prog.stage_end):
        got = net.forward_op(xs, op_index).double().cpu().permute(0, 3, 1, 2)
        r = feats[stage]
        err = (got - r).abs().max().item()
        assert err <= stage_rel * r.abs().max().item() + 1e-5, (what, stage, op_index, err, r.abs().max().item())
    assert max_abs <= gate[0] and cos >= gate[1], (what, max_abs, cos)
    return max_abs, cos


# ---- a / b / c: the sweep, fp16 and bf16 -------------------------------------------------------------------------------
@pytest.mark.parametrize("ops", nas_cases.SWEEP, ids=_ids(nas_cases.SWEEP))
def test_sweep_fp16(ops, record_property):
    """Default settings. The plan holds tail launches exactly for nets of expansion-1 blocks without SE (and skip): there
    layer 0 leaves the 32 x 32 x 32 map whose stride-2 depthwise conv / max-pool the front kernel fuses, and every later op
    has a tail shape. SE ops, the e3 / s4 / e6 widths and a layer-0 block without that fused stage keep one kernel per op."""
    net, sd = nas_cases.build(ops, **SMALL)
    max_abs, cos = _check(net.cuda(), ops, sd, FP16)
    record_property("desc_max_abs", max_abs)
    record_property("desc_min_cos", cos)
    plan = net.resident_plan()
    assert bool(plan) == nas_cases.expects_tail(ops), plan


@pytest.mark.parametrize("ops", nas_cases.SWEEP, ids=_ids(nas_cases.SWEEP))
def test_sweep_bf16(ops, record_property):
    """bf16 activations never fuse the front depthwise stage nor run the tail kernel: the fp32-math depthwise kernels and
    one kernel per op at every shape."""
    net, sd = nas_cases.build(ops, act_dtype="bf16", **SMALL)
    max_abs, cos = _check(net.cuda(), ops, sd, BF16, stage_rel=STAGE_REL_BF16)
    record_property("desc_max_abs", max_abs)
    record_property("desc_min_cos", cos)
    assert net.resident_plan() == []


# ---- d: switches ----------------------------------------------------------------------------------------------------------
def _switch_cases():
    cases = []
    for ops in nas_cases.SWEEP:
        cases.append((ops, "HN_NAS_DW_SMEM", "0"))
        cases.append((ops, "HN_NAS_DW_F32", "1"))
    for ops in nas_cases.SWEEP:   # 5x5 stride-1 depthwise convs: the 8-row strips
        if any(ops[l].startswith("ir_k5") for l in (1, 3)):
            cases.append((ops, "HN_NAS_DW_SH8", "0"))
    for ops in nas_cases.SWEEP:   # what sits behind the stem: fused pointwise, fused depthwise / max-pool
        if ops[1:] == ["skip"] * 5:
            cases.append((ops, "HN_NAS_FRONT", "0"))
            cases.append((ops, "HN_NAS_FRONT_DW", "0"))
    return cases


SWITCH_CASES = _switch_cases()


@pytest.mark.parametrize("ops,var,value", SWITCH_CASES, ids=[f"{nas_cases.case_id(o)}-{v}={x}" for o, v, x in SWITCH_CASES])
def test_switch_fp16(ops, var, value, monkeypatch):
    monkeypatch.setenv(var, value)
    net, sd = nas_cases.build(ops, **SMALL)
    _check(net.cuda(), ops, sd, FP16, f"{var}={value}")
    plan = net.resident_plan()
    if var in ("HN_NAS_FRONT", "HN_NAS_FRONT_DW"):   # the tail kernel runs only behind the fused front depthwise stage
        assert plan == []
    else:
        assert bool(plan) == nas_cases.expects_tail(ops), plan


TAIL_CASES = [ops for ops in nas_cases.SWEEP if nas_cases.expects_tail(ops)] + nas_cases.ARCHS_E1 + nas_cases.FOLD_CORNERS


@pytest.mark.parametrize("ops", TAIL_CASES, ids=_ids(TAIL_CASES))
def test_tail_nets_against_the_per_op_path(ops, monkeypatch):
    """Nets that run tail launches: the output of EVERY packed op (the dump runs the unfolded tail cut short behind that op)
    against the HN_NAS_TAIL=0 net, and the descriptors of the HN_NAS_TAIL=0 and HN_NAS_FOLD=0 nets against the oracle."""
    net, sd = nas_cases.build(ops, **SMALL)
    net = net.cuda()
    _check(net, ops, sd, FP16)
    assert net.resident_plan()
    n_ops = len(net.compile_program().ops)
    xs = X[:N_DUMP].cuda()
    outs = [net.forward_op(xs, i).float().cpu() for i in range(n_ops - 1)]
    d_tail = net(X.cuda()).float()
    monkeypatch.setenv("HN_NAS_FOLD", "0")
    unfolded, _ = nas_cases.build(ops, **SMALL)
    _check(unfolded.cuda(), ops, sd, FP16, "HN_NAS_FOLD=0")
    assert unfolded.resident_plan()
    monkeypatch.delenv("HN_NAS_FOLD")
    monkeypatch.setenv("HN_NAS_TAIL", "0")
    base, _ = nas_cases.build(ops, **SMALL)
    base = base.cuda()
    _check(base, ops, sd, FP16, "HN_NAS_TAIL=0")
    assert base.resident_plan() == []
    for i in range(n_ops - 1):
        b = base.forward_op(xs, i).float().cpu()
        assert (outs[i] - b).abs().max().item() <= 6e-3 * b.abs().max().item() + 1e-5, i
    assert (d_tail - base(X.cuda()).float()).abs().max().item() <= 5e-4


# ---- e: full architectures ------------------------------------------------------------------------------------------------
FULL = nas_cases.ARCHS_FULL + nas_cases.ARCHS_E1 + nas_cases.FOLD_CORNERS


@pytest.mark.parametrize("ops", FULL, ids=_ids(FULL))
def test_full_architecture(ops, record_property):
    net, sd = nas_cases.build(ops, **SMALL)
    max_abs, cos = _check(net.cuda(), ops, sd, FP16)
    record_property("desc_max_abs", max_abs)
    assert bool(net.resident_plan()) == nas_cases.expects_tail(ops)


# ---- f: uint8 patches through each front variant ------------------------------------------------------------------------
FRONTS = ["skip", "ir_k3_e1", "ir_k5_e1", "ir_k3_s2", "ir_k3_e3", "ir_k3_s4", "ir_k3_e1_se"]


@pytest.mark.parametrize("block", FRONTS)
def test_uint8_patches_through_the_front(block):
    """stem + fused pointwise (e1, and s2 with its shuffle-permuted block-diagonal weights) or stem alone (skip, e3, s4,
    e1_se), with and without the fused stride-2 stage, on uint8 input (each byte's value, as x8.float() gives it)."""
    ops = nas_cases.single(0, block)
    net, sd = nas_cases.build(ops, **SMALL)
    x8 = (synth.make_patches(150, 8, edge_cases=False) * 255).round().to(torch.uint8)
    ref, _ = _oracle(ops, sd, x8.float(), key="u8")
    max_abs, cos = _cmp(net.cuda()(x8.cuda()), ref)
    assert max_abs <= FP16[0] and cos >= FP16[1], (max_abs, cos)


# ---- g: passes capped by the 4 GiB slot budget ----------------------------------------------------------------------------
@pytest.mark.parametrize("block,pass_patches", [("ir_k3_s4", 5460), ("ir_k5_e3", 7280)])
def test_capped_passes(block, pass_patches):
    """Layer 0 = s4 (128 x 32 x 32 per patch) or e3 (96 x 32 x 32): a pass holds min(chunk, 4 GiB / (6 slot_elems)) & ~1
    patches, not a multiple of 128. 12 001 patches are two or more full passes plus a ragged one; every row against the fp32
    oracle (within 1.4e-7 of float64 for these nets)."""
    ops = nas_cases.single(0, block)
    net, sd = nas_cases.build(ops)
    net = net.cuda()
    x = synth.make_patches(12001, 21, edge_cases=False)
    net.forward_op(x[:pass_patches].cuda(), 1)   # a dump is one pass: the pass size is exactly pass_patches
    with pytest.raises(HardnetB200Error, match=f"chunk={pass_patches}"):
        net.forward_op(x[:pass_patches + 1].cuda(), 1)
    ref = torch.cat([nas_oracle.nas_forward(x[i:i + 1024], ops, sd) for i in range(0, x.size(0), 1024)]).double()
    xc = x.cuda()
    max_abs, cos = _cmp(net(xc), ref)
    assert max_abs <= FP16[0] and cos >= FP16[1], (max_abs, cos)
    out = torch.full((x.size(0), 128), float("nan"), dtype=torch.float16, device="cuda")
    assert net(xc, out=out) is out
    max_abs, cos = _cmp(out, ref)
    # + the output rounding: half an fp16 ulp of a unit-norm descriptor's entries (|v| < 1)
    assert max_abs <= FP16[0] + 2 ** -12 and cos >= FP16[1], (max_abs, cos)


# ---- h: the nets LookUpTable(engine="b200") times ------------------------------------------------------------------------
LATENCY = [nas_cases.single(0, "skip")] + [nas_cases.single(l, b) for l in range(6) for b in CANDIDATE_BLOCKS if b != "skip"]


@pytest.mark.parametrize("ops", LATENCY, ids=_ids(LATENCY))
def test_latency_table_nets(ops):
    """LookUpTable._calculate_latency's configuration: chunk_patches=1024, head_rows=1024, batch 1000, a preallocated out."""
    net, sd = nas_cases.build(ops, chunk_patches=1024, head_rows=1024)
    x = synth.make_patches(1000, 17, edge_cases=False)
    out = torch.empty((1000, 128), device="cuda")
    net.cuda()(x.cuda(), out=out)
    rows = torch.cat([torch.arange(128), torch.arange(1000 - 128, 1000)])
    ref, _ = _oracle(ops, sd, x[rows], key="latency")
    max_abs, cos = _cmp(out[rows.cuda()], ref)
    assert max_abs <= FP16[0] and cos >= FP16[1], (max_abs, cos)


def test_latency_table_covers_the_candidates():
    """The nets above are the ones LookUpTable builds: the same layer parameters and candidate names."""
    t = LookUpTable()
    assert list(t.lookup_table_operations) == CANDIDATE_BLOCKS
    assert len(LATENCY) == 1 + t.cnt_layers * (len(CANDIDATE_BLOCKS) - 1)


# ---- i: e6 at the last layer --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("block", nas_cases.E6_BLOCKS)
def test_e6_at_the_last_layer_is_rejected(block):
    """128 -> 768 channels is past the pointwise GEMM's 512: hn_pack_nas names the op and the forward returns nothing. The
    same object then packs and runs a valid net."""
    ops = nas_cases.single(5, block)
    net, _ = nas_cases.build(ops, **SMALL)
    net = net.cuda()
    bad = next(i for i, o in enumerate(net.compile_program().ops) if o.kind == 1 and o.cout > 512)
    out = torch.full((8, 128), 7.0, device="cuda")
    with pytest.raises(HardnetB200Error, match=re.escape(f"hn_pack_nas: op {bad} (kind 1) failed validation")):
        net(X[:8].cuda(), out=out)
    assert (out == 7.0).all()
    with pytest.raises(HardnetB200Error, match="failed validation"):   # still rejected, nothing stale is run instead
        net(X[:8].cuda())
    net.stages[5] = PRIMITIVES["ir_k3_e3"](128, 128, -999, 1).cuda().eval()
    net.op_names[5] = "ir_k3_e3"
    valid = nas_cases.single(5, "ir_k3_e3")
    sd = {k: v.detach().cpu().clone() for k, v in net.state_dict().items()}
    ref = nas_oracle.nas_forward(X[:8].double(), valid, nas_oracle.state_dict_f64(sd))
    max_abs, cos = _cmp(net(X[:8].cuda()), ref)
    assert max_abs <= FP16[0] and cos >= FP16[1], (max_abs, cos)

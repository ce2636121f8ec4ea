"""Every NAS candidate block at every searched layer, on the CPU: the mirror modules and the compiled op program against the
float64 oracle (oracle/nas_oracle.py). A GPU failure of tests/test_nas_candidates_gpu.py on a case that passes here lies in
the kernels or the C++ planner, not in the host-side compiler."""
import pytest
import torch

from oracle import nas_cases, nas_oracle, synth

CASES = (nas_cases.SWEEP + nas_cases.E6_AT_LAST_LAYER + nas_cases.ARCHS_FULL + nas_cases.ARCHS_E1 + nas_cases.FOLD_CORNERS)
IDS = [nas_cases.case_id(ops) for ops in CASES]

# The blob hn_pack_nas receives is float32: every folded weight is the float32 product of the BatchNorm scale and the conv
# weight (a few float32 roundings, relative 2^-24 each, ~2e-7 together), over ~20 ops. Measured against the float64 oracle:
# 4.3e-8 on the descriptors, 2.2e-7 of max|feature| on the stage outputs. The gates leave 20x and 10x of that; a wrong
# permutation, a lost bias or a wrong layout moves them by 1e-3 and more.
PROG_DESC_MAX_ABS = 1e-6
PROG_STAGE_REL = 2e-6


@pytest.fixture(scope="module")
def patches():
    return synth.make_patches(16, 1234, edge_cases=False).double()


def _oracle64(ops, sd, x):
    return nas_oracle.nas_forward(x, ops, nas_oracle.state_dict_f64(sd), return_features=True)


@pytest.mark.parametrize("ops", CASES, ids=IDS)
def test_mirror_equals_oracle_in_float64(ops, patches):
    """SampledDescriptorNet.forward_torch (the module tree of fbnet_builder.py) and the functional oracle, both in float64."""
    net, sd = nas_cases.build(ops)
    ref, _ = _oracle64(ops, sd, patches)
    with torch.no_grad():
        got = net.double().forward_torch(patches)
    assert torch.isfinite(ref).all()
    err = (got - ref).abs().max().item()
    assert err <= 1e-10, err


@pytest.mark.parametrize("ops", CASES, ids=IDS)
def test_compiled_program_equals_oracle(ops, patches):
    """compile_program().ops + the parameter blob, run by a float64 interpreter that knows only the C ABI's op semantics,
    against the float64 oracle: descriptors, and the slot named by stage_end[i] against the oracle's feats[i]."""
    net, sd = nas_cases.build(ops)
    ref, feats = _oracle64(ops, sd, patches)
    prog = net.compile_program()
    blob = torch.cat(prog.params)
    assert blob.dtype == torch.float32 and blob.numel() == prog.n
    desc, outs = nas_oracle.run_program(patches, prog.ops, blob)
    assert len(prog.stage_end) == len(feats) == 7 and prog.stage_end == sorted(prog.stage_end)
    for stage, (op_index, f) in enumerate(zip(prog.stage_end, feats)):
        got = outs[op_index]
        assert got.shape == f.shape, (stage, op_index, tuple(got.shape), tuple(f.shape))
        err = (got - f).abs().max().item()
        assert err <= PROG_STAGE_REL * f.abs().max().item(), (stage, op_index, err)
    err = (desc - ref).abs().max().item()
    assert err <= PROG_DESC_MAX_ABS, err


def test_case_lists_cover_the_search_space():
    """Every (layer, block) of CANDIDATE_BLOCKS, the e6 blocks at every layer, two lists of 24 full architectures."""
    from hardnetnas_b200.nas.lookup_table import CANDIDATE_BLOCKS
    pairs = {(l, ops[l]) for ops in nas_cases.SWEEP + nas_cases.E6_AT_LAST_LAYER for l in range(6)}
    assert pairs == {(l, b) for l in range(6) for b in CANDIDATE_BLOCKS + nas_cases.E6_BLOCKS}
    assert len(nas_cases.SWEEP) == 1 + 6 * 16 + 5 * 4
    assert len(nas_cases.ARCHS_FULL) == 24 and all(o in CANDIDATE_BLOCKS for a in nas_cases.ARCHS_FULL for o in a)
    assert len(nas_cases.ARCHS_E1) == 24 and all(o in nas_cases.E1_SPACE for a in nas_cases.ARCHS_E1 for o in a)
    assert len(set(IDS)) == len(IDS)

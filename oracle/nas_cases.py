"""NAS architectures the candidate tests run (tests/test_nas_candidates_{cpu,gpu}.py) — test infrastructure only.

Every list is written out literally so that a failing case can be rebuilt by name."""
from __future__ import annotations

import torch

from hardnetnas_b200.nas import SampledDescriptorNet
from hardnetnas_b200.nas.fbnet_builder import PRIMITIVES
from hardnetnas_b200.nas.lookup_table import CANDIDATE_BLOCKS

from . import synth

N_LAYERS = 6
E6_BLOCKS = ["ir_k3_e6", "ir_k3_e6_se", "ir_k5_e6", "ir_k5_e6_se"]   # in PRIMITIVES, not in CANDIDATE_BLOCKS
E1_SPACE = ["skip", "ir_k3_e1", "ir_k5_e1", "ir_k3_s2", "ir_k5_s2"]  # expansion-1 blocks without SE
assert sorted(CANDIDATE_BLOCKS + E6_BLOCKS) == sorted(PRIMITIVES)


def single(layer: int, block: str) -> list[str]:
    """`block` at `layer`, `skip` at the other five (the nets LookUpTable(engine="b200") times)."""
    ops = ["skip"] * N_LAYERS
    ops[layer] = block
    return ops


def case_id(ops) -> str:
    """'all_skip', 'L<layer>-<block>' for a single-candidate net, else the op names joined by '+'."""
    ops = list(ops)
    if ops == ["skip"] * N_LAYERS:
        return "all_skip"
    picked = [i for i, o in enumerate(ops) if o != "skip"]
    if len(picked) == 1:
        return f"L{picked[0]}-{ops[picked[0]]}"
    return "+".join(ops)


# every CANDIDATE_BLOCKS entry at every layer (skip everywhere = one net), plus the e6 blocks where hn_pack_nas takes them
SWEEP = ([["skip"] * N_LAYERS] + [single(l, b) for l in range(N_LAYERS) for b in CANDIDATE_BLOCKS if b != "skip"]
         + [single(l, b) for l in range(N_LAYERS - 1) for b in E6_BLOCKS])
E6_AT_LAST_LAYER = [single(N_LAYERS - 1, b) for b in E6_BLOCKS]     # 128 -> 768 channels: rejected by hn_pack_nas

# 24 draws from CANDIDATE_BLOCKS^6 with random.Random(20261021).choice
ARCHS_FULL = [
    ["ir_k5_s4_se", "skip", "ir_k5_s4_se", "ir_k5_s4_se", "ir_k5_e1_se", "ir_k3_e1_se"],
    ["ir_k3_s2_se", "ir_k5_s4_se", "ir_k5_s4_se", "skip", "ir_k3_e1_se", "skip"],
    ["ir_k3_e1", "ir_k3_e1", "ir_k3_s4", "ir_k5_s2", "ir_k3_s2", "ir_k3_e3"],
    ["ir_k3_s4", "ir_k3_s4_se", "ir_k3_e3_se", "ir_k5_e3", "ir_k5_e1", "ir_k5_e1"],
    ["ir_k3_s4", "ir_k3_e1", "ir_k3_s4", "ir_k3_e1", "ir_k3_e3_se", "ir_k5_e3"],
    ["ir_k5_e3_se", "skip", "ir_k5_e3_se", "ir_k3_e3_se", "ir_k5_s2_se", "ir_k3_s4"],
    ["ir_k5_e1", "ir_k3_s4", "ir_k3_s4_se", "ir_k5_s2", "ir_k3_e3", "ir_k3_s4"],
    ["ir_k5_s4", "ir_k5_s4_se", "ir_k3_s4", "ir_k5_s4_se", "ir_k3_s2", "ir_k5_s4"],
    ["skip", "ir_k5_e3", "ir_k5_e1_se", "ir_k3_e3_se", "skip", "ir_k3_e3"],
    ["ir_k3_e3_se", "ir_k5_s2_se", "ir_k3_e1_se", "ir_k5_e1_se", "ir_k3_e3_se", "ir_k5_e1_se"],
    ["ir_k5_e3", "ir_k3_e1", "ir_k5_s2_se", "ir_k3_e3_se", "ir_k3_e3_se", "ir_k3_e3"],
    ["ir_k5_s2_se", "ir_k5_e3_se", "ir_k3_e3", "ir_k5_s4", "ir_k3_s4_se", "ir_k3_e1_se"],
    ["ir_k5_s4", "ir_k3_e1", "skip", "ir_k5_s2", "ir_k5_s4", "ir_k5_e3"],
    ["ir_k5_e1", "ir_k5_e1", "ir_k5_s2_se", "ir_k3_s2_se", "ir_k5_s2_se", "ir_k5_e3_se"],
    ["ir_k5_e3", "ir_k3_s4_se", "ir_k3_s2", "ir_k3_e1_se", "ir_k3_s2_se", "ir_k5_s2_se"],
    ["ir_k5_e3_se", "ir_k5_s2", "ir_k3_e1", "ir_k5_e1", "ir_k5_s4_se", "ir_k3_e1_se"],
    ["ir_k3_e3_se", "ir_k3_s4_se", "ir_k5_e1", "ir_k5_e3_se", "ir_k5_s2", "ir_k3_e3"],
    ["ir_k3_e3_se", "ir_k5_s2", "ir_k5_e1_se", "ir_k5_e3", "ir_k3_e1_se", "ir_k5_e1_se"],
    ["ir_k3_e1", "ir_k5_s4", "ir_k5_e3_se", "ir_k3_e3_se", "ir_k5_s2_se", "skip"],
    ["ir_k5_e1", "ir_k5_s4", "ir_k3_s4", "ir_k3_e3_se", "ir_k3_e1", "ir_k5_s2_se"],
    ["ir_k3_e3", "ir_k3_e1_se", "ir_k3_s4", "ir_k3_s4", "ir_k3_s2", "ir_k5_e1_se"],
    ["ir_k5_s4_se", "ir_k5_e1_se", "ir_k5_s2_se", "ir_k3_e3_se", "ir_k5_e1_se", "ir_k5_e1_se"],
    ["ir_k3_s4", "ir_k3_e1", "ir_k3_e3_se", "ir_k3_e1", "ir_k5_s4_se", "ir_k5_s4"],
    ["ir_k3_s2_se", "ir_k3_s4_se", "ir_k3_e1_se", "skip", "ir_k5_e1_se", "ir_k5_s4_se"],
]

# 24 draws from E1_SPACE^6 with random.Random(20261022).choice: where tail launches and folding apply
ARCHS_E1 = [
    ["ir_k5_e1", "ir_k5_s2", "ir_k5_e1", "ir_k3_e1", "skip", "ir_k3_e1"],
    ["ir_k3_e1", "ir_k3_e1", "skip", "ir_k5_s2", "ir_k3_e1", "skip"],
    ["ir_k3_e1", "ir_k3_e1", "ir_k5_e1", "ir_k5_s2", "skip", "ir_k3_e1"],
    ["ir_k3_e1", "ir_k5_s2", "skip", "ir_k3_e1", "ir_k5_s2", "ir_k3_s2"],
    ["skip", "ir_k5_s2", "skip", "ir_k5_e1", "ir_k3_e1", "ir_k5_s2"],
    ["ir_k5_e1", "ir_k3_s2", "skip", "skip", "ir_k3_e1", "ir_k3_e1"],
    ["ir_k3_s2", "skip", "skip", "ir_k5_s2", "ir_k3_e1", "ir_k5_s2"],
    ["ir_k5_s2", "ir_k5_e1", "skip", "ir_k3_e1", "ir_k3_s2", "ir_k5_s2"],
    ["ir_k3_s2", "skip", "ir_k3_s2", "ir_k3_s2", "skip", "ir_k3_e1"],
    ["ir_k3_s2", "ir_k5_s2", "ir_k3_e1", "skip", "skip", "ir_k5_e1"],
    ["skip", "ir_k5_e1", "ir_k5_s2", "ir_k3_e1", "skip", "skip"],
    ["skip", "ir_k3_s2", "ir_k3_e1", "ir_k5_s2", "ir_k3_s2", "ir_k3_s2"],
    ["skip", "ir_k5_s2", "skip", "ir_k5_e1", "skip", "ir_k5_s2"],
    ["ir_k3_s2", "skip", "ir_k3_s2", "skip", "ir_k3_e1", "skip"],
    ["ir_k3_e1", "ir_k5_e1", "ir_k5_s2", "ir_k5_s2", "ir_k5_s2", "ir_k5_e1"],
    ["skip", "ir_k5_e1", "ir_k3_s2", "skip", "skip", "skip"],
    ["ir_k5_e1", "ir_k5_s2", "ir_k5_s2", "skip", "skip", "ir_k5_s2"],
    ["skip", "ir_k3_s2", "ir_k5_s2", "ir_k5_e1", "ir_k3_s2", "skip"],
    ["ir_k3_s2", "ir_k5_e1", "ir_k3_e1", "ir_k5_e1", "ir_k5_s2", "ir_k5_s2"],
    ["ir_k5_s2", "ir_k5_s2", "ir_k3_s2", "ir_k5_e1", "ir_k5_e1", "ir_k5_e1"],
    ["ir_k5_s2", "ir_k3_s2", "ir_k5_s2", "ir_k5_s2", "ir_k5_e1", "ir_k5_e1"],
    ["ir_k3_e1", "ir_k3_e1", "ir_k5_s2", "ir_k3_e1", "ir_k3_s2", "ir_k5_s2"],
    ["ir_k5_e1", "ir_k3_s2", "ir_k3_e1", "skip", "skip", "ir_k3_s2"],
    ["ir_k5_s2", "ir_k5_e1", "ir_k5_s2", "ir_k5_s2", "ir_k3_e1", "skip"],
]

# op graphs the tail / fold planner meets nowhere else
FOLD_CORNERS = [
    ["ir_k3_e1", "ir_k3_e1", "skip", "ir_k5_e1", "skip", "ir_k3_e1"],   # skip at layers 2 and 4 behind a linear (residual) pwl
    ["ir_k3_e1", "ir_k5_s2", "skip", "skip", "skip", "skip"],           # skip at layer 2 behind a linear s2 pwl
    ["ir_k3_s2", "ir_k5_s2", "skip", "skip", "skip", "skip"],           # s2 at layers 0 and 1
    ["skip", "ir_k3_e1", "skip", "ir_k5_e1", "skip", "ir_k3_e1"],       # residual e1 at layers 1, 3 and 5
]


def expects_tail(ops) -> bool:
    """fp16 nets whose ops behind the front stage all have a tail-kernel shape: expansion-1 blocks without SE (and skip), so
    that layer 0 leaves a 32 x 32 x 32 map whose stride-2 depthwise conv / max-pool runs inside the front kernel."""
    return all(o in E1_SPACE for o in ops)


def build(ops, **kw):
    """(eval net, its float32 state_dict): weights from torch.manual_seed(0), every BatchNorm from randomize_nas_state(4)."""
    torch.manual_seed(0)
    net = SampledDescriptorNet(list(ops), **kw)
    net.load_state_dict(synth.randomize_nas_state(net.state_dict(), 4))
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    return net.eval(), sd

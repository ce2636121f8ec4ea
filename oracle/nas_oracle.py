"""CPU restatement of the sampled NAS descriptor net — test infrastructure only (see oracle/__init__.py).

Follows hardnetNAS/supernet_functions/model_supernet.py:57-58,64-68,70-85 (stem, head, y/||y||) and, for the
searched layers, hardnetNAS/fbnet_building_blocks/fbnet_builder.py: Identity :202-228, ChannelShuffle :332-349,
ConvBNRelu :352-404, SEModule :407-421, IRFBlock :455-570, with the op table PRIMITIVES :36-155 and the layer
shapes SEARCH_SPACE2 (supernet_functions/lookup_table_builder.py:22-45).

Evaluated functionally from a state_dict whose keys are `first.*`, `stages.{i}.*`, `last_stages.*`
(the key layout of a MixedOperation's selected op with the `stages_to_search.{i}.ops.{k}.` prefix replaced).
"""
from __future__ import annotations

import re

import torch
import torch.nn.functional as F

LAYERS = [(32, 32, 2), (32, 32, 1), (32, 64, 2), (64, 64, 1), (64, 128, 2), (128, 128, 1)]  # (C_in, C_out, stride)
BN_EPS = 1e-5


def parse_op(name: str):
    """op name -> None for 'skip' or dict(kernel, expansion, group, shuffle, se) (fbnet_builder.py:36-155)."""
    if name == "skip":
        return None
    m = re.fullmatch(r"ir_k(\d)_(e(\d)|s(\d))(_se)?", name)
    assert m, f"unknown op {name}"
    kernel = int(m.group(1))
    if m.group(3):
        return dict(kernel=kernel, expansion=int(m.group(3)), group=1, shuffle=False, se=bool(m.group(5)))
    g = int(m.group(4))
    return dict(kernel=kernel, expansion=4 if g == 4 else 1, group=g, shuffle=True, se=bool(m.group(5)))


def _bn(x, sd, prefix, affine=True):
    w = sd[prefix + "weight"] if affine else None
    b = sd[prefix + "bias"] if affine else None
    return F.batch_norm(x, sd[prefix + "running_mean"], sd[prefix + "running_var"], w, b, False, 0.0, BN_EPS)


def _conv_bn(x, sd, prefix, stride=1, pad=0, groups=1, relu=True):
    y = F.conv2d(x, sd[prefix + "conv.weight"], None, stride=stride, padding=pad, groups=groups)
    y = _bn(y, sd, prefix + "bn.")
    return F.relu(y) if relu else y


def _shuffle(x, g):
    n, c, h, w = x.shape
    return x.view(n, g, c // g, h, w).permute(0, 2, 1, 3, 4).contiguous().view(n, c, h, w)


def _stage(x, sd, prefix, name, cin, cout, stride):
    spec = parse_op(name)
    if spec is None:                                   # Identity, fbnet_builder.py:202-228
        if stride != 1:
            x = F.max_pool2d(x, 3, 2, 1)
            if cin != cout:
                x = _conv_bn(x, sd, prefix + "conv.1.")
        elif cin != cout:
            x = _conv_bn(x, sd, prefix + "conv.")
        return x
    mid = cin * spec["expansion"]                      # IRFBlock, fbnet_builder.py:455-570
    y = _conv_bn(x, sd, prefix + "pw.", groups=spec["group"])
    if spec["shuffle"]:
        y = _shuffle(y, spec["group"])
    y = _conv_bn(y, sd, prefix + "dw.", stride=stride, pad=spec["kernel"] // 2, groups=mid)
    y = _conv_bn(y, sd, prefix + "pwl.", groups=spec["group"], relu=False)
    if stride == 1 and cin == cout:
        y = y + x
    if spec["se"]:                                     # SEModule, fbnet_builder.py:407-421
        s = F.adaptive_avg_pool2d(y, 1)
        s = F.relu(F.conv2d(s, sd[prefix + "se4.op.1.weight"], sd[prefix + "se4.op.1.bias"]))
        s = torch.sigmoid(F.conv2d(s, sd[prefix + "se4.op.3.weight"], sd[prefix + "se4.op.3.bias"]))
        y = y * s
    return y


def nas_forward(x: torch.Tensor, op_names, sd: dict, return_features: bool = False):
    """[B,1,32,32] -> [B,128]; NaN rows where the head output is exactly zero (torch.norm has no eps)."""
    with torch.no_grad():
        y = _conv_bn(x, sd, "first.", stride=1, pad=1)                     # model_supernet.py:57-58
        feats = [y]
        for i, (name, (cin, cout, stride)) in enumerate(zip(op_names, LAYERS)):
            y = _stage(y, sd, f"stages.{i}.", name, cin, cout, stride)
            feats.append(y)
        y = F.conv2d(y, sd["last_stages.conv_k1.weight"])                  # model_supernet.py:64-68
        y = _bn(y, sd, "last_stages.batchnorm.", affine=False)
        y = y.reshape(y.size(0), -1)
        y = y / torch.norm(y, p=2, dim=-1, keepdim=True)                   # model_supernet.py:84
    return (y, feats) if return_features else y


def state_dict_f64(sd: dict) -> dict:
    """The state_dict with every floating tensor in float64 (for nas_forward as a float64 reference)."""
    return {k: (v.double() if v.dtype.is_floating_point else v) for k, v in sd.items()}


OP_STEM, OP_PW, OP_DW, OP_MAXPOOL, OP_SE, OP_HEAD = 0, 1, 2, 3, 4, 5


def run_program(x: torch.Tensor, ops, params: torch.Tensor):
    """Float64 interpreter of exactly what hn_pack_nas receives: the `hn_nas_op` list of
    SampledDescriptorNet.compile_program() and the flat parameter blob (torch.cat(prog.params)). It knows nothing of the
    module tree, so it checks every host-side transformation in front of the C ABI (BatchNorm folding, shuffle folding,
    grouped-to-dense expansion, weight layouts, slot assignment).

    x [B,1,32,32] -> (descriptors [B,128], outs) with outs[i] the NCHW tensor in op i's dst slot after op i ran."""
    p = params.double()
    x = x.double()
    B = x.size(0)
    slots = [None, None, None]
    outs = []
    desc = None

    def take(off, n):
        assert 0 <= off and off + n <= p.numel(), "parameter range outside the blob"
        return p[off:off + n]

    with torch.no_grad():
        for o in ops:
            if o.kind == OP_STEM:                               # [9][32] taps-major, + shift, ReLU
                w = take(o.w_off, 9 * o.cout).view(9, o.cout).t().reshape(o.cout, 1, 3, 3)
                y = F.conv2d(x, w, take(o.b_off, o.cout), padding=1)
                y = F.relu(y) if o.relu else y
            elif o.kind == OP_PW:                               # dense [cout][cin] (+ res slot), optional ReLU
                w = take(o.w_off, o.cout * o.cin).view(o.cout, o.cin, 1, 1)
                y = F.conv2d(slots[o.src], w, take(o.b_off, o.cout))
                if o.res >= 0:
                    y = y + slots[o.res]
                y = F.relu(y) if o.relu else y
            elif o.kind == OP_DW:                               # [k*k][C], pad k // 2
                k = o.kernel
                w = take(o.w_off, k * k * o.cin).view(k * k, o.cin).t().reshape(o.cin, 1, k, k)
                y = F.conv2d(slots[o.src], w, take(o.b_off, o.cin), stride=o.stride, padding=k // 2, groups=o.cin)
                y = F.relu(y) if o.relu else y
            elif o.kind == OP_MAXPOOL:
                y = F.max_pool2d(slots[o.src], 3, 2, 1)
            elif o.kind == OP_SE:                               # fc1 [mid][C], fc2 [C][mid], in place
                v = slots[o.src]
                s = v.mean(dim=(2, 3))
                s = F.relu(s @ take(o.w_off, o.mid * o.cin).view(o.mid, o.cin).t() + take(o.b_off, o.mid))
                s = torch.sigmoid(s @ take(o.w2_off, o.cin * o.mid).view(o.cin, o.mid).t() + take(o.b2_off, o.cin))
                y = v * s[:, :, None, None]
            elif o.kind == OP_HEAD:                             # [128][(y*k + x)*C + c], + shift, L2 norm
                v = slots[o.src]
                assert v.shape[1:] == (o.cin, o.kernel, o.kernel)
                w = take(o.w_off, o.cout * o.kernel * o.kernel * o.cin).view(o.cout, -1)
                y = v.permute(0, 2, 3, 1).reshape(B, -1) @ w.t() + take(o.b_off, o.cout)
                desc = y / torch.norm(y, p=2, dim=-1, keepdim=True)
                outs.append(desc)
                continue
            else:
                raise ValueError(f"unknown op kind {o.kind}")
            assert y.shape[1:] == (o.cout, o.hout, o.hout), (o.kind, tuple(y.shape))
            slots[o.dst] = y
            outs.append(y)
    return desc, outs

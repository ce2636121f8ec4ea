"""Deployed (sampled) NAS descriptor net.

The reference search writes the argmax op of every MixedOperation into fbnet_modeldef.py
(hardnetNAS/supernet_main_file.py:105-108) but contains no class that builds the sampled descriptor net
(SURVEY.md §3.4). This module defines it exactly as the supernet does minus the mixing
(hardnetNAS/supernet_functions/model_supernet.py:57-58,64-68,70-85):

    first = ConvBNRelu(1 -> 32, k3, BN affine, ReLU)
    stages[i] = PRIMITIVES[op_i](*LookUpTable().layers_parameters[i])          (6 layers, SEARCH_SPACE2)
    last_stages = Conv2d(128, 128, k=4, no bias) -> BatchNorm2d(128, affine=False) -> Flatten
    y / ||y||_2     (no eps, no per-patch input normalisation)

eval() forward on CUDA tensors runs on the B200 kernels: the module tree is compiled into a flat op list
(BatchNorm folded, channel shuffles folded into the producing 1x1 conv, grouped 1x1 convs expanded to
block-diagonal dense matrices for the tensor cores) and handed to hn_pack_nas / hn_forward_nas.
train() forward is the stock torch path.
"""
from __future__ import annotations

import ctypes as C
from collections import OrderedDict

import torch
import torch.nn as nn

from .. import _lib
from ..hardnet import _Engine, _EngineOwner, _OUT_DTYPES
from .fbnet_builder import PRIMITIVES, ConvBNRelu, Flatten, IRFBlock, Identity
from .fbnet_modeldef import MODEL_ARCH, arch_ops
from .lookup_table import LookUpTable

OP_STEM, OP_PW, OP_DW, OP_MAXPOOL, OP_SE, OP_HEAD = 0, 1, 2, 3, 4, 5


class NasOp(C.Structure):
    """Mirror of `hn_nas_op` in include/hardnet_b200.h."""
    _fields_ = [("kind", C.c_int), ("cin", C.c_int), ("cout", C.c_int), ("kernel", C.c_int), ("stride", C.c_int),
                ("hin", C.c_int), ("hout", C.c_int), ("relu", C.c_int), ("src", C.c_int), ("dst", C.c_int),
                ("res", C.c_int), ("mid", C.c_int), ("w_off", C.c_longlong), ("b_off", C.c_longlong),
                ("w2_off", C.c_longlong), ("b2_off", C.c_longlong)]


def _fold_bn(conv: nn.Conv2d, bn: nn.BatchNorm2d | None):
    """Per-output-channel (scale, shift) of eval-mode BatchNorm following `conv` (which has no bias here)."""
    cout = conv.out_channels
    if bn is None:
        scale = torch.ones(cout)
        shift = torch.zeros(cout)
    else:
        inv = 1.0 / torch.sqrt(bn.running_var.detach().float().cpu() + bn.eps)
        gamma = bn.weight.detach().float().cpu() if bn.affine else torch.ones(cout)
        beta = bn.bias.detach().float().cpu() if bn.affine else torch.zeros(cout)
        scale = gamma * inv
        shift = beta - bn.running_mean.detach().float().cpu() * scale
    if conv.bias is not None:
        shift = shift + conv.bias.detach().float().cpu() * scale
    return scale, shift


def _dense_1x1(conv: nn.Conv2d) -> torch.Tensor:
    """[C_out, C_in] matrix of a (grouped) 1x1 conv; groups become diagonal blocks."""
    w = conv.weight.detach().float().cpu()[:, :, 0, 0]
    g = conv.groups
    cout, cin = conv.out_channels, conv.in_channels
    dense = torch.zeros(cout, cin)
    og, ig = cout // g, cin // g
    for k in range(g):
        dense[k * og:(k + 1) * og, k * ig:(k + 1) * ig] = w[k * og:(k + 1) * og]
    return dense


class _Program:
    def __init__(self):
        self.ops: list[NasOp] = []
        self.params: list[torch.Tensor] = []
        self.n = 0
        self.max_elems = 0
        self.stage_end: list[int] = []   # index of the op that produces the output of stem / each searched layer

    def blob(self, t: torch.Tensor) -> int:
        t = t.detach().float().cpu().contiguous().view(-1)
        pad = (-t.numel()) % 4            # keep every tensor 16-byte aligned in the blob
        off = self.n
        self.params.append(t)
        if pad:
            self.params.append(torch.zeros(pad))
        self.n += t.numel() + pad
        return off

    def add(self, **kw) -> NasOp:
        op = NasOp(**{k: int(v) for k, v in kw.items()})
        self.ops.append(op)
        for c, h in ((op.cin, op.hin), (op.cout, op.hout)):
            self.max_elems = max(self.max_elems, c * h * h)
        return op


class SampledDescriptorNet(_EngineOwner, nn.Module):
    def __init__(self, ops, act_dtype: str = "fp16", chunk_patches: int = 0, head_rows: int = 0):
        super().__init__()
        if isinstance(ops, str):
            ops = arch_ops(ops)
        table = LookUpTable()
        assert len(ops) == table.cnt_layers, f"expected {table.cnt_layers} op names"
        self.op_names = list(ops)
        self.first = ConvBNRelu(input_depth=1, output_depth=32, kernel=3, stride=1, pad=1, no_bias=1, use_relu="relu",
                                bn_type="bn")
        self.stages = nn.ModuleList([PRIMITIVES[name](*table.layers_parameters[i]) for i, name in enumerate(ops)])
        self.last_stages = nn.Sequential(OrderedDict([
            ("conv_k1", nn.Conv2d(table.layers_parameters[-1][1], 128, kernel_size=4, bias=False)),
            ("batchnorm", nn.BatchNorm2d(128, affine=False)),
            ("flatten", Flatten()),
        ]))
        self.act_dtype = act_dtype
        self._chunk_patches, self._head_rows = chunk_patches, head_rows
        self._engine: _Engine | None = None
        self._packed_key = None

    # ---- reference-equivalent torch path (training / definition) --------------------------------------
    def forward_torch(self, x):
        y = self.first(x)
        for st in self.stages:
            y = st(y)
        y = self.last_stages(y)
        return y / torch.norm(y, p=2, dim=-1, keepdim=True)

    def forward(self, x, out_dtype: torch.dtype = torch.float32, out: torch.Tensor | None = None):
        if self.training:
            return self.forward_torch(x)
        return self._forward_b200(x, out_dtype, out)

    def load_from_supernet(self, state_dict: dict, candidate_names: list[str]):
        """Copy the selected ops' weights out of an FBNet_Stochastic_SuperNet state_dict
        (keys `first.*`, `stages_to_search.{i}.ops.{k}.*`, `last_stages.*`)."""
        sd = {k[len("module."):] if k.startswith("module.") else k: v for k, v in state_dict.items()}
        mine = {}
        for k, v in sd.items():
            if k.startswith("first.") or k.startswith("last_stages."):
                mine[k] = v
        for i, name in enumerate(self.op_names):
            prefix = f"stages_to_search.{i}.ops.{candidate_names.index(name)}."
            for k, v in sd.items():
                if k.startswith(prefix):
                    mine[f"stages.{i}." + k[len(prefix):]] = v
        self.load_state_dict(mine)

    # ---- compiler: module tree -> op list ---------------------------------------------------------------
    def compile_program(self) -> _Program:
        prog = _Program()
        # stem: [tap][co] fp32 with the BN scale folded
        scale, shift = _fold_bn(self.first.conv, self.first.bn)
        w = self.first.conv.weight.detach().float().cpu().view(32, 9) * scale.view(-1, 1)
        prog.add(kind=OP_STEM, cin=1, cout=32, kernel=3, stride=1, hin=32, hout=32, relu=1, src=-1, dst=0, res=-1, mid=0,
                 w_off=prog.blob(w.t().contiguous()), b_off=prog.blob(shift), w2_off=0, b2_off=0)
        cur, h, c = 0, 32, 32
        prog.stage_end.append(0)

        def free_slots(*busy):
            return [s for s in range(3) if s not in busy]

        def pointwise(cbr: ConvBNRelu, src, dst, res, h, perm=None):
            conv = cbr.conv
            scale, shift = _fold_bn(conv, getattr(cbr, "bn", None))
            dense = _dense_1x1(conv) * scale.view(-1, 1)
            if perm is not None:                       # channel shuffle folded into the producer
                dense, shift = dense[perm], shift[perm]
            prog.add(kind=OP_PW, cin=conv.in_channels, cout=conv.out_channels, kernel=1, stride=1, hin=h, hout=h,
                     relu=int(hasattr(cbr, "relu")), src=src, dst=dst, res=res, mid=0,
                     w_off=prog.blob(dense), b_off=prog.blob(shift), w2_off=0, b2_off=0)

        for st in self.stages:
            if isinstance(st, Identity):
                mods = [] if st.conv is None else (list(st.conv) if isinstance(st.conv, nn.Sequential) and not isinstance(st.conv, ConvBNRelu) else [st.conv])
                for m in mods:
                    dst = free_slots(cur)[0]
                    if isinstance(m, nn.MaxPool2d):
                        prog.add(kind=OP_MAXPOOL, cin=c, cout=c, kernel=3, stride=2, hin=h, hout=h // 2, relu=0, src=cur,
                                 dst=dst, res=-1, mid=0, w_off=0, b_off=0, w2_off=0, b2_off=0)
                        h //= 2
                    else:
                        pointwise(m, cur, dst, -1, h)
                        c = m.conv.out_channels
                    cur = dst
            elif isinstance(st, IRFBlock):
                s1, s2 = free_slots(cur)
                perm = st.shuffle.source_channels(st.pw.conv.out_channels) if st.shuffle_type == "mid" else None
                pointwise(st.pw, cur, s1, -1, h, perm)
                mid = st.pw.conv.out_channels
                dw = st.dw.conv
                scale, shift = _fold_bn(dw, getattr(st.dw, "bn", None))
                k, stride = dw.kernel_size[0], dw.stride[0]
                wdw = dw.weight.detach().float().cpu().view(mid, k * k) * scale.view(-1, 1)
                prog.add(kind=OP_DW, cin=mid, cout=mid, kernel=k, stride=stride, hin=h, hout=h // stride,
                         relu=int(hasattr(st.dw, "relu")), src=s1, dst=s2, res=-1, mid=0,
                         w_off=prog.blob(wdw.t().contiguous()), b_off=prog.blob(shift), w2_off=0, b2_off=0)
                h //= stride
                pointwise(st.pwl, s2, s1, cur if st.use_res_connect else -1, h)
                c = st.output_depth
                cur = s1
                if isinstance(st.se4, nn.Module) and len(list(st.se4.children())) and hasattr(st.se4, "op"):
                    fc1, fc2 = st.se4.op[1], st.se4.op[3]
                    prog.add(kind=OP_SE, cin=c, cout=c, kernel=1, stride=1, hin=h, hout=h, relu=0, src=cur, dst=cur, res=-1,
                             mid=fc1.out_channels, w_off=prog.blob(fc1.weight.view(fc1.out_channels, c)),
                             b_off=prog.blob(fc1.bias), w2_off=prog.blob(fc2.weight.view(c, fc1.out_channels)),
                             b2_off=prog.blob(fc2.bias))
            else:
                raise TypeError(f"unsupported stage module {type(st).__name__}")
            prog.stage_end.append(len(prog.ops) - 1)
        # head: [co][(y*k + x)*C + ci], BN(affine=False) folded
        conv, bn = self.last_stages.conv_k1, self.last_stages.batchnorm
        scale, shift = _fold_bn(conv, bn)
        k = conv.kernel_size[0]
        assert h == k, "the head conv must cover the whole remaining feature map"
        wh = (conv.weight.detach().float().cpu() * scale.view(-1, 1, 1, 1)).permute(0, 2, 3, 1).contiguous().view(128, -1)
        prog.add(kind=OP_HEAD, cin=c, cout=128, kernel=k, stride=1, hin=h, hout=1, relu=0, src=cur, dst=-1, res=-1, mid=0,
                 w_off=prog.blob(wh), b_off=prog.blob(shift), w2_off=0, b2_off=0)
        return prog

    # ---- B200 path -------------------------------------------------------------------------------------
    def _ensure_packed(self, device):
        key = (device, self.act_dtype) + tuple((p._version, p.data_ptr()) for p in self.parameters()) + tuple(
            (b._version, b.data_ptr()) for b in self.buffers())
        if self._engine is None or self._engine.device != device:
            if self._engine is not None:
                self._engine.close()
            self._engine = _Engine(device, self._chunk_patches, self._head_rows)
            self._packed_key = None
        if self._packed_key == key:
            return
        prog = self.compile_program()
        ops = (NasOp * len(prog.ops))(*prog.ops)
        blob = torch.cat(prog.params).contiguous()
        eng = self._engine
        with torch.cuda.device(device):
            _lib.check(eng.lib.hn_pack_nas(eng.handle, ops, len(prog.ops), C.c_void_p(blob.data_ptr()), blob.numel(),
                                           _lib.HN_F16 if self.act_dtype == "fp16" else _lib.HN_BF16), "hn_pack_nas")
        self._packed_key = key

    def resident_plan(self, device=None):
        """[(first_op, last_op, patches_in_flight_per_cta, 0)] of the tail launches on `device`: runs of ops that execute
        patch-resident (one launch, activations in shared memory); ops outside every run are one kernel each."""
        device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self._ensure_packed(device)
        buf = (C.c_int * (4 * 32))()
        n = self._engine.lib.hn_nas_plan(self._engine.handle, buf, 32)
        if n < 0:
            _lib.check(n, "hn_nas_plan")
        return [tuple(buf[4 * i:4 * i + 4]) for i in range(n)]

    def forward_op(self, x, op_index: int):
        """Test hook: NHWC 16-bit output of op `op_index` of the compiled program, [B,H,W,C]."""
        self._ensure_packed(x.device)
        op = self.compile_program().ops[op_index]
        dt = torch.float16 if self.act_dtype == "fp16" else torch.bfloat16
        out = torch.empty((x.size(0), op.hout, op.hout, op.cout), dtype=dt, device=x.device)
        eng = self._engine
        with torch.cuda.device(x.device):
            stream = torch.cuda.current_stream().cuda_stream
            _lib.check(eng.lib.hn_forward_nas_dump(eng.handle, x.contiguous().data_ptr(), _lib.HN_F32, x.size(0), op_index,
                                                   out.data_ptr(), C.c_void_p(stream)), "hn_forward_nas_dump")
        return out

    def _forward_b200(self, x, out_dtype=torch.float32, out=None):
        if not isinstance(x, torch.Tensor) or not x.is_cuda:
            raise _lib.HardnetB200Error("SampledDescriptorNet eval forward runs on B200 CUDA tensors only (no CPU fallback)")
        if x.dim() != 4 or tuple(x.shape[1:]) != (1, 32, 32):
            raise ValueError(f"expected input of shape [B,1,32,32], got {tuple(x.shape)}")
        in_dt = _lib.HN_U8 if x.dtype == torch.uint8 else _lib.HN_F32
        x = x.contiguous() if x.dtype in (torch.uint8, torch.float32) else x.float().contiguous()
        self._ensure_packed(x.device)
        if out is None:
            out = torch.empty((x.size(0), 128), dtype=out_dtype, device=x.device)
        elif not (out.is_cuda and out.is_contiguous() and tuple(out.shape) == (x.size(0), 128) and out.dtype in _OUT_DTYPES):
            raise ValueError("out must be a contiguous CUDA [B,128] tensor of dtype float32 / float16 / bfloat16")
        eng = self._engine
        with torch.cuda.device(x.device):
            stream = torch.cuda.current_stream().cuda_stream
            _lib.check(eng.lib.hn_forward_nas(eng.handle, x.data_ptr(), in_dt, x.size(0), out.data_ptr(),
                                              _OUT_DTYPES[out.dtype], C.c_void_p(stream)), "hn_forward_nas")
        return out

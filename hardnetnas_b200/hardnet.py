"""Drop-in mirror of the reference's HardNet surface (hardnet/HardNet.py:275-324, hardnet/Utils.py:15-22).

`HardNet` keeps the reference's module tree, so `state_dict()` / `load_state_dict()` use the same keys
(`features.{0,3,...,19}.weight`, `features.{1,4,...,20}.running_{mean,var}`) and reference checkpoints
(`{'epoch', 'state_dict'}`, HardNet.py:440-441) load unchanged.

  * eval mode  -> the B200 kernels behind the C ABI (hn_pack_hardnet / hn_forward). CUDA tensors only;
                  there is no CPU fallback and a missing extension raises.
  * train mode -> the stock torch modules (batch-statistics BatchNorm and Dropout are training-time
                  behaviour and out of the accelerated path's scope).
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.nn as nn

from . import _lib

_DTYPES = {"fp16": _lib.HN_F16, "bf16": _lib.HN_BF16}
_OUT_DTYPES = {torch.float32: _lib.HN_F32, torch.float16: _lib.HN_F16, torch.bfloat16: _lib.HN_BF16,
               torch.float8_e4m3fn: _lib.HN_F8E4M3}


class L2Norm(nn.Module):
    """x / sqrt(sum(x*x, dim=1) + 1e-10) — hardnet/Utils.py:15-22."""

    def __init__(self):
        super().__init__()
        self.eps = 1e-10

    def forward(self, x):
        norm = torch.sqrt(torch.sum(x * x, dim=1) + self.eps)
        return x / norm.unsqueeze(-1).expand_as(x)


def weights_init(m):
    """Orthogonal init, gain 0.6, for every conv (hardnet/HardNet.py:317-324)."""
    if isinstance(m, nn.Conv2d):
        nn.init.orthogonal_(m.weight.data, gain=0.6)
        if m.bias is not None:
            nn.init.constant_(m.bias.data, 0.01)


class _Engine:
    """Owns one hn_handle on one CUDA device."""

    def __init__(self, device: torch.device, chunk_patches: int, head_rows: int):
        self.lib = _lib.load()
        self.device = device
        self.handle = C.c_void_p()
        with torch.cuda.device(device):
            _lib.check(self.lib.hn_create(C.byref(self.handle), int(chunk_patches), int(head_rows)), "hn_create")

    def close(self):
        if getattr(self, "handle", None) is not None and self.handle.value:
            self.lib.hn_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _EngineOwner:
    """Mixin of the modules that own an `_Engine` (a ctypes handle: neither picklable nor shareable).

    Copies made by copy.deepcopy / pickle / torch.save(model) / EMA-SWA wrappers and nn.DataParallel replicas drop the
    engine and re-create their own lazily on their first eval forward. `repack()` forces a fresh weight pack: the pack
    is keyed on the tensors' version counters and storage pointers, which in-place edits through `.data` (as the
    reference's weights_init does, hardnet/HardNet.py:317-324) do not change."""

    def __getstate__(self):
        state = self.__dict__.copy()
        state["_engine"] = None
        state["_packed_key"] = None
        return state

    def _replicate_for_data_parallel(self):
        replica = super()._replicate_for_data_parallel()
        replica._engine = None
        replica._packed_key = None
        return replica

    def repack(self):
        """Invalidate the packed weights (call after editing parameters or BatchNorm buffers through `.data`)."""
        self._packed_key = None
        return self


class HardNet(_EngineOwner, nn.Module):
    """HardNet model definition (same constructor contract as the reference: no required arguments)."""

    def __init__(self, act_dtype: str = "fp16", chunk_patches: int = 0, head_rows: int = 0):
        super().__init__()
        self.features = nn.Sequential(
            nn.Conv2d(1, 32, kernel_size=3, padding=1, bias=False),
            nn.BatchNorm2d(32, affine=False),
            nn.ReLU(),
            nn.Conv2d(32, 32, kernel_size=3, padding=1, bias=False),
            nn.BatchNorm2d(32, affine=False),
            nn.ReLU(),
            nn.Conv2d(32, 64, kernel_size=3, stride=2, padding=1, bias=False),
            nn.BatchNorm2d(64, affine=False),
            nn.ReLU(),
            nn.Conv2d(64, 64, kernel_size=3, padding=1, bias=False),
            nn.BatchNorm2d(64, affine=False),
            nn.ReLU(),
            nn.Conv2d(64, 128, kernel_size=3, stride=2, padding=1, bias=False),
            nn.BatchNorm2d(128, affine=False),
            nn.ReLU(),
            nn.Conv2d(128, 128, kernel_size=3, padding=1, bias=False),
            nn.BatchNorm2d(128, affine=False),
            nn.ReLU(),
            nn.Dropout(0.3),
            nn.Conv2d(128, 128, kernel_size=8, bias=False),
            nn.BatchNorm2d(128, affine=False),
        )
        self.features.apply(weights_init)
        if act_dtype not in _DTYPES:
            raise ValueError(f"act_dtype must be one of {sorted(_DTYPES)}")
        self.act_dtype = act_dtype
        self._chunk_patches = chunk_patches
        self._head_rows = head_rows
        self._engine: _Engine | None = None
        self._packed_key = None

    # ---- reference surface -------------------------------------------------------------------------
    INPUT_NORM_EPS = 1e-7    # hardnet/HardNet.py:309
    L2_EPS = 1e-10           # hardnet/Utils.py:18 (under the root)

    def input_norm(self, x):
        flat = x.view(x.size(0), -1)
        mp = torch.mean(flat, dim=1)
        sp = torch.std(flat, dim=1) + self.INPUT_NORM_EPS
        return (x - mp.detach().view(-1, 1, 1, 1)) / sp.detach().view(-1, 1, 1, 1)

    def forward(self, input, out_dtype: torch.dtype = torch.float32, out: torch.Tensor | None = None):
        if self.training:
            x_features = self.features(self.input_norm(input))
            x = x_features.view(x_features.size(0), -1)
            return L2Norm()(x)
        return self._forward_b200(input, out_dtype, out)

    def forward_stock(self, input):
        """The reference's own op sequence (HardNet.py:312-315) on whatever device the stock torch modules live on.
        Comparison arm for bench.py (cuDNN / cuBLAS on the same B200); never used by the accelerated path."""
        x_features = self.features(self.input_norm(input))
        x = x_features.view(x_features.size(0), -1)
        return L2Norm()(x)

    # ---- B200 path ---------------------------------------------------------------------------------
    def _convs_and_bns(self):
        convs = [m for m in self.features if isinstance(m, nn.Conv2d)]
        bns = [m for m in self.features if isinstance(m, nn.BatchNorm2d)]
        return convs, bns

    def _ensure_packed(self, device: torch.device):
        convs, bns = self._convs_and_bns()
        key = (device, self.act_dtype) + tuple(c.weight._version for c in convs) + tuple(
            (b.running_mean._version, b.running_var._version) for b in bns) + tuple(c.weight.data_ptr() for c in convs)
        if self._engine is None or self._engine.device != device:
            if self._engine is not None:
                self._engine.close()
            self._engine = _Engine(device, self._chunk_patches, self._head_rows)
            self._packed_key = None
        if self._packed_key == key:
            return
        ws = [c.weight.detach().to("cpu", torch.float32).contiguous() for c in convs]
        means = [b.running_mean.detach().to("cpu", torch.float32).contiguous() for b in bns]
        vars_ = [b.running_var.detach().to("cpu", torch.float32).contiguous() for b in bns]
        eng = self._engine
        with torch.cuda.device(device):
            _lib.check(eng.lib.hn_pack_hardnet(eng.handle, _lib.float_ptr_array(ws), _lib.float_ptr_array(means),
                                               _lib.float_ptr_array(vars_), C.c_float(bns[0].eps),
                                               _DTYPES[self.act_dtype]), "hn_pack_hardnet")
            _lib.check(eng.lib.hn_set_hardnet_eps(eng.handle, C.c_float(self.INPUT_NORM_EPS), C.c_float(self.L2_EPS)),
                       "hn_set_hardnet_eps")
        self._packed_key = key

    def _check_input(self, input):
        if not isinstance(input, torch.Tensor) or not input.is_cuda:
            raise _lib.HardnetB200Error(
                "HardNet eval forward runs on B200 CUDA tensors only (no CPU fallback); got a "
                f"{'CPU tensor' if isinstance(input, torch.Tensor) else type(input).__name__}")
        if input.dim() != 4 or tuple(input.shape[1:]) != (1, 32, 32):
            raise ValueError(f"expected input of shape [B,1,32,32], got {tuple(input.shape)}")
        if input.dtype == torch.float32:
            return input.contiguous(), _lib.HN_F32
        if input.dtype == torch.uint8:
            return input.contiguous(), _lib.HN_U8
        return input.float().contiguous(), _lib.HN_F32

    def _forward_b200(self, input, out_dtype=torch.float32, out=None):
        x, in_dt = self._check_input(input)
        self._ensure_packed(x.device)
        if out is None:
            out = torch.empty((x.size(0), 128), dtype=out_dtype, device=x.device)
        else:
            if out.shape != (x.size(0), 128) or out.device != x.device or not out.is_contiguous():
                raise ValueError("out must be a contiguous [B,128] tensor on the input's device")
            out_dtype = out.dtype
        eng = self._engine
        with torch.cuda.device(x.device):
            stream = torch.cuda.current_stream().cuda_stream
            _lib.check(eng.lib.hn_forward(eng.handle, x.data_ptr(), in_dt, x.size(0), out.data_ptr(),
                                          _OUT_DTYPES[out_dtype], C.c_void_p(stream)), "hn_forward")
        return out

    def forward_clip(self, kpts_byxc, kpts_scale, kpts_ori, im_info, images, out_dtype: torch.dtype = torch.float32):
        """`self(clip_patch(kpts_byxc, kpts_scale, kpts_ori, im_info, images, 32))` in one call (eval mode): the crop runs in the
        loader warps of the first conv kernel, so the [N,1,32,32] patch tensor is never materialised, and `images` may be uint8.
        Replaces the two calls of RFNetSO.inference (FDLNet-master/latency/rfnet/model/rf_net_so.py:160-180). Descriptors are
        bit-identical to the two-call form on `images.float()`."""
        if self.training:
            raise _lib.HardnetB200Error("forward_clip is the eval-mode path; in train mode call clip_patch and the module")
        if not (isinstance(images, torch.Tensor) and images.is_cuda):
            raise _lib.HardnetB200Error("forward_clip runs on B200 CUDA tensors only (no CPU fallback)")
        assert kpts_byxc.size(0) == kpts_scale.size(0)   # image_utils.py:22
        dev = images.device
        B, Cc, H, W = images.size()
        if Cc != 1:
            raise ValueError("forward_clip expects single-channel images [B,1,H,W] (the reference flattens them as such)")
        img_dt = _lib.HN_U8 if images.dtype == torch.uint8 else _lib.HN_F32
        img = images.detach().contiguous() if images.dtype == torch.uint8 else images.detach().to(torch.float32).contiguous()
        n = kpts_byxc.size(0)
        byxc = kpts_byxc.detach().to(device=dev, dtype=torch.int64).contiguous()
        scale = kpts_scale.detach().to(device=dev, dtype=torch.float32).contiguous().view(-1)
        ori = None if kpts_ori is None else kpts_ori.detach().to(device=dev, dtype=torch.float32).contiguous()
        info = im_info.detach().to(device=dev, dtype=torch.float32).contiguous()
        self._ensure_packed(dev)
        out = torch.empty((n, 128), dtype=out_dtype, device=dev)
        eng = self._engine
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream().cuda_stream
            _lib.check(eng.lib.hn_forward_clip(eng.handle, img.data_ptr(), img_dt, B, H, W, byxc.data_ptr(), scale.data_ptr(),
                                               None if ori is None else ori.data_ptr(), info.data_ptr(), n, out.data_ptr(),
                                               _OUT_DTYPES[out_dtype], C.c_void_p(stream)), "hn_forward_clip")
        return out

    # ---- measurement hooks (bench.py) ---------------------------------------------------------------
    # stage 0 (input_norm + conv1 on its own) only runs for activation dumps: the forward path fuses it into stage 1
    STAGE_NAMES = ("conv1_only_dump_path", "front_fused_norm_conv1_conv2", "conv3_s2_64", "conv4_64", "conv5_s2_128", "conv6_128",
                   "head_8x8_l2norm")
    # multiply-accumulates per patch of each stage (SURVEY.md §8a); stage 1 = a2 + a3
    STAGE_MACS = (294912, 294912 + 9437184, 4718592, 9437184, 4718592, 9437184, 1048576)

    @classmethod
    def stage_table(cls, launches):
        """(names, MACs per patch) of the seven timed stages for an engine whose per-stage launch counts are `launches`:
        with conv3 + conv4 fused into one kernel (csrc/tc_conv34.cuh, the default) stage 2 carries both layers and stage 3
        launches nothing."""
        names, macs = list(cls.STAGE_NAMES), list(cls.STAGE_MACS)
        if launches[2] > 0 and launches[3] == 0 and launches[4] > 0:
            names[2], macs[2] = "conv3_conv4_fused", macs[2] + macs[3]
            names[3], macs[3] = "conv4_64 (inside the fused kernel)", 0
        return names, macs

    def profile_enable(self, stage_mask: int):
        if self._engine is None:
            raise _lib.HardnetB200Error("profile_enable: run one eval forward first")
        _lib.check(self._engine.lib.hn_profile_enable(self._engine.handle, int(stage_mask)), "hn_profile_enable")

    def profile_read(self):
        """-> (ms per stage [7], launches per stage [7]); waits for the recorded events."""
        ms = (C.c_double * 7)()
        n = (C.c_longlong * 7)()
        _lib.check(self._engine.lib.hn_profile_read(self._engine.handle, ms, n), "hn_profile_read")
        return list(ms), list(n)

    def forward_stage(self, input, layer: int):
        """Test hook: NHWC activations after conv stage `layer` (1..6) as a [B,H,W,C] 16-bit tensor."""
        x, in_dt = self._check_input(input)
        self._ensure_packed(x.device)
        shapes = {1: (32, 32, 32), 2: (32, 32, 32), 3: (16, 16, 64), 4: (16, 16, 64), 5: (8, 8, 128), 6: (8, 8, 128)}
        dt = torch.float16 if self.act_dtype == "fp16" else torch.bfloat16
        out = torch.empty((x.size(0),) + shapes[layer], dtype=dt, device=x.device)
        eng = self._engine
        with torch.cuda.device(x.device):
            stream = torch.cuda.current_stream().cuda_stream
            _lib.check(eng.lib.hn_forward_dump(eng.handle, x.data_ptr(), in_dt, x.size(0), layer, out.data_ptr(),
                                               C.c_void_p(stream)), "hn_forward_dump")
        if layer == 1:
            return out
        # stages 2..6 are channel-planar on the device ([B][C/8][H][W][8]; stages feeding a stride-2 conv hold the
        # four row/column parity sub-planes [B][C/8][ypar][xpar][H/2][W/2][8]) -> NHWC for the caller
        H, W, Cc = shapes[layer]
        raw = out.view(-1)
        if layer in (2, 4):
            v = raw.view(x.size(0), Cc // 8, 2, 2, H // 2, W // 2, 8).permute(0, 4, 2, 5, 3, 1, 6)
        else:
            v = raw.view(x.size(0), Cc // 8, H, W, 8).permute(0, 2, 3, 1, 4)
        return v.reshape(x.size(0), H, W, Cc).contiguous()

"""clip_patch (FDLNet-master/utils/image_utils.py:11-158): oracle vs the reference-generated golden (CPU) and the
CUDA kernel behind hn_clip_patches vs the oracle (GPU)."""
import numpy as np
import pytest
import torch

from oracle import clip_oracle

TOL = 1e-5   # fp32 bilinear weights; the reference's stacked matmuls and the per-pixel form differ by ~2e-6


def test_oracle_matches_reference_golden(golden_dir):
    g = np.load(golden_dir / "clip_patch.npz")
    byxc, scale, ori, im_info, images = clip_oracle.make_clip_inputs()
    assert abs(images.double().sum().item() - float(g["images_sum"])) < 1e-6   # same seeded inputs
    out = clip_oracle.clip_patch(byxc, scale, ori, im_info, images, 32)
    assert out.shape == (byxc.size(0), 1, 32, 32)
    assert (out - torch.from_numpy(g["patches"])).abs().max().item() <= TOL
    out = clip_oracle.clip_patch(byxc, scale, None, im_info, images, 32)
    assert (out - torch.from_numpy(g["patches_no_ori"])).abs().max().item() <= TOL


@pytest.mark.gpu
@pytest.mark.parametrize("with_ori", [True, False])
def test_kernel_matches_oracle_and_golden(with_ori, golden_dir):
    from hardnetnas_b200.image_utils import clip_patch
    byxc, scale, ori, im_info, images = clip_oracle.make_clip_inputs()
    got = clip_patch(byxc.cuda(), scale.cuda(), ori.cuda() if with_ori else None, im_info.cuda(), images.cuda(), 32).cpu()
    ref = clip_oracle.clip_patch(byxc, scale, ori if with_ori else None, im_info, images, 32)
    assert got.shape == ref.shape
    assert (got - ref).abs().max().item() <= TOL
    gold = torch.from_numpy(np.load(golden_dir / "clip_patch.npz")["patches" if with_ori else "patches_no_ori"])
    assert (got - gold).abs().max().item() <= TOL


@pytest.mark.gpu
def test_kernel_larger_set_and_feeds_descriptor():
    """2048 keypoints over 8 images (other seed, other patch size), then straight into HardNet.forward."""
    from hardnetnas_b200.hardnet import HardNet
    from hardnetnas_b200.image_utils import clip_patch
    byxc, scale, ori, im_info, images = clip_oracle.make_clip_inputs(seed=5, B=8, H=240, W=320, k=256)
    for psize in (32, 17):
        got = clip_patch(byxc.cuda(), scale.cuda(), ori.cuda(), im_info.cuda(), images.cuda(), psize).cpu()
        ref = clip_oracle.clip_patch(byxc, scale, ori, im_info, images, psize)
        assert (got - ref).abs().max().item() <= TOL
    torch.manual_seed(0)
    model = HardNet().cuda().eval()
    desc = model(clip_patch(byxc.cuda(), scale.cuda(), ori.cuda(), im_info.cuda(), images.cuda(), 32))
    assert desc.shape == (2048, 128) and torch.isfinite(desc).all()


@pytest.mark.gpu
def test_cpu_tensors_fail_loudly():
    from hardnetnas_b200._lib import HardnetB200Error
    from hardnetnas_b200.image_utils import clip_patch
    byxc, scale, ori, im_info, images = clip_oracle.make_clip_inputs()
    with pytest.raises(HardnetB200Error):
        clip_patch(byxc, scale, ori, im_info, images, 32)


def _hardnet(**kw):
    """HardNet with the reference init and randomised BN statistics (oracle/synth.py), as the descriptor parity tests use."""
    from hardnetnas_b200.hardnet import HardNet
    from oracle import synth
    w, m, v = synth.hardnet_weights_from_seed(0, 3)
    torch.manual_seed(0)
    model = HardNet(**kw)
    sd = model.state_dict()
    for i, bi in enumerate(synth.BN_IDX):
        sd[f"features.{bi}.running_mean"] = m[i]
        sd[f"features.{bi}.running_var"] = v[i]
    model.load_state_dict(sd)
    return model.cuda().eval(), (w, m, v)


@pytest.mark.gpu
@pytest.mark.parametrize("with_ori", [True, False])
def test_forward_clip_is_bit_identical_to_clip_then_forward(with_ori):
    """hn_forward_clip (crop inside the front kernel's loader warps, no patch tensor) == hn_clip_patches + hn_forward, bit for
    bit; and against the CPU oracle of both steps within the descriptor tolerance of BASELINE.json (max-abs 1e-3). The small
    chunk makes the 2048 keypoints span several passes and head launches (keypoint offsets) with a ragged last pass."""
    from oracle import hardnet_oracle
    from hardnetnas_b200.image_utils import clip_patch
    byxc, scale, ori, im_info, images = clip_oracle.make_clip_inputs(seed=5, B=8, H=240, W=320, k=256)
    ori_c = ori.cuda() if with_ori else None
    for chunk in (0, 300):
        model, (w, m, v) = _hardnet(chunk_patches=chunk, head_rows=600 if chunk else 0)
        two = model(clip_patch(byxc.cuda(), scale.cuda(), ori_c, im_info.cuda(), images.cuda(), 32))
        one = model.forward_clip(byxc.cuda(), scale.cuda(), ori_c, im_info.cuda(), images.cuda())
        assert one.shape == (2048, 128)
        assert torch.equal(one, two)
    patches = clip_oracle.clip_patch(byxc, scale, ori if with_ori else None, im_info, images, 32)[:256]
    ref = hardnet_oracle.hardnet_forward(patches, w, m, v)
    assert (one[:256].cpu() - ref).abs().max().item() <= 1e-3


@pytest.mark.gpu
def test_forward_clip_uint8_images_and_bad_image_index():
    from hardnetnas_b200.image_utils import clip_patch
    byxc, scale, ori, im_info, images = clip_oracle.make_clip_inputs(seed=9, B=4, H=200, W=264, k=75)
    img8 = (images * 255).round().clamp(0, 255).to(torch.uint8)
    model, _ = _hardnet()
    two = model(clip_patch(byxc.cuda(), scale.cuda(), ori.cuda(), im_info.cuda(), img8.float().cuda(), 32))
    one = model.forward_clip(byxc.cuda(), scale.cuda(), ori.cuda(), im_info.cuda(), img8.cuda())
    assert torch.equal(one, two) and torch.isfinite(one).all()
    half = model.forward_clip(byxc.cuda(), scale.cuda(), ori.cuda(), im_info.cuda(), img8.cuda(), out_dtype=torch.float16)
    assert (half.float() - one).abs().max().item() <= 1e-3
    bad = byxc.clone()
    bad[7, 0] = 4          # image index out of range: NaN descriptor for that keypoint only, no out-of-bounds read
    out = model.forward_clip(bad.cuda(), scale.cuda(), ori.cuda(), im_info.cuda(), img8.cuda())
    assert torch.isnan(out[7]).all() and torch.equal(out[:7], one[:7]) and torch.equal(out[8:], one[8:])
    from hardnetnas_b200._lib import HardnetB200Error
    with pytest.raises(HardnetB200Error):
        model.train().forward_clip(byxc.cuda(), scale.cuda(), ori.cuda(), im_info.cuda(), img8.cuda())


@pytest.mark.gpu
def test_forward_clip_on_the_rf_net_descriptor():
    """RFNetSO.inference (FDLNet-master/latency/rfnet/model/rf_net_so.py:160-180) calls clip_patch and then its descriptor
    `self.des` = HardNetNeiMask (input_norm eps 1e-8, plain x / ||x|| head): the fused call carries both epsilons."""
    from hardnetnas_b200.image_utils import clip_patch
    from hardnetnas_b200.rf_des import HardNetNeiMask
    byxc, scale, ori, im_info, images = clip_oracle.make_clip_inputs(seed=3, B=2, H=96, W=128, k=40)
    torch.manual_seed(1)
    des = HardNetNeiMask(1.0, 8).cuda().eval()
    args = (byxc.cuda(), scale.cuda(), ori.cuda(), im_info.cuda(), images.cuda())
    two = des(clip_patch(*args, 32))
    one = des.forward_clip(*args)
    assert torch.equal(one, two) and torch.isfinite(one).all()
    assert (one.norm(dim=1) - 1).abs().max().item() <= 1e-5


def test_float_domain_clamp_gives_the_reference_taps():
    """csrc/clip.cuh clamps floor(x) in the float domain (fminf / fmaxf) where the reference clamps int64 indices
    (image_utils.py:98-112): same taps x0, x1 for every finite coordinate, incl. far outside the image and at integers."""
    rng = np.random.default_rng(0)
    for W in (1, 2, 17, 640, 4096):
        x = np.concatenate([rng.uniform(-3 * W - 5, 3 * W + 5, 20000), np.arange(-4, W + 4, dtype=np.float64),
                            np.array([-1e9, -2.0 ** 31, 2.0 ** 31, 1e9, 3e18, -3e18, -0.0, np.nextafter(0, -1), W - 1 - 1e-6])]).astype(np.float32)
        fx = np.floor(x)
        ref0 = np.clip(fx.astype(np.int64), 0, W - 1)
        ref1 = np.clip(fx.astype(np.int64) + 1, 0, W - 1)
        got0 = np.minimum(np.maximum(fx, np.float32(0)), np.float32(W - 1))
        got1 = np.minimum(np.maximum(fx + np.float32(1), np.float32(0)), np.float32(W - 1))
        assert np.array_equal(got0.astype(np.int64), ref0) and np.array_equal(got1.astype(np.int64), ref1)
        # the weights use the clamped taps as floats: identical values
        assert np.array_equal(got0, ref0.astype(np.float32)) and np.array_equal(got1, ref1.astype(np.float32))


def test_forward_clip_rejects_cpu_tensors_and_train_mode():
    from hardnetnas_b200._lib import HardnetB200Error
    from hardnetnas_b200.hardnet import HardNet
    byxc, scale, ori, im_info, images = clip_oracle.make_clip_inputs()
    model = HardNet().eval()
    with pytest.raises(HardnetB200Error):
        model.forward_clip(byxc, scale, ori, im_info, images)          # no CPU fallback
    with pytest.raises(HardnetB200Error):
        model.train().forward_clip(byxc, scale, ori, im_info, images)  # eval-mode path only


@pytest.mark.gpu
def test_forward_clip_with_several_passes():
    """A forward runs in passes of chunk_patches keypoints inside head launches of head_rows: the keypoint offset of every pass
    must follow (hardnet_forward.cu: input_at). 700 keypoints, passes of 200, head launches of 400 -> offsets 0, 200, 400, 600."""
    from hardnetnas_b200.image_utils import clip_patch
    byxc, scale, ori, im_info, images = clip_oracle.make_clip_inputs(seed=4, B=7, H=150, W=210, k=100)
    args = (byxc.cuda(), scale.cuda(), ori.cuda(), im_info.cuda(), images.cuda())
    ref_model, _ = _hardnet()
    want = ref_model(clip_patch(*args, 32))
    model, _ = _hardnet(chunk_patches=200, head_rows=400)
    assert torch.equal(model.forward_clip(*args), model(clip_patch(*args, 32)))
    assert (model.forward_clip(*args) - want).abs().max().item() <= 1e-4   # other pass sizes: same values up to the head's K split

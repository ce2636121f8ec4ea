"""HardNetNeiMask (FDLNet-master/latency/rfnet/model/rf_des.py:11-116): mirror class, oracle and CUDA path against
descriptors / losses produced by the unmodified reference class (oracle/make_golden_neimask.py)."""
import numpy as np
import pytest
import torch

from hardnetnas_b200.rf_des import HardNetNeiMask
from oracle import hardnet_oracle, synth
from oracle.make_golden_neimask import keypoints


def _model():
    torch.manual_seed(0)
    model = HardNetNeiMask(1.0, 8.0)
    model.load_state_dict(synth.randomize_bn_stats(model.state_dict(), 3))
    return model.eval()


def _inputs(g):
    x = synth.make_patches(64, 1234)
    x[5] = torch.from_numpy(g["x5"])
    return x


def _wmv(model):
    convs = [m for m in model.features if isinstance(m, torch.nn.Conv2d)]
    bns = [m for m in model.features if isinstance(m, torch.nn.BatchNorm2d)]
    return ([c.weight.detach() for c in convs], [b.running_mean for b in bns], [b.running_var for b in bns])


def test_mirror_regenerates_reference_weights_and_state_dict_keys(golden_dir):
    g = np.load(golden_dir / "neimask.npz")
    model = _model()
    w, m, v = _wmv(model)
    # orthogonal_ runs a LAPACK QR whose last bits depend on the host's CPU and thread count: bit for bit the mirror draws
    # what the reference recipe draws on this host, and the golden (another host) it matches to float32 rounding
    recipe = synth.hardnet_weights_from_seed(0, 3)[0]
    assert len(w) == len(recipe) and all(torch.equal(a, b) for a, b in zip(w, recipe))
    np.testing.assert_allclose(synth.weights_fingerprint(w), g["weights_fingerprint"], rtol=1e-5, atol=1e-6)
    assert np.array_equal(synth.weights_fingerprint(list(m) + list(v)), g["bn_fingerprint"])
    keys = set(model.state_dict().keys())
    assert "features.18.weight" in keys and "features.19.running_mean" in keys and not any(k.startswith("features.20") for k in keys)


def test_pairwise_distances_match_reference(golden_dir):
    from hardnetnas_b200.matching import pairwise_distances
    from oracle.make_golden_match_scores import inputs
    g = np.load(golden_dir / "match_scores.npz")
    _, _, kp1w, kp2, _ = inputs()
    assert np.allclose(pairwise_distances(kp1w[:16, 1:3], kp2[:24, 1:3]).numpy(), g["pairwise_16"], atol=1e-4)
    assert np.allclose(pairwise_distances(kp1w[:16, 1:3]).numpy(), g["pairwise_self_16"], atol=1e-2)   # sqrt near 0 on the diagonal


def test_oracle_and_train_mode_expressions_match_reference(golden_dir):
    g = np.load(golden_dir / "neimask.npz")
    model = _model()
    x = _inputs(g)
    ref = torch.from_numpy(g["desc"])
    got = hardnet_oracle.hardnet_forward(x, *_wmv(model), norm_eps=1e-8, l2_eps=0.0)
    assert (got - ref).abs().max().item() <= 2e-6
    # the tiny-std patch tells the two epsilons apart: with HardNet's 1e-7 the descriptor moves by far more
    other = hardnet_oracle.hardnet_forward(x[5:6], *_wmv(model))
    assert (other - ref[5:6]).abs().max().item() > 2e-3
    a, p = ref[:32], ref[32:]
    assert abs(model.loss(a, p, keypoints(32, 1), keypoints(32, 2)).item() - float(g["loss_c8"])) <= 1e-6
    model.C = 0.0
    assert abs(model.loss(a, p, keypoints(32, 1), keypoints(32, 2)).item() - float(g["loss_c0"])) <= 1e-6


@pytest.mark.gpu
def test_cuda_forward_matches_reference(golden_dir):
    g = np.load(golden_dir / "neimask.npz")
    model = _model().cuda()
    x = _inputs(g)
    ref = torch.from_numpy(g["desc"])
    got = model(x.cuda()).float().cpu()
    # 16-bit conv stack: the repo's stated bound (max-abs 1e-3, cosine 0.9999), including row 5 whose std (~3e-8) is of the
    # order of the input_norm epsilon
    assert (got - ref).abs().max().item() <= 1e-3
    assert torch.nn.functional.cosine_similarity(got, ref, dim=1).min().item() >= 0.9999
    # with HardNet's epsilons the same engine gives a clearly different row 5: the setting is really applied
    from hardnetnas_b200.hardnet import HardNet
    plain = HardNet()
    sd = {}
    for k, v in model.state_dict().items():
        idx = int(k.split(".")[1])
        sd[k.replace(f"features.{idx}.", f"features.{idx + 1 if idx >= 18 else idx}.")] = v   # HardNet has Dropout at 18
    plain.load_state_dict(sd)
    other = plain.cuda().eval()(x[5:6].cuda()).float().cpu()
    assert (other - ref[5:6]).abs().max().item() > 2e-3


def _torch_loss(model, a, p, akp, pkp):
    """The reference's expression sequence (rf_des.py:57-96) in plain torch, for gradients and large batches."""
    from hardnetnas_b200.matching import distance_matrix_vector, pairwise_distances
    d = distance_matrix_vector(a, p)
    pos = d.diag()
    masked = d + torch.eye(d.size(1), device=d.device) * 10
    for kp in (akp, pkp):
        masked = masked + pairwise_distances(kp[:, 1:3].to(torch.float)).lt(model.C).to(torch.float) * 10
    return torch.clamp(model.MARGIN + pos - torch.min(masked.min(dim=1)[0], masked.min(dim=0)[0]), min=0.0).mean()


@pytest.mark.gpu
def test_fused_neighbour_mask_loss_matches_reference_and_autograd(golden_dir):
    """HardNetNeiMask.loss on CUDA descriptors = hn_dist_min_ex with the keypoint masks fused into the distance epilogue:
    equal to the unmodified reference's loss values (golden), to the torch expression on larger / denser keypoint sets, and its
    sparse backward equal to autograd through the materialised matrix."""
    g = np.load(golden_dir / "neimask.npz")
    model = _model().cuda()
    ref = torch.from_numpy(g["desc"]).cuda()
    a, p = ref[:32], ref[32:]
    # random-init descriptors of random patches are nearly parallel (d ~ 0.03): sqrt(2 - 2 a.p) amplifies the 2e-6 error of the
    # tensor-core dot product to ~5e-5 in d, hence the looser bound here; the well-conditioned sets below hold 1e-5
    assert abs(model.loss(a, p, keypoints(32, 1).cuda(), keypoints(32, 2).cuda()).item() - float(g["loss_c8"])) <= 1e-4
    model.C = 0.0
    assert abs(model.loss(a, p, keypoints(32, 1).cuda(), keypoints(32, 2).cuda()).item() - float(g["loss_c0"])) <= 1e-4
    gen = torch.Generator().manual_seed(3)
    for n, c, span in ((257, 8.0, 64), (1024, 16.0, 200), (700, 5.0, 40)):
        model.C = c
        a = torch.nn.functional.normalize(torch.randn(n, 128, generator=gen), dim=1)
        p = torch.nn.functional.normalize(a + 0.25 * torch.randn(n, 128, generator=gen), dim=1)
        akp = torch.cat([torch.zeros(n, 1), torch.randint(0, span, (n, 2), generator=gen).float(), torch.zeros(n, 1)], 1)
        pkp = torch.cat([torch.zeros(n, 1), torch.randint(0, span, (n, 2), generator=gen).float(), torch.zeros(n, 1)], 1)
        want = _torch_loss(model, a, p, akp, pkp).item()      # CPU fp32 expression
        ac, pc = a.cuda().requires_grad_(True), p.cuda().requires_grad_(True)
        got = model.loss(ac, pc, akp.cuda(), pkp.cuda())
        assert abs(got.item() - want) <= 1e-5, (n, c, got.item(), want)
        got.backward()
        a2, p2 = a.clone().requires_grad_(True), p.clone().requires_grad_(True)
        _torch_loss(model, a2, p2, akp, pkp).backward()
        assert (ac.grad.cpu() - a2.grad).abs().max().item() <= 2e-5 and (pc.grad.cpu() - p2.grad).abs().max().item() <= 2e-5, (n, c)

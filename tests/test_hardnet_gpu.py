"""GPU parity: the B200 HardNet forward (through the C ABI) against the CPU oracle and the reference goldens."""
import numpy as np
import pytest
import torch

from oracle import hardnet_oracle, synth

pytestmark = pytest.mark.gpu

# 16-bit activations (fp16: 10-bit mantissa like TF32). Gates from BASELINE.json north_star.
DESC_MAX_ABS = 1e-3
DESC_MIN_COS = 0.9999


def _model(bn_seed, act_dtype="fp16", **kw):
    from hardnetnas_b200.hardnet import HardNet
    w, m, v = synth.hardnet_weights_from_seed(0, bn_seed)
    torch.manual_seed(0)
    model = HardNet(act_dtype=act_dtype, **kw)
    sd = model.state_dict()
    for i, (ci, bi) in enumerate(zip(synth.CONV_IDX, synth.BN_IDX)):
        assert torch.equal(sd[f"features.{ci}.weight"], w[i])  # same init stream as the reference
        sd[f"features.{bi}.running_mean"] = m[i]
        sd[f"features.{bi}.running_var"] = v[i]
    model.load_state_dict(sd)
    return model.cuda().eval(), (w, m, v)


def _cmp(desc, ref):
    desc = desc.float().cpu()
    max_abs = (desc - ref).abs().max().item()
    nz = ref.norm(dim=1) > 0
    cos = torch.nn.functional.cosine_similarity(desc[nz], ref[nz], dim=1).min().item()
    return max_abs, cos


@pytest.mark.parametrize("bn_seed", [3, None])
def test_stage_activations_match_oracle(bn_seed):
    model, (w, m, v) = _model(bn_seed)
    x = synth.make_patches(64, 1234)
    acts = hardnet_oracle.hardnet_stages(x, w, m, v, upto=6)
    xg = x.cuda()
    for layer in range(1, 7):
        got = model.forward_stage(xg, layer).float().cpu().permute(0, 3, 1, 2)
        ref = acts[layer - 1]
        scale = ref.abs().max().item()
        err = (got - ref).abs().max().item()
        assert err <= 4e-3 * scale + 1e-6, f"stage {layer}: max err {err:.3e} vs scale {scale:.3e}"


@pytest.mark.parametrize("bn_seed", [3, None])
def test_descriptors_match_oracle_and_golden(bn_seed, golden_dir):
    model, (w, m, v) = _model(bn_seed)
    x = synth.make_patches(64, 1234)
    desc = model(x.cuda())
    ref = hardnet_oracle.hardnet_forward(x, w, m, v)
    max_abs, cos = _cmp(desc, ref)
    assert max_abs <= DESC_MAX_ABS and cos >= DESC_MIN_COS, (max_abs, cos)
    g = np.load(golden_dir / "hardnet_forward.npz")
    gold = torch.from_numpy(g["desc" if bn_seed == 3 else "desc_fresh_bn"])
    max_abs, cos = _cmp(desc, gold)
    assert max_abs <= DESC_MAX_ABS and cos >= DESC_MIN_COS, (max_abs, cos)
    if bn_seed is None:
        assert torch.all(desc[-1] == 0)  # constant patch -> exactly zero descriptor, not NaN
    assert torch.isfinite(desc).all()


@pytest.mark.parametrize("batch", [1, 2, 3, 127, 129, 1024])
def test_ragged_batches(batch):
    model, (w, m, v) = _model(3, chunk_patches=64, head_rows=256)
    x = synth.make_patches(batch, 99, edge_cases=False)
    desc = model(x.cuda())
    ref = hardnet_oracle.hardnet_forward(x, w, m, v)
    max_abs, cos = _cmp(desc, ref)
    assert desc.shape == (batch, 128)
    assert max_abs <= DESC_MAX_ABS and cos >= DESC_MIN_COS, (max_abs, cos)


def test_empty_batch():
    model, _ = _model(3)
    out = model(torch.empty(0, 1, 32, 32, device="cuda"))
    assert out.shape == (0, 128)


def test_uint8_input_and_half_output():
    model, (w, m, v) = _model(None)
    g = torch.Generator().manual_seed(5)
    xu8 = torch.randint(0, 256, (96, 1, 32, 32), generator=g, dtype=torch.uint8)
    ref = hardnet_oracle.hardnet_forward(xu8.float(), w, m, v)
    d32 = model(xu8.cuda())
    max_abs, cos = _cmp(d32, ref)
    assert max_abs <= DESC_MAX_ABS and cos >= DESC_MIN_COS, (max_abs, cos)
    d16 = model(xu8.cuda(), out_dtype=torch.float16)
    assert d16.dtype == torch.float16
    assert (d16.float() - d32).abs().max().item() <= 1e-3


def test_bf16_activations_looser_bound():
    # stated bf16 bound (8-bit mantissa): max-abs <= 3e-3, cosine >= 0.9999 (SURVEY.md §8d)
    model, (w, m, v) = _model(None, act_dtype="bf16")
    x = synth.make_patches(256, 1234)
    max_abs, cos = _cmp(model(x.cuda()), hardnet_oracle.hardnet_forward(x, w, m, v))
    assert max_abs <= 3e-3 and cos >= 0.9999, (max_abs, cos)


def test_train_mode_uses_stock_torch_path():
    model, _ = _model(None)
    model.train()
    x = synth.make_patches(8, 3).cuda()
    out = model(x)
    assert out.requires_grad and out.shape == (8, 128)


def test_cpu_input_fails_loudly():
    from hardnetnas_b200._lib import HardnetB200Error
    model, _ = _model(None)
    with pytest.raises(HardnetB200Error):
        model(synth.make_patches(4, 1))


def test_full_size_properties():
    """Config-sized batch: finite, unit norm, deterministic, and chunking-invariant (size-independent checks)."""
    model, _ = _model(None)
    x = synth.make_patches(8192, 77, edge_cases=False).cuda()
    d1 = model(x)
    d2 = model(x)
    assert torch.equal(d1, d2)
    assert torch.isfinite(d1).all()
    assert (d1.norm(dim=1) - 1).abs().max().item() < 1e-4
    small, _ = _model(None, chunk_patches=32, head_rows=128)
    d3 = small(x[:1000])
    # the conv stack is chunking-invariant bit for bit; the head of a small batch runs split-K (another fp32 summation order
    # than the bulk head), which may move the last bit of a descriptor component
    assert (d3 - d1[:1000]).abs().max().item() <= 1e-6
    d4 = small(x[:1000])
    assert torch.equal(d3, d4)


def test_fpr95_agrees_with_reference_path():
    """FPR95 on a synthetic patch-pair set must agree to 0.1 pt (BASELINE.json north_star): label-1 pairs are
    (patch, patch + 0.1 * noise), label-0 pairs are independent patches (SURVEY.md section 8d)."""
    import numpy as np
    from hardnetnas_b200 import metrics
    from oracle import losses_oracle
    model, (w, m, v) = _model(3)
    n = 50000   # SURVEY.md section 8d; the oracle forward of the 200 000 patches takes ~40 s of host time
    a = synth.make_patches(2 * n, 11, edge_cases=False)
    p = torch.cat([synth.make_positives(a[:n], 0.1, 7), synth.make_patches(n, 12, edge_cases=False)])
    labels = torch.cat([torch.ones(n), torch.zeros(n)]).long()
    da, dp = model(a.cuda()), model(p.cuda())
    dist = metrics.pair_distances(da, dp)
    fpr_dev = metrics.ErrorRateAt95Recall(labels.cuda(), 1.0 / (dist + 1e-8))
    ra = torch.cat([hardnet_oracle.hardnet_forward(c, w, m, v) for c in a.split(8192)])
    rp = torch.cat([hardnet_oracle.hardnet_forward(c, w, m, v) for c in p.split(8192)])
    rdist = torch.sqrt(torch.sum((ra - rp) ** 2, 1)).numpy()
    fpr_ref = losses_oracle.error_rate_at_95_recall(labels.numpy(), 1.0 / (rdist + 1e-8))
    assert abs(fpr_dev - fpr_ref) <= 1e-3, (fpr_dev, fpr_ref)
    assert 0.0 < fpr_ref < 0.5   # the set is non-degenerate
    # the device metric itself equals the reference metric on identical inputs
    assert metrics.ErrorRateAt95Recall(labels, torch.from_numpy(1.0 / (rdist + 1e-8))) == fpr_ref


@pytest.mark.parametrize("n,pos_frac,ties", [(1, 1.0, False), (7, 0.0, False), (1000, 0.5, False), (100003, 0.3, False), (50000, 0.5, True),
                                             (4096, 1.0, True), (2049, 0.02, True)])
def test_fpr95_selection_kernel_equals_the_sorted_reference(n, pos_frac, ties):
    """hn_fpr95 (radix selection of the threshold element, no sort) against hardnet/EvalMetrics.py:6-19 evaluated with a STABLE
    sort on identical inputs: FP, TN and the threshold index must be equal, including heavy ties (quantised distances), all /
    no positives and tiny inputs."""
    import numpy as np
    from hardnetnas_b200 import metrics
    rng = np.random.RandomState(n)
    labels = (rng.rand(n) < pos_frac).astype(np.int64)
    dist = rng.rand(n).astype(np.float32) * 2.0
    dist[labels == 1] *= 0.6                                  # positives tend to be closer
    if ties:
        dist = np.round(dist * 16).astype(np.float32) / 16    # 33 distinct values: long runs of equal distances
    scores = (1.0 / (dist + np.float32(1e-8))).astype(np.float32)
    d2 = (1.0 / (scores + np.float32(1e-8))).astype(np.float32)
    lab_sorted = labels[np.argsort(d2, kind="stable")]
    thr = int(np.argmax(np.cumsum(lab_sorted) >= 0.95 * np.sum(lab_sorted)))
    fp, tn = int(np.sum(lab_sorted[:thr] == 0)), int(np.sum(lab_sorted[thr:] == 0))
    got = metrics.fpr95_counts(torch.from_numpy(labels).cuda(), torch.from_numpy(scores).cuda()).tolist()
    assert got == [fp, tn, int(labels.sum()), thr], (got, fp, tn, thr)
    if fp + tn:
        assert metrics.ErrorRateAt95Recall(torch.from_numpy(labels).cuda(), torch.from_numpy(scores).cuda()) == float(fp) / float(fp + tn)


def test_host_pipeline_matches_direct_forward():
    """extract_descriptors (pinned host in / out, H2D + forward + D2H pipelined) returns what forward() returns."""
    from hardnetnas_b200.extract import DescriptorExtractor, extract_descriptors
    model, _ = _model(3, chunk_patches=256, head_rows=512)
    x = synth.make_patches(1500, 21, edge_cases=False)
    ref = model(x.cuda()).cpu()
    out = extract_descriptors(model, x.pin_memory())
    assert torch.equal(out, ref)
    ext = DescriptorExtractor(model, batch=300)          # ragged: 5 batches, the last one partial
    assert torch.equal(ext(x.pin_memory()), ref)
    assert torch.equal(ext(x[:7].pin_memory()), ref[:7])


@pytest.mark.parametrize("n,chunk", [(1, 0), (2, 0), (301, 0), (333, 96), (1000, 256), (4097, 0)])
def test_fused_conv3_conv4_kernel_against_the_two_kernel_reference(n, chunk, monkeypatch):
    """conv3 + conv4 in one kernel (csrc/tc_conv34.cuh, the default: conv4's kx taps stacked on N and finished by
    tcgen05.shift + warp shuffles) against HN_FUSE34=0 (two CTA-pair kernels). The fused kernel accumulates in another order:
    conv4's output differs by at most one fp16 rounding step here and there, the descriptors by ~2e-5; both paths meet the
    oracle gate. Odd batch sizes leave one CTA of the last pair without a patch; chunks 96 and 256 make several (ragged)
    passes."""
    x = synth.make_patches(n, 77 + n, edge_cases=False)
    xg = x.cuda()
    outs = {}
    for mode in ("0", "fused"):
        if mode == "0":
            monkeypatch.setenv("HN_FUSE34", "0")
        else:
            monkeypatch.delenv("HN_FUSE34", raising=False)
        model, (w, m, v) = _model(3, chunk_patches=chunk, head_rows=0 if chunk == 0 else 1024)
        outs[mode] = {"desc": model(xg)}
        if n <= 512 and (chunk == 0 or n <= chunk):   # a stage dump covers one pass
            for layer in (4, 5, 6):
                outs[mode][layer] = model.forward_stage(xg, layer)
        torch.cuda.synchronize()
    for k, ref in outs["0"].items():
        d = (outs["fused"][k].float() - ref.float()).abs().max().item()
        assert d <= (1e-4 if k == "desc" else 1e-3), f"{k}: {d:.3e}"
    if n == 4097:
        # races between the kernel's roles (producer / issuer / shifter / epilogue warps of two CTAs) would show as run-to-run
        # differences: the default kernel is bit-reproducible over a full pass and a large batch
        big = synth.make_patches(40000, 5, edge_cases=False).cuda()
        a = model(big)
        assert torch.equal(model(big), a)
        # (a 4097-patch batch runs the head GEMM split-K: another fp32 summation order, hence a tolerance instead of equality)
        assert (model(big[:4097]) - a[:4097]).abs().max().item() <= 1e-6
    ref = hardnet_oracle.hardnet_forward(x[:256], w, m, v)
    for mode in ("0", "fused"):
        max_abs, cos = _cmp(outs[mode]["desc"][:256], ref)
        assert max_abs <= DESC_MAX_ABS and cos >= DESC_MIN_COS, (mode, max_abs, cos)


def test_head_gemm_two_tiles_per_weight_stream_is_bit_identical():
    """Bulk batches run the head GEMM with two 128-row tiles per streamed weight block (gemm_l2norm_kernel<N, 2>, used when a head
    launch has more tiles than SMs; default head batch = 2 x #SM x 128 patches). Same K order per tile: bit-identical to the
    one-tile kernel, also with an odd tile count (the phantom tile reads zero-filled rows and stores nothing)."""
    x = synth.make_patches(37888, 21, edge_cases=False).cuda()
    one_tile, _ = _model(3, head_rows=18944)     # 148 + <= 148 tiles per head launch: one tile per work item, K not split
    two_tiles, _ = _model(3)                     # one head launch of up to 296 tiles: two tiles per work item
    ref = one_tile(x)
    assert torch.equal(two_tiles(x), ref)                                # 296 tiles
    n = 37888 - 128 - 55                                                 # 295 tiles (odd), ragged last tile
    assert torch.equal(two_tiles(x[:n]), one_tile(x[:n]))


def test_second_gpu_in_the_same_process():
    """Kernel attributes (dynamic shared memory limits) are per device: a process may use more than one GPU."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    model0, (w, m, v) = _model(3)
    x = synth.make_patches(200, 41, edge_cases=False)
    ref = hardnet_oracle.hardnet_forward(x, w, m, v)
    d0 = model0(x.cuda(0))
    model1, _ = _model(3)
    model1 = model1.to("cuda:1")
    d1 = model1(x.to("cuda:1"))
    for d in (d0, d1):
        max_abs, cos = _cmp(d, ref)
        assert max_abs <= DESC_MAX_ABS and cos >= DESC_MIN_COS
    from hardnetnas_b200.matching import match_top2
    q, g, _ = synth.make_match_set(300, 900, seed=4)
    a = [t.cpu() for t in match_top2(q.cuda(0), g.cuda(0))]
    b = [t.cpu() for t in match_top2(q.to("cuda:1"), g.to("cuda:1"))]
    for s, t in zip(a, b):
        assert torch.equal(s, t)


def test_direct_parity_at_a_full_default_pass_65536_patches():
    """One direct comparison at bulk size (VERDICT r1 weak #2): 65 536 patches through the default 18 944-patch passes
    (three full passes + a ragged one, full head batches) against the CPU oracle on every row - not a sample, not a
    small-chunk engine."""
    model, (w, m, v) = _model(3)
    x = synth.make_patches(65536, 77)
    desc = model(x.cuda()).float().cpu()
    ref = torch.cat([hardnet_oracle.hardnet_forward(x[i:i + 8192], w, m, v) for i in range(0, 65536, 8192)])
    max_abs, cos = _cmp(desc, ref)
    assert max_abs <= DESC_MAX_ABS and cos >= DESC_MIN_COS, (max_abs, cos)

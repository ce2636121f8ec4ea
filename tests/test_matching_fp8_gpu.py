"""fp8 e4m3 descriptors end to end: forward outputs in e4m3 equal the fp32 output rounded to e4m3, byte for byte; matching on
e4m3 rows (packed e4m3 operands, kind::f8f6f4 GEMM) returns exactly what the same call returns on the rows' .float(); the fp8
GEMM's accumulation error stays within the bound the re-rank and verification margins are made of (dist.cu, kF8DotBound).
e4m3 tensors are compared through .view(torch.uint8): torch.equal is not implemented for fp8."""
import pytest
import torch

from oracle import synth
from test_matching_batched_gpu import _keypoints
from test_matching_pairs_gpu import _table, _two_sets

pytestmark = pytest.mark.gpu

E4M3 = torch.float8_e4m3fn
F8_DOT_BOUND = 5.9e-4          # dist.cu kF8DotBound (unscaled dot units)
SCALED = 256.0 * 256.0         # the GEMM's units: operands are x * 2^8


@pytest.fixture
def force_kernel():
    from hardnetnas_b200 import _lib
    lib = _lib.load()
    yield lambda mode: _lib.check(lib.hn_match_force_kernel(int(mode)), "hn_match_force_kernel")
    lib.hn_match_force_kernel(-1)


def _bytes(t):
    return t.view(torch.uint8) if t.dtype == E4M3 else t


def _equal(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        if isinstance(x, torch.Tensor):
            assert x.dtype == y.dtype and x.shape == y.shape
            assert torch.equal(_bytes(x), _bytes(y))
        else:
            assert x == y


def _both(fn, *xs):
    """fn on the e4m3 tensors and on their fp32 conversions."""
    return fn(*xs), fn(*[x.float() if x.is_floating_point() else x for x in xs])


def _set8(nq, ng, seed):
    q, g, _ = synth.make_match_set(nq, ng, seed=seed)
    return q.to("cuda", E4M3), g.to("cuda", E4M3)


# ---- forward ----------------------------------------------------------------------------------------------------------------

def _hardnet():
    from hardnetnas_b200.hardnet import HardNet
    torch.manual_seed(0)
    m = HardNet()
    m.load_state_dict(synth.randomize_bn_stats(m.state_dict(), 3))
    return m.cuda().eval()


def _assert_e4m3_of(got, ref32):
    assert got.dtype == E4M3 and got.shape == ref32.shape
    assert torch.equal(got.view(torch.uint8), ref32.to(E4M3).view(torch.uint8))


@pytest.mark.parametrize("n", [64, 1500])   # 64: the split-K head (head_finalize_kernel); 1500: the head GEMM's own epilogue
def test_forward_hardnet(n):
    model = _hardnet()
    x = synth.make_patches(n, 1234).cuda()
    _assert_e4m3_of(model(x, out_dtype=E4M3), model(x))
    out = torch.empty(n, 128, dtype=E4M3, device="cuda")
    assert model(x, out=out) is out
    _assert_e4m3_of(out, model(x))


def test_forward_neimask():
    from hardnetnas_b200.rf_des import HardNetNeiMask
    torch.manual_seed(0)
    model = HardNetNeiMask(1.0, 8.0)
    model.load_state_dict(synth.randomize_bn_stats(model.state_dict(), 3))
    model = model.cuda().eval()
    x = synth.make_patches(300, 99).cuda()
    _assert_e4m3_of(model(x, out_dtype=E4M3), model(x))


@pytest.mark.parametrize("n", [64, 1000])
def test_forward_nas_wang2(n):
    from hardnetnas_b200.nas import SampledDescriptorNet
    from hardnetnas_b200.nas.fbnet_modeldef import arch_ops
    torch.manual_seed(0)
    net = SampledDescriptorNet(arch_ops("wang2"))
    net.load_state_dict(synth.randomize_nas_state(net.state_dict(), 4))
    net = net.cuda().eval()
    x = synth.make_patches(n, 4321).cuda()
    _assert_e4m3_of(net(x, out_dtype=E4M3), net(x))


def test_forward_clip():
    from oracle import clip_oracle
    byxc, scale, ori, im_info, images = clip_oracle.make_clip_inputs(seed=5, B=4, H=240, W=320, k=200)
    model = _hardnet()
    args = (byxc.cuda(), scale.cuda(), ori.cuda(), im_info.cuda(), images.cuda())
    _assert_e4m3_of(model.forward_clip(*args, out_dtype=E4M3), model.forward_clip(*args))


def test_extract_descriptors():
    from hardnetnas_b200.extract import extract_descriptors
    model = _hardnet()
    x = synth.make_patches(1000, 77).pin_memory()
    got = extract_descriptors(model, x, batch=384, out_dtype=E4M3)
    _assert_e4m3_of(got, extract_descriptors(model, x, batch=384))


# ---- packing ----------------------------------------------------------------------------------------------------------------

def test_pack_is_the_exact_e4m3_scaling():
    from hardnetnas_b200._ops import pack_descriptors
    q, g = _special_rows()
    x = torch.cat([q, g, _set8(1000, 1, 4)[0]])
    p = pack_descriptors(x)
    assert p.dtype == E4M3 and p.shape == x.shape
    want = (x.float() * 256).to(E4M3)
    assert torch.equal(p.view(torch.uint8), want.view(torch.uint8))
    assert torch.equal(p.float(), x.float() * 256)   # no rounding happened
    out = torch.empty_like(p)
    assert pack_descriptors(x, out=out) is out and torch.equal(out.view(torch.uint8), p.view(torch.uint8))
    with pytest.raises(ValueError):
        pack_descriptors(x, out=torch.empty(x.size(0), 128, dtype=torch.float16, device="cuda"))


# ---- bit identity with the call on .float() ---------------------------------------------------------------------------------

@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("nq,ng", [(1, 1), (7, 129), (129, 1000), (1000, 7), (8192 + 33, 2048)])
def test_single_problem(mode, nq, ng, force_kernel):
    from hardnetnas_b200.matching import match_top2, mutual_nn_ratio
    force_kernel(mode)
    q, g = _set8(nq, ng, seed=nq + ng)
    _equal(*_both(match_top2, q, g))
    _equal(*_both(mutual_nn_ratio, q, g))


def test_given_packed_operands(force_kernel):
    from hardnetnas_b200 import _ops
    q, g = _set8(3000, 5000, seed=17)
    q8, g8 = _ops.pack_descriptors(q), _ops.pack_descriptors(g)
    for mode in (0, 1):
        force_kernel(mode)
        want = _ops.match_top2(q.float(), g.float())
        _equal(_ops.match_top2(q, g, q16=q8, g16=g8), want)
        _equal(_ops.match_mutual(q, g, q8, g8), _ops.match_mutual(q.float(), g.float()))
    with pytest.raises(ValueError, match="e4m3 for e4m3 rows"):
        _ops.match_top2(q, g, q16=_ops.pack_descriptors(q.float()))
    with pytest.raises(ValueError, match="e4m3 for e4m3 rows"):
        _ops.match_top2(q.float(), g.float(), g16=g8)


def _padded_8(lens, n, seed, fill):
    rows = torch.full((len(lens), n, 128), fill)
    for b, k in enumerate(lens):
        if k:
            rows[b, :k] = synth.unit_vectors(k, 128, seed + b)
    return rows.to("cuda", E4M3)


@pytest.mark.parametrize("mutual", [False, True])
def test_batched_ragged(mutual):
    from hardnetnas_b200 import _ops
    gen = torch.Generator().manual_seed(3)
    lq = [0, 1, 2, 257, 129, 256, 17, 200, 0, 64] + torch.randint(0, 258, (6,), generator=gen).tolist()
    lg = [5, 0, 1, 257, 128, 255, 0, 3, 0, 257] + torch.randint(0, 258, (6,), generator=gen).tolist()
    G = _padded_8(lg, 257, 100, float("inf"))   # e4m3fn has no inf: padding becomes NaN, which padding may hold
    Q = _padded_8(lq, 257, 200, float("nan"))
    for b, k in enumerate(lq):
        m = min(k, lg[b])
        if m:
            Q[b, :m] = torch.nn.functional.normalize(G[b, :m].float() + 0.04 * torch.randn(m, 128, device="cuda"), dim=1).to(E4M3)
    L1 = torch.tensor(lq, dtype=torch.int32, device="cuda")
    L2 = torch.tensor(lg, dtype=torch.int32, device="cuda")
    got, want = _both(lambda q, g: _ops.match_batched(q, g, L1, L2, mutual=mutual), Q, G)
    _equal(got, want)
    assert torch.all(got[2][0] == -1) and torch.all(got[2][6] == -1)


def test_pair_tables():
    from hardnetnas_b200 import _ops
    Q, sq, nq, G, sg, ng = _two_sets([500, 129, 1024, 7, 1], [1024, 600, 1, 300, 257], seed=60)
    Q, G = Q.to("cuda", E4M3), G.to("cuda", E4M3)
    rows = [[sq[i], nq[i], sg[j], ng[j]] for i, j in [(0, 0), (0, 1), (2, 0), (1, 4), (3, 4), (4, 3), (2, 2), (0, 3)]]
    T = _table(rows).cuda()
    for mutual in (False, True):
        got, want = _both(lambda q, g: _ops.match_pairs(q, g, T, 1024, 1024, mutual=mutual), Q, G)
        _equal(got, want)
        q8, g8 = _ops.pack_descriptors(Q), _ops.pack_descriptors(G)
        assert q8.dtype == E4M3
        _equal(_ops.match_pairs(Q, G, T, 1024, 1024, q8, g8, mutual=mutual), got)
        with pytest.raises(ValueError, match="e4m3 for e4m3 rows"):
            _ops.match_pairs(Q, G, T, 1024, 1024, _ops.pack_descriptors(Q.float()), g8)
    S = torch.cat([Q, G])
    off = Q.size(0)
    T2 = _table([[sq[0], nq[0], sq[0], nq[0]], [sq[2], nq[2], off + sg[1], ng[1]], [off + sg[4], ng[4], sq[1], nq[1]]]).cuda()
    S32 = S.float()
    want = _ops.match_pairs(S32, S32, T2, 1024, 1024, mutual=True)
    _equal(_ops.match_pairs(S, S, T2, 1024, 1024, mutual=True), want)
    s8 = _ops.pack_descriptors(S)
    _equal(_ops.match_pairs(S, S, T2, 1024, 1024, g16=s8, mutual=True), want)


def _special_rows():
    """Awkward e4m3 values: one-hot rows (exactly +-1), all-zero rows, exact duplicates, rows with e4m3 subnormal components
    (2^-9, the smallest), and near-ties: rows one e4m3 ulp apart in one component."""
    g = synth.unit_vectors(200, 128, 9)
    g[100:110] = 0.0
    g[100:110, torch.arange(10)] = 1.0
    g[110:120] = 0.0
    g[110:120, torch.arange(10, 20)] = -1.0
    g[120:126] = 0.0
    g[130:140, 40:60] = 2.0 ** -9
    g[140:150, 60:80] = -(2.0 ** -9)
    g = g.to(E4M3)
    # near-ties: rows 160..179 are rows 0..19 with one component moved by one e4m3 ulp (byte + 1 on the magnitude)
    b = g.view(torch.uint8).clone()
    col = torch.arange(20) * 5 % 128
    rows = torch.arange(20)
    mag = b[rows, col] & 0x7F
    b[160 + rows, :] = b[rows, :]
    b[160 + rows, col] = torch.where(mag < 0x7E, b[rows, col] + 1, b[rows, col] - 1).to(torch.uint8)
    g = b.view(E4M3)
    g = torch.cat([g, g[:50]])        # rows 200..249 duplicate rows 0..49 exactly
    gf = g.float()
    q = torch.nn.functional.normalize(gf[:100] + 0.03 * torch.randn(100, 128, generator=torch.Generator().manual_seed(1)), dim=1)
    q = torch.cat([q.to(E4M3), g[100:180], torch.zeros(3, 128, dtype=E4M3)])
    return q.cuda(), g.cuda()


def test_special_values_and_ties():
    from hardnetnas_b200 import _ops
    from hardnetnas_b200.matching import match_top2, mutual_nn_ratio
    q, g = _special_rows()
    got, want = _both(match_top2, q, g)
    _equal(got, want)
    _equal(*_both(mutual_nn_ratio, q, g))
    dup = (got[2][:100] < 50).nonzero().flatten()
    assert dup.numel() > 0
    assert torch.equal(got[3][dup], got[2][dup] + 200) and torch.equal(got[0][dup], got[1][dup])
    _equal(*_both(lambda a, b: _ops.match_batched(a.unsqueeze(0), b.unsqueeze(0), mutual=True), q, g))
    T = _table([[0, q.size(0), 0, g.size(0)], [100, 63, 50, 200]]).cuda()
    _equal(*_both(lambda a, b: _ops.match_pairs(a, b, T, q.size(0), g.size(0), mutual=True), q, g))


def test_score_counters():
    from hardnetnas_b200 import matching
    gen = torch.Generator().manual_seed(5)
    sets = []
    for b, (a, c) in enumerate([(500, 1000), (768, 2048), (100, 1), (40, 300)]):
        q, g, truth = synth.make_match_set(a, c, seed=70 + b)
        sets.append((q, g, *_keypoints(a, c, truth, gen)))
    B, NQ, NG = len(sets), 768, 2048
    Q, G = torch.zeros(B, NQ, 128), torch.zeros(B, NG, 128)
    KP1, KP2 = torch.zeros(B, NQ, 3), torch.zeros(B, NG, 3)
    VIS = torch.zeros(B, NQ, dtype=torch.bool)
    for b, (q, g, kp1w, kp2, vis) in enumerate(sets):
        Q[b, :q.size(0)], G[b, :g.size(0)], KP1[b, :q.size(0)], KP2[b, :g.size(0)], VIS[b, :q.size(0)] = q, g, kp1w, kp2, vis
    L1 = torch.tensor([s[0].size(0) for s in sets], device="cuda")
    L2 = torch.tensor([s[1].size(0) for s in sets], device="cuda")
    Q8, G8, KP1, KP2, VIS = Q.to("cuda", E4M3), G.to("cuda", E4M3), KP1.cuda(), KP2.cuda(), VIS.cuda()
    for fn, extra in ((matching.nearest_neighbor_match_score_batched, ()),
                      (matching.nearest_neighbor_threshold_match_score_batched, (1.0,)),
                      (matching.nearest_neighbor_distance_ratio_match_score_batched, ())):
        args = (*extra, 5.0) if extra else (5.0,)
        _equal(fn(Q8, G8, KP1, KP2, VIS, *args, len1=L1, len2=L2), fn(Q8.float(), G8.float(), KP1, KP2, VIS, *args, len1=L1, len2=L2))
    X1 = torch.cat([s[0] for s in sets]).to("cuda", E4M3)
    X2 = torch.cat([s[1] for s in sets]).to("cuda", E4M3)
    kp2_all = torch.cat([s[3] for s in sets]).cuda()
    T = matching.pair_table(torch.tensor([s[0].size(0) for s in sets]), list(range(B)), list(range(B)),
                            counts2=torch.tensor([s[1].size(0) for s in sets])).cuda()
    for fn, extra in ((matching.nearest_neighbor_match_score_pairs, ()),
                      (matching.nearest_neighbor_threshold_match_score_pairs, (1.0,)),
                      (matching.nearest_neighbor_distance_ratio_match_score_pairs, ())):
        args = (*extra, 5.0) if extra else (5.0,)
        _equal(fn(X1, X2, T, KP1, kp2_all, VIS, *args), fn(X1.float(), X2.float(), T, KP1, kp2_all, VIS, *args))


# ---- float64 oracle ---------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("mode", [0, 1])
def test_top2_equals_a_float64_brute_force(mode, force_kernel):
    """On e4m3-valued rows every product is exact in fp32 and every partial sum of the re-rank is a multiple of 2^-18 below
    2, so the re-rank's fp32 dot is exact, and sqrtf of the exact 2 - 2ab rounds like the float64 root rounded to fp32. Top-2
    distances and indices therefore equal a float64 brute force, ties resolved to the lower index."""
    from hardnetnas_b200.matching import match_top2
    force_kernel(mode)
    q, g = _set8(3000, 4000, seed=23)
    g = torch.cat([g, g[:300]])   # exact duplicates: ties
    d1, d2, i1, i2 = match_top2(q, g)
    dot = q.double() @ g.double().t()
    lo = torch.tensor(1e-8, dtype=torch.float32).double()
    d = torch.sqrt((2.0 - 2.0 * dot).clamp(min=lo, max=4.0)).float()
    ds, idx = torch.sort(d, dim=1, stable=True)
    assert torch.equal(d1, ds[:, 0]) and torch.equal(d2, ds[:, 1])
    assert torch.equal(i1.long(), idx[:, 0]) and torch.equal(i2.long(), idx[:, 1])


# ---- accumulation probe -----------------------------------------------------------------------------------------------------

def _probe_rows(seed):
    """Adversarial e4m3 rows for the fp8 GEMM's accumulation: long runs of equal-magnitude terms of alternating sign, mixes of
    2^-9 and ~1 components, large terms that cancel ahead of small ones, and random unit rows."""
    gen = torch.Generator().manual_seed(seed)
    t = 2.0 ** -9
    c = 0.0859375                                   # an e4m3 value near 128^-0.5
    alt = torch.tensor([1.0, -1.0]).repeat(64)
    rows = [
        c * alt, c * torch.ones(128), c * alt.roll(1), c * torch.cat([torch.ones(64), -torch.ones(64)]),
        c * torch.sign(torch.randn(128, generator=gen)), c * torch.sign(torch.randn(128, generator=gen)),
        torch.cat([torch.tensor([0.9375]), torch.full((127,), t)]),
        torch.cat([torch.tensor([1.0]), torch.full((127,), t)]),
        torch.cat([torch.tensor([-1.0]), torch.full((127,), t)]),
        torch.cat([torch.tensor([0.5, -0.5]), torch.full((126,), t)]),
        torch.cat([torch.tensor([0.6875, 0.6875]), t * alt[:126]]),
        torch.cat([torch.full((32,), t), torch.tensor([1.0]), torch.full((95,), t)]),
        torch.cat([torch.full((96,), t), torch.tensor([0.9375]), torch.full((31,), -t)]),
        torch.full((128,), t),
        torch.cat([torch.tensor([0.125] * 32), torch.full((96,), t)]),
        torch.cat([torch.tensor([0.125, -0.125] * 16), torch.full((96,), -t)]),
    ]
    rows = torch.stack(rows)
    rand = synth.unit_vectors(64 - rows.size(0), 128, seed + 1)
    mixed = rand.clone()
    mixed[:, 1::2] = t * torch.sign(mixed[:, 1::2])
    mixed = torch.nn.functional.normalize(mixed, dim=1)
    x = torch.cat([rows, rand[: (64 - rows.size(0)) // 2], mixed[: 64 - rows.size(0) - (64 - rows.size(0)) // 2]])
    return x.to(E4M3)


@pytest.mark.parametrize("mode", [0, 1])
def test_accumulation_within_the_margin_bound(mode, force_kernel):
    """Every (32-row, 8-column) cell holds ONE distinct dot product (32 copies of a query row against 8 copies of a gallery row),
    so the GEMM's cell maxima are single fp8-GEMM dot products; compared with the float64 dot of the scaled rows."""
    from hardnetnas_b200 import _ops
    force_kernel(mode)
    a, b = _probe_rows(1), _probe_rows(2)
    x = torch.cat([a, b.flip(0)]).cuda()                  # 128 distinct rows, each side
    y = torch.cat([b, a]).cuda()
    q = x.repeat_interleave(32, dim=0)                      # 4096 rows: row block r = x[r]
    g = y.repeat_interleave(8, dim=0)                       # 1024 columns: chunk c = y[c]
    bm = torch.empty(_ops.block_max_elems(q.size(0), g.size(0)), dtype=torch.float32, device="cuda")
    _ops.match_top2(q, g, block_max=bm)
    got = bm.view(g.size(0) // 8, q.size(0) // 32).t().double()   # [query row block][gallery chunk]
    want = (x.double() * 256) @ (y.double() * 256).t()
    err = (got - want).abs().max().item() / SCALED
    print(f"\nfp8 GEMM (mode {mode}): max |dot error| over {want.numel()} adversarial dot products = {err:.3e} "
          f"(bound {F8_DOT_BOUND:.1e}, fp16-path bound {2.0 ** -10:.3e})")
    assert err <= F8_DOT_BOUND


# ---- memory and graphs ------------------------------------------------------------------------------------------------------

def _peak_bytes(fn):
    fn()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    out = fn()
    torch.cuda.synchronize()
    del out
    return torch.cuda.max_memory_allocated() - base


def test_peak_memory_not_above_the_fp16_call():
    from hardnetnas_b200.matching import match_top2, match_top2_batched, match_top2_pairs, mutual_nn_ratio
    n = 1 << 16
    X = torch.nn.functional.normalize(torch.randn(n, 128, device="cuda"), dim=1).to(E4M3)
    H = X.half()
    T = _table([[4096 * i, 1024, 4096 * i + 2048, 1024] for i in range(8)]).cuda()
    for call in (lambda x: match_top2_pairs(x, x, T, 1024, 1024), lambda x: match_top2(x[: n // 2], x[n // 2:]),
                 lambda x: mutual_nn_ratio(x[: n // 2], x[n // 2:], return_pairs=False),
                 lambda x: match_top2_batched(x.view(16, n // 16, 128)[:8], x.view(16, n // 16, 128)[8:])):
        assert _peak_bytes(lambda: call(X)) <= _peak_bytes(lambda: call(H))


def test_batched_graph_replay():
    from hardnetnas_b200 import _ops
    Q, sq, nq, G, sg, ng = _two_sets([500, 129, 1024, 7], [1024, 600, 1, 300], seed=80)
    Qb = torch.zeros(4, 1024, 128, device="cuda", dtype=E4M3)
    Gb = torch.zeros(4, 1024, 128, device="cuda", dtype=E4M3)
    for i in range(4):
        Qb[i, :nq[i]], Gb[i, :ng[i]] = Q[sq[i]:sq[i] + nq[i]].to("cuda", E4M3), G[sg[i]:sg[i] + ng[i]].to("cuda", E4M3)
    L1 = torch.tensor(nq, dtype=torch.int32, device="cuda")
    L2 = torch.tensor(ng, dtype=torch.int32, device="cuda")
    fn = lambda: _ops.match_batched(Qb, Gb, L1, L2, mutual=True)   # noqa: E731
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        eager = fn()
        torch.cuda.set_sync_debug_mode("error")
        try:
            again = fn()
        finally:
            torch.cuda.set_sync_debug_mode("default")
        _equal(eager, again)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        captured = fn()
    Gb[1, :300] = Gb[1, 300:600].clone()
    L2.copy_(torch.tensor([1024, 300, 1, 17], dtype=torch.int32))
    for t in captured:
        t.zero_()
    graph.replay()
    torch.cuda.synchronize()
    want = _ops.match_batched(Qb.float(), Gb.float(), L1, L2, mutual=True)
    _equal(captured, want)
    graph.replay()
    torch.cuda.synchronize()
    _equal(captured, want)

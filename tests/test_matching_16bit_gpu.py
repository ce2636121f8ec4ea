"""Matching on fp16 / bf16 descriptor rows (the *_typed entry points): every output equals the same call on the rows converted
to fp32, bit for bit (d1, d2, i1, i2, mutual, padding rows included), for the single-problem, batched and pair-table forms,
the packing and the score counters; a 16-bit call makes no fp32 copy of its rows and needs no host synchronisation."""
import pytest
import torch

from oracle import synth
from test_matching_batched_gpu import _keypoints
from test_matching_pairs_gpu import _table, _two_sets

pytestmark = pytest.mark.gpu

DTYPES = [torch.float16, torch.bfloat16]
IDS = ["fp16", "bf16"]


@pytest.fixture
def force_kernel():
    """hn_match_force_kernel(mode): -1 by size, 0 single-CTA GEMM, 1 CTA-pair GEMM; restored afterwards."""
    from hardnetnas_b200 import _lib
    lib = _lib.load()
    yield lambda mode: _lib.check(lib.hn_match_force_kernel(int(mode)), "hn_match_force_kernel")
    lib.hn_match_force_kernel(-1)


def _equal(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        if isinstance(x, torch.Tensor):
            assert x.dtype == y.dtype and x.shape == y.shape
            assert torch.equal(x, y)
        else:
            assert x == y


def _set16(nq, ng, dt, seed):
    q, g, _ = synth.make_match_set(nq, ng, seed=seed)
    return q.to("cuda", dt), g.to("cuda", dt)


def _both(fn, *xs):
    """fn on the 16-bit tensors and on their fp32 conversions."""
    return fn(*xs), fn(*[x.float() if x.is_floating_point() else x for x in xs])


@pytest.mark.parametrize("dt", DTYPES, ids=IDS)
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("nq,ng", [(1, 1), (7, 129), (129, 1000), (1000, 7), (8192 + 33, 2048)])
def test_single_problem(dt, mode, nq, ng, force_kernel):
    from hardnetnas_b200.matching import match_top2, mutual_nn_ratio
    force_kernel(mode)
    q, g = _set16(nq, ng, dt, seed=nq + ng)
    _equal(*_both(match_top2, q, g))
    _equal(*_both(mutual_nn_ratio, q, g))


def _padded_16(lens, n, dt, seed, fill):
    rows = torch.full((len(lens), n, 128), fill)
    for b, k in enumerate(lens):
        if k:
            rows[b, :k] = synth.unit_vectors(k, 128, seed + b)
    return rows.to("cuda", dt)


@pytest.mark.parametrize("dt", DTYPES, ids=IDS)
@pytest.mark.parametrize("mutual", [False, True])
def test_batched_ragged(dt, mutual):
    from hardnetnas_b200 import _ops
    gen = torch.Generator().manual_seed(3)
    lq = [0, 1, 2, 257, 129, 256, 17, 200, 0, 64] + torch.randint(0, 258, (6,), generator=gen).tolist()
    lg = [5, 0, 1, 257, 128, 255, 0, 3, 0, 257] + torch.randint(0, 258, (6,), generator=gen).tolist()
    G = _padded_16(lg, 257, dt, 100, float("inf"))
    Q = _padded_16(lq, 257, dt, 200, float("nan"))
    for b, k in enumerate(lq):   # queries: noisy copies of the pair's gallery rows where it has some
        m = min(k, lg[b])
        if m:
            Q[b, :m] = torch.nn.functional.normalize(G[b, :m].float() + 0.04 * torch.randn(m, 128, device="cuda"), dim=1).to(dt)
    L1 = torch.tensor(lq, dtype=torch.int32, device="cuda")
    L2 = torch.tensor(lg, dtype=torch.int32, device="cuda")
    got, want = _both(lambda q, g: _ops.match_batched(q, g, L1, L2, mutual=mutual), Q, G)
    _equal(got, want)
    assert torch.all(got[2][0] == -1) and torch.all(got[2][6] == -1)   # pairs without gallery rows


@pytest.mark.parametrize("dt", DTYPES, ids=IDS)
def test_pair_tables(dt):
    from hardnetnas_b200 import _ops
    Q, sq, nq, G, sg, ng = _two_sets([500, 129, 1024, 7, 1], [1024, 600, 1, 300, 257], seed=60)
    Q, G = Q.to("cuda", dt), G.to("cuda", dt)
    # reused images, odd starts (the sets begin with unrelated rows), a range ending at the last row of each set
    rows = [[sq[i], nq[i], sg[j], ng[j]] for i, j in [(0, 0), (0, 1), (2, 0), (1, 4), (3, 4), (4, 3), (2, 2), (0, 3)]]
    T = _table(rows).cuda()
    assert sq[-1] + nq[-1] == Q.size(0) and sg[-1] + ng[-1] == G.size(0)
    for mutual in (False, True):
        got, want = _both(lambda q, g: _ops.match_pairs(q, g, T, 1024, 1024, mutual=mutual), Q, G)
        _equal(got, want)
        # given vs internal packing
        q16, g16 = _ops.pack_descriptors(Q), _ops.pack_descriptors(G)
        _equal(_ops.match_pairs(Q, G, T, 1024, 1024, q16, g16, mutual=mutual), got)
    # self pairs over one set with g is q (packed once)
    S = torch.cat([Q, G])
    off = Q.size(0)
    T2 = _table([[sq[0], nq[0], sq[0], nq[0]], [sq[2], nq[2], off + sg[1], ng[1]], [off + sg[4], ng[4], sq[1], nq[1]]]).cuda()
    S32 = S.float()
    _equal(_ops.match_pairs(S, S, T2, 1024, 1024, mutual=True), _ops.match_pairs(S32, S32, T2, 1024, 1024, mutual=True))


def _special_rows(dt):
    """A gallery and queries of exact and awkward values: one-hot rows (exactly +-1), all-zero rows, exact duplicates,
    components that are fp16 subnormals, and components whose 2^8 image (the packed operand) is an fp16 subnormal."""
    g = synth.unit_vectors(200, 128, 9)
    g[100:110] = 0.0
    g[100:110, torch.arange(10)] = 1.0
    g[110:120] = 0.0
    g[110:120, torch.arange(10, 20)] = -1.0
    g[120:126] = 0.0
    g[130:140, 40:60] = 3e-6          # fp16 subnormals (below 2^-14)
    g[140:150, 60:80] = 1.5e-7        # x * 2^8 below 2^-14: a subnormal packed operand
    g[150:160, 80:90] = -2e-9
    g = torch.cat([g, g[:50]])        # rows 200..249 duplicate rows 0..49 exactly
    q = torch.nn.functional.normalize(g[:100] + 0.03 * torch.randn(100, 128, generator=torch.Generator().manual_seed(1)), dim=1)
    q = torch.cat([q, g[100:160], torch.zeros(3, 128)])
    return q.to("cuda", dt), g.to("cuda", dt)


@pytest.mark.parametrize("dt", DTYPES, ids=IDS)
def test_special_values_and_ties(dt):
    from hardnetnas_b200 import _ops
    from hardnetnas_b200.matching import match_top2, mutual_nn_ratio
    q, g = _special_rows(dt)
    got, want = _both(match_top2, q, g)
    _equal(got, want)
    _equal(*_both(mutual_nn_ratio, q, g))
    # queries near rows 0..49, each duplicated at 200 + j: exact ties go to the lower index
    dup = (got[2][:100] < 50).nonzero().flatten()
    assert dup.numel() > 0
    assert torch.equal(got[3][dup], got[2][dup] + 200) and torch.equal(got[0][dup], got[1][dup])
    # the same rows through the batched and the pair-table forms
    _equal(*_both(lambda a, b: _ops.match_batched(a.unsqueeze(0), b.unsqueeze(0), mutual=True), q, g))
    T = _table([[0, q.size(0), 0, g.size(0)], [100, 63, 50, 200]]).cuda()
    _equal(*_both(lambda a, b: _ops.match_pairs(a, b, T, q.size(0), g.size(0), mutual=True), q, g))


@pytest.mark.parametrize("dt", DTYPES, ids=IDS)
def test_packing_is_bitwise_the_fp32_packing(dt):
    from hardnetnas_b200._ops import pack_descriptors
    q, g = _special_rows(dt)
    x = torch.cat([q, g, _set16(1000, 1, dt, 4)[0]])
    a, b = pack_descriptors(x), pack_descriptors(x.float())
    assert a.dtype == torch.float16 and torch.equal(a.view(torch.int16), b.view(torch.int16))


@pytest.mark.parametrize("dt", DTYPES, ids=IDS)
def test_real_descriptors(dt):
    from hardnetnas_b200.hardnet import HardNet
    from hardnetnas_b200.matching import match_top2, mutual_nn_ratio
    torch.manual_seed(0)
    model = HardNet()
    model.load_state_dict(synth.randomize_bn_stats(model.state_dict(), 3))
    model = model.cuda().eval()
    x = synth.make_patches(1024, 1234)
    p = synth.make_positives(x, 0.1, 7)
    a16, p16 = model(x.cuda(), out_dtype=dt), model(p.cuda(), out_dtype=dt)
    assert a16.dtype == dt
    got, want = _both(match_top2, a16, p16)
    _equal(got, want)
    _equal(*_both(mutual_nn_ratio, a16, p16))


@pytest.mark.parametrize("dt", DTYPES, ids=IDS)
def test_score_counters(dt):
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
    Q16, G16, KP1, KP2, VIS = Q.to("cuda", dt), G.to("cuda", dt), KP1.cuda(), KP2.cuda(), VIS.cuda()
    for fn, extra in ((matching.nearest_neighbor_match_score_batched, ()),
                      (matching.nearest_neighbor_threshold_match_score_batched, (1.0,)),
                      (matching.nearest_neighbor_distance_ratio_match_score_batched, ())):
        args = (*extra, 5.0) if extra else (5.0,)
        _equal(fn(Q16, G16, KP1, KP2, VIS, *args, len1=L1, len2=L2), fn(Q16.float(), G16.float(), KP1, KP2, VIS, *args, len1=L1, len2=L2))
    # pair form over the concatenated sets
    X1 = torch.cat([s[0] for s in sets]).to("cuda", dt)
    X2 = torch.cat([s[1] for s in sets]).to("cuda", dt)
    kp2_all = torch.cat([s[3] for s in sets]).cuda()
    T = matching.pair_table(torch.tensor([s[0].size(0) for s in sets]), list(range(B)), list(range(B)),
                            counts2=torch.tensor([s[1].size(0) for s in sets])).cuda()
    for fn, extra in ((matching.nearest_neighbor_match_score_pairs, ()),
                      (matching.nearest_neighbor_threshold_match_score_pairs, (1.0,)),
                      (matching.nearest_neighbor_distance_ratio_match_score_pairs, ())):
        args = (*extra, 5.0) if extra else (5.0,)
        _equal(fn(X1, X2, T, KP1, kp2_all, VIS, *args), fn(X1.float(), X2.float(), T, KP1, kp2_all, VIS, *args))


def _peak_bytes(fn):
    fn()   # warm-up: the workspace is grown, kernel attributes are set
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    out = fn()
    torch.cuda.synchronize()
    del out
    return torch.cuda.max_memory_allocated() - base


@pytest.mark.parametrize("dt", DTYPES, ids=IDS)
def test_no_fp32_copy(dt):
    """A 16-bit call on N rows allocates less than the N * 512 bytes an fp32 copy of them would take."""
    from hardnetnas_b200.matching import match_top2, match_top2_batched, match_top2_pairs, mutual_nn_ratio
    n = 1 << 16
    X = torch.nn.functional.normalize(torch.randn(n, 128, device="cuda"), dim=1).to(dt)
    T = _table([[4096 * i, 1024, 4096 * i + 2048, 1024] for i in range(8)]).cuda()
    assert _peak_bytes(lambda: match_top2_pairs(X, X, T, 1024, 1024)) < n * 512
    assert _peak_bytes(lambda: match_top2(X[: n // 2], X[n // 2:])) < n * 512
    assert _peak_bytes(lambda: mutual_nn_ratio(X[: n // 2], X[n // 2:], return_pairs=False)) < n * 512
    Xb = X.view(16, n // 16, 128)
    assert _peak_bytes(lambda: match_top2_batched(Xb[:8], Xb[8:])) < n * 512


@pytest.mark.parametrize("dt", DTYPES, ids=IDS)
def test_no_host_sync_and_graph_replay(dt):
    from hardnetnas_b200 import _ops
    Q, sq, nq, G, sg, ng = _two_sets([500, 129, 1024, 7], [1024, 600, 1, 300], seed=80)
    Qc, Gc = Q.to("cuda", dt), G.to("cuda", dt)
    T = _table([[sq[i], nq[i], sg[i], ng[i]] for i in range(4)]).cuda()
    Qb = torch.zeros(4, 1024, 128, device="cuda", dtype=dt)
    Gb = torch.zeros(4, 1024, 128, device="cuda", dtype=dt)
    for i in range(4):
        Qb[i, :nq[i]], Gb[i, :ng[i]] = Qc[sq[i]:sq[i] + nq[i]], Gc[sg[i]:sg[i] + ng[i]]
    L1 = torch.tensor(nq, dtype=torch.int32, device="cuda")
    L2 = torch.tensor(ng, dtype=torch.int32, device="cuda")
    calls = {"pairs": lambda: _ops.match_pairs(Qc, Gc, T, 1024, 1024, mutual=True),
             "batched": lambda: _ops.match_batched(Qb, Gb, L1, L2, mutual=True)}
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graphs, captured = {}, {}
    with torch.cuda.stream(s):
        for k, fn in calls.items():
            eager = fn()                                  # warm-up: workspace, kernel attributes
            torch.cuda.set_sync_debug_mode("error")
            try:
                again = fn()
            finally:
                torch.cuda.set_sync_debug_mode("default")
            _equal(eager, again)
    torch.cuda.synchronize()
    for k, fn in calls.items():
        graphs[k] = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graphs[k], stream=s):
            captured[k] = fn()
    # in-place edits of the rows, the table and the lengths; the replayed graphs follow them
    Qc.copy_(torch.nn.functional.normalize(Qc.float() + 0.05 * torch.randn_like(Qc, dtype=torch.float32), dim=1).to(dt))
    Gb[1, :300] = Gb[1, 300:600].clone()
    T.copy_(_table([[sq[2], 700, sg[0], 1024], [sq[0], 500, sg[3], 300], [sq[1], 129, sg[1], 0], [sq[3], 7, sg[2], 1]]).cuda())
    L2.copy_(torch.tensor([1024, 300, 1, 17], dtype=torch.int32))
    for k in calls:
        for t in captured[k]:
            t.zero_()
        graphs[k].replay()
    torch.cuda.synchronize()
    _equal(captured["pairs"], _ops.match_pairs(Qc.float(), Gc.float(), T, 1024, 1024, mutual=True))
    _equal(captured["batched"], _ops.match_batched(Qb.float(), Gb.float(), L1, L2, mutual=True))

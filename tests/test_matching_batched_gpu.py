"""Batched matching (hn_match_batched): every pair of a padded batch equals the per-pair calls bit for bit, padding never leaks
into another row or pair, and the call needs no host synchronisation."""
import numpy as np
import pytest
import torch

from oracle import losses_oracle, synth

pytestmark = pytest.mark.gpu

TIE_TAU = 1e-5
DIST_TOL = 2e-6
INF = float("inf")
EDGE = [0, 1, 2, 127, 128, 129, 255, 256, 257]


def _padded(sets, n):
    """[B, n, 128] with the per-pair rows in front and NaN padding behind them."""
    out = torch.full((len(sets), n, 128), float("nan"))
    for b, s in enumerate(sets):
        out[b, :s.size(0)] = s
    return out


def _batch(lq, lg, nq=None, ng=None, seed=0):
    qs, gs = [], []
    for b, (a, c) in enumerate(zip(lq, lg)):
        q, g, _ = synth.make_match_set(a, c, seed=seed + 7 * b)
        qs.append(q)
        gs.append(g)
    return qs, gs, _padded(qs, nq or max(max(lq), 1)), _padded(gs, ng or max(max(lg), 1))


def _lens(v):
    return torch.tensor(v, dtype=torch.int32, device="cuda")


def _assert_fill(d1, d2, i1, i2, rows):
    assert torch.all(d1[rows] == INF) and torch.all(d2[rows] == INF)
    assert torch.all(i1[rows] == -1) and torch.all(i2[rows] == -1)


def _oracle_parity(q, g, d1, d2, i1):
    """The _check rules of test_matching_gpu.py on one pair's valid rows."""
    d1, d2, i1 = d1.cpu(), d2.cpu(), i1.cpu()
    if g.size(0) < 2:
        v, i = losses_oracle.nn_match(q, g)
        assert (d1 - v).abs().max().item() <= DIST_TOL and torch.equal(i1, i)
        return
    lab, ia, da, db = losses_oracle.ratio_match(q, g, 0.7)
    assert (d1 - da).abs().max().item() <= DIST_TOL
    assert (d2 - db).abs().max().item() <= DIST_TOL
    bad = (i1 != ia).nonzero().flatten().tolist()
    if bad:
        d = losses_oracle.distance_matrix_vector_fdl(q[bad], g)
        for r, i in enumerate(bad):
            assert abs(d[r, i1[i]].item() - d[r, ia[i]].item()) <= TIE_TAU
    for i in ((d1 / d2 < 0.7) != lab).nonzero().flatten().tolist():
        assert abs((da[i] / db[i]).item() - 0.7) <= 1e-4


def _check_batch(qs, gs, Q, G, lq, lg, oracle=True):
    from hardnetnas_b200.matching import match_top2, match_top2_batched
    d1, d2, i1, i2 = match_top2_batched(Q.cuda(), G.cuda(), _lens(lq), _lens(lg))
    assert d1.shape == (Q.size(0), Q.size(1)) and i1.dtype == torch.int64
    for b, (q, g) in enumerate(zip(qs, gs)):
        a, c = lq[b], lg[b]
        if a and c:
            ref = match_top2(q.cuda(), g.cuda())
            for got, want in zip((d1[b, :a], d2[b, :a], i1[b, :a], i2[b, :a]), ref):
                assert torch.equal(got, want), (b, a, c)
            if oracle:
                _oracle_parity(q, g, d1[b, :a], d2[b, :a], i1[b, :a])
        _assert_fill(d1, d2, i1, i2, (b, slice(a if c else 0, None)))
    return d1, d2, i1, i2


def test_single_pair():
    qs, gs, Q, G = _batch([500], [700], seed=1)
    _check_batch(qs, gs, Q, G, [500], [700])


def test_lengths_default_to_all_rows():
    from hardnetnas_b200.matching import match_top2, match_top2_batched
    qs, gs, Q, G = _batch([300] * 3, [400] * 3, seed=2)
    out = match_top2_batched(Q.cuda(), G.cuda())
    for b in range(3):
        for got, want in zip(out, match_top2(qs[b].cuda(), gs[b].cuda())):
            assert torch.equal(got[b], want)


def test_eight_pairs_1000():
    qs, gs, Q, G = _batch([1000] * 8, [1000] * 8, seed=3)
    _check_batch(qs, gs, Q, G, [1000] * 8, [1000] * 8)


def test_300_small_pairs():
    qs, gs, Q, G = _batch([64] * 300, [64] * 300, seed=4)
    _check_batch(qs, gs, Q, G, [64] * 300, [64] * 300, oracle=False)


@pytest.mark.parametrize("nq,ng", [(300, 900), (900, 300), (129, 4097)])
def test_unequal_sides(nq, ng):
    qs, gs, Q, G = _batch([nq] * 5, [ng] * 5, seed=5)
    _check_batch(qs, gs, Q, G, [nq] * 5, [ng] * 5)


def test_ragged_lengths():
    """Lengths 0, 1, 2, 127, 128, 129, 255, 256, 257 on both sides and in many combinations; a length above the padded size
    is clamped to it, a negative one to 0."""
    lq = EDGE + EDGE + [257, 3]
    lg = EDGE[::-1] + EDGE[3:] + EDGE[:3] + [0, 257]
    qs, gs, Q, G = _batch(lq, lg, 257, 257, seed=6)
    _check_batch(qs, gs, Q, G, lq, lg)
    # out-of-range lengths are clamped on the device
    from hardnetnas_b200.matching import match_top2_batched
    clamped = match_top2_batched(Q.cuda(), G.cuda(), _lens([min(a, 257) for a in lq]), _lens(lg))
    wild = match_top2_batched(Q.cuda(), G.cuda(), _lens([1000 if a == 257 else a for a in lq]), _lens([-5 if c == 0 else c for c in lg]))
    for x, y in zip(clamped, wild):
        assert torch.equal(x, y)


def test_isolation_between_pairs_and_ties():
    from hardnetnas_b200.matching import match_top2_batched
    qs, gs, Q, G = _batch([200, 200], [600, 600], seed=7)
    gs[0][300] = gs[0][20]
    gs[0][40] = gs[0][20]
    qs[0][0] = gs[0][20]            # duplicate gallery rows inside pair 0: the lowest local index wins
    gs[1][5] = qs[0][0]             # a copy of pair 0's query in pair 1's gallery
    qs[1][7] = gs[0][20]
    Q, G = _padded(qs, 200), _padded(gs, 600)
    d1, d2, i1, i2 = _check_batch(qs, gs, Q, G, [200, 200], [600, 600])
    assert i1[0, 0].item() == 20 and i2[0, 0].item() == 40
    assert i1[1, 7].item() == 5
    assert torch.all(i1 < 600) and torch.all(i1 >= 0)
    # pair 1's planted row does not change what pair 0 sees
    alone = match_top2_batched(Q[:1].cuda(), G[:1].cuda())
    for x, y in zip(alone, (d1, d2, i1, i2)):
        assert torch.equal(x[0], y[0])


def test_mutual_matches_per_pair_and_oracle():
    from hardnetnas_b200.matching import mutual_nn_ratio, mutual_nn_ratio_batched
    lq, lg = [700, 1000, 333, 0, 2, 900], [800, 1500, 1, 50, 0, 1200]
    qs, gs, _, _ = _batch(lq, lg, seed=8)
    qs[1] = synth.unit_vectors(1000, 128, 6)          # unstructured: many weak claims
    gs[1] = synth.unit_vectors(1500, 128, 5)
    qs[5][10] = gs[5][100]
    qs[5][11] = gs[5][100]                            # two identical queries claim the same column: the lower row is mutual
    Q, G = _padded(qs, 1000), _padded(gs, 1500)
    mutual, ratio, ia, da, db = mutual_nn_ratio_batched(Q.cuda(), G.cuda(), _lens(lq), _lens(lg))
    assert mutual.dtype == torch.bool and mutual.shape == (6, 1000)
    for b, (q, g) in enumerate(zip(qs, gs)):
        a, c = lq[b], lg[b]
        assert not mutual[b, a if c else 0:].any()
        if not (a and c):
            continue
        _, m, r, f, d1, d2 = mutual_nn_ratio(q.cuda(), g.cuda(), return_pairs=False)
        assert torch.equal(mutual[b, :a], m) and torch.equal(ia[b, :a], f) and torch.equal(da[b, :a], d1), b
        assert torch.equal(ratio[b, :a], r) and torch.equal(db[b, :a], d2)
        rows = mutual[b, :a].nonzero().flatten()
        pairs = torch.stack([rows, ia[b, :a][rows]], dim=1).cpu()
        assert torch.equal(pairs, losses_oracle.mutual_nn(q, g)), b
    assert mutual[5, 10].item() and not mutual[5, 11].item() and ia[5, 10].item() == 100 and ia[5, 11].item() == 100


def _keypoints(n_q, n_g, truth, gen):
    kp2 = torch.cat([torch.zeros(n_g, 1), torch.rand(n_g, 2, generator=gen) * 480.0], dim=1)
    kp1w = torch.cat([torch.zeros(n_q, 1), torch.rand(n_q, 2, generator=gen) * 480.0], dim=1)
    has = truth >= 0
    kp1w[has, 1:3] = kp2[truth[has], 1:3] + 3.0 * torch.randn(int(has.sum()), 2, generator=gen)
    return kp1w, kp2, torch.rand(n_q, generator=gen) < 0.85


def test_score_counters_golden_pair_and_per_pair_equality(golden_dir):
    from hardnetnas_b200 import matching
    from oracle.make_golden_match_scores import COO_THRSH, DES_THRSH, inputs
    gold = np.load(golden_dir / "match_scores.npz")
    q0, g0, kp1w0, kp20, vis0 = inputs()
    gen = torch.Generator().manual_seed(5)
    sets = [(q0, g0, kp1w0, kp20, vis0)]
    for b, (a, c) in enumerate([(500, 1000), (768, 2048), (100, 1), (0, 30), (40, 0)]):
        q, g, truth = synth.make_match_set(a, c, seed=50 + b)
        sets.append((q, g, *_keypoints(a, c, truth, gen)))
    lq = [s[0].size(0) for s in sets]
    lg = [s[1].size(0) for s in sets]
    Q, G = _padded([s[0] for s in sets], 768).cuda(), _padded([s[1] for s in sets], 2048).cuda()
    KP1 = torch.full((len(sets), 768, 3), float("nan"))
    KP2 = torch.full((len(sets), 2048, 3), float("nan"))
    VIS = torch.ones(len(sets), 768, dtype=torch.bool)   # padding rows "visible": the lengths must still exclude them
    for b, s in enumerate(sets):
        KP1[b, :lq[b]], KP2[b, :lg[b]], VIS[b, :lq[b]] = s[2], s[3], s[4]
    KP1, KP2, VIS = KP1.cuda(), KP2.cuda(), VIS.cuda()
    L1, L2 = _lens(lq), _lens(lg)
    got = {
        "nn": matching.nearest_neighbor_match_score_batched(Q, G, KP1, KP2, VIS, COO_THRSH, L1, L2),
        "nn_thresh": matching.nearest_neighbor_threshold_match_score_batched(Q, G, KP1, KP2, VIS, DES_THRSH, COO_THRSH, L1, L2),
        "nn_ratio": matching.nearest_neighbor_distance_ratio_match_score_batched(Q, G, KP1, KP2, VIS, COO_THRSH, 0.7, L1, L2),
    }
    for key, (correct, predicted) in got.items():
        assert correct.is_cuda and correct.dtype == torch.int64 and correct.shape == (len(sets),)
        assert [correct[0].item(), predicted[0].item()] == gold[key].tolist(), key
    for b, (q, g, kp1w, kp2, vis) in enumerate(sets):
        if not (lq[b] and lg[b]):
            assert all(got[k][0][b].item() == 0 and got[k][1][b].item() == 1 for k in got)
            continue
        qc, gc, k1, k2, v = q.cuda(), g.cuda(), kp1w.cuda(), kp2.cuda(), vis.cuda()
        want = {
            "nn": matching.nearest_neighbor_match_score(qc, gc, k1, k2, v, COO_THRSH),
            "nn_thresh": matching.nearest_neighbor_threshold_match_score(qc, gc, k1, k2, v, DES_THRSH, COO_THRSH),
            "nn_ratio": matching.nearest_neighbor_distance_ratio_match_score(qc, gc, k1, k2, v, COO_THRSH),
        }
        for key in got:
            assert (got[key][0][b].item(), got[key][1][b].item()) == tuple(want[key]), (b, key)


def test_no_host_sync_and_graph_capture():
    from hardnetnas_b200 import _ops
    lq, lg = [500, 0, 129, 1024], [1024, 7, 1, 600]
    _, _, Q, G = _batch(lq, lg, 1024, 1024, seed=9)
    Q, G, L1, L2 = Q.cuda(), G.cuda(), _lens(lq), _lens(lg)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        eager = _ops.match_batched(Q, G, L1, L2, mutual=True)        # warm-up: workspace of this stream, kernel attributes
        torch.cuda.set_sync_debug_mode("error")
        try:
            again = _ops.match_batched(Q, G, L1, L2, mutual=True)
        finally:
            torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    for x, y in zip(eager, again):
        assert torch.equal(x, y)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        captured = _ops.match_batched(Q, G, L1, L2, mutual=True)
    for t in captured:
        t.fill_(0)
    graph.replay()
    torch.cuda.synchronize()
    for x, y in zip(eager, captured):
        assert torch.equal(x, y)


def test_argument_errors():
    from hardnetnas_b200 import _lib
    from hardnetnas_b200.matching import match_top2_batched
    q = torch.randn(2, 10, 128, device="cuda")
    with pytest.raises(ValueError):
        match_top2_batched(q[0], q[0])                                # rank 2
    with pytest.raises(ValueError):
        match_top2_batched(q[..., :64], q[..., :64])                  # not 128-d
    with pytest.raises(ValueError):
        match_top2_batched(q, q, torch.tensor([3, 4, 5], device="cuda"))   # lengths of the wrong shape
    with pytest.raises(ValueError):
        match_top2_batched(q, q, None, torch.tensor([3.0, 4.0], device="cuda"))
    with pytest.raises(ValueError):
        match_top2_batched(q, q[:1])                                   # different pair counts
    with pytest.raises(_lib.HardnetB200Error):
        match_top2_batched(q[:, :0], q)                                # no query rows
    d1, _, i1, _ = match_top2_batched(q, q, torch.tensor([3, 4]))      # CPU lengths are copied to the device
    assert torch.all(i1[0, 3:] == -1) and torch.all(i1[1, 4:] == -1)


def test_flat_rows_past_2_25():
    """More than 2^25 flat query rows: the row index fits 32 bits, the element offset row * 128 does not. Pairs at the end of
    the batch must still read their own query rows (bit-equal to per-pair calls)."""
    from hardnetnas_b200.matching import match_top2, match_top2_batched
    B, nq, ng = (1 << 21) + 64, 16, 8          # 2^25 + 1024 query rows (17 GB fp32), 8.6 GB of gallery rows
    if torch.cuda.mem_get_info()[0] < (64 << 30):
        pytest.skip("needs 64 GB of free device memory")
    gen = torch.Generator(device="cuda").manual_seed(12)
    Q = torch.randn(B, nq, 128, device="cuda", generator=gen)
    Q /= Q.norm(dim=2, keepdim=True)
    G = torch.randn(B, ng, 128, device="cuda", generator=gen)
    G /= G.norm(dim=2, keepdim=True)
    out = match_top2_batched(Q, G)
    for b in (0, (1 << 21) - 1, 1 << 21, B - 2, B - 1):   # pair 2^21 starts at flat row 2^25
        ref = match_top2(Q[b], G[b])
        for got, want in zip(out, ref):
            assert torch.equal(got[b], want), b
    del Q, G, out
    torch.cuda.empty_cache()

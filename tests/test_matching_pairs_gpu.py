"""Pair-table matching (hn_match_pairs): every pair of a table over concatenated descriptor sets equals the per-pair calls on
its slices bit for bit, equals the padded form, never reads rows outside its ranges, and needs no host synchronisation."""
import numpy as np
import pytest
import torch

from oracle import synth
from test_matching_batched_gpu import _keypoints, _oracle_parity

pytestmark = pytest.mark.gpu

INF = float("inf")
LENS = [0, 1, 2, 127, 128, 129, 255, 256, 257, 997, 1001]


def _concat(blocks, lead=3, seed=0):
    """One set from per-image blocks, after `lead` unrelated rows (so that image starts are odd). -> (set, starts, lengths)."""
    rows = [synth.unit_vectors(lead, 128, seed)] if lead else []
    starts, off = [], lead
    for b in blocks:
        starts.append(off)
        rows.append(b)
        off += b.size(0)
    return torch.cat(rows), starts, [b.size(0) for b in blocks]


def _two_sets(lq, lg, seed):
    """Query and gallery images of make_match_set pairs (image i of one set matches image i of the other)."""
    qs, gs = [], []
    for i, (a, c) in enumerate(zip(lq, lg)):
        q, g, _ = synth.make_match_set(a, c, seed=seed + 7 * i)
        qs.append(q)
        gs.append(g)
    Q, sq, nq = _concat(qs, 3, seed + 1)
    G, sg, ng = _concat(gs, 5, seed + 2)
    return Q, sq, nq, G, sg, ng


def _clamp(table, nq_rows, ng_rows, max_q, max_g):
    """The device-side clamping of hn_match_pairs, on the host."""
    out = []
    for qs, ql, gs, gl in table.tolist():
        qs, gs = min(max(qs, 0), nq_rows), min(max(gs, 0), ng_rows)
        out.append((qs, max(0, min(ql, max_q, nq_rows - qs)), gs, max(0, min(gl, max_g, ng_rows - gs))))
    return out


def _fill_ok(d1, d2, i1, i2, p, start):
    assert torch.all(d1[p, start:] == INF) and torch.all(d2[p, start:] == INF)
    assert torch.all(i1[p, start:] == -1) and torch.all(i2[p, start:] == -1)


def _check_pairs(Q, G, table, max_q, max_g, mutual=True, oracle_every=0, same=False):
    """Every pair against match_top2 / mutual_nn_ratio on its clamped slices; rows past the pair's length are fill."""
    from hardnetnas_b200.matching import match_top2, match_top2_pairs, mutual_nn_ratio, mutual_nn_ratio_pairs
    Qc = Q.cuda()
    Gc = Qc if same else G.cuda()
    T = table.cuda()
    d1, d2, i1, i2 = match_top2_pairs(Qc, Gc, T, max_q, max_g)
    assert d1.shape == (table.size(0), max_q) and i1.dtype == torch.int64
    mu = mutual_nn_ratio_pairs(Qc, Gc, T, max_q, max_g) if mutual else None
    for p, (qs, ql, gs, gl) in enumerate(_clamp(table, Q.size(0), Gc.size(0), max_q, max_g)):
        if ql and gl:
            q, g = Qc[qs:qs + ql], Gc[gs:gs + gl]
            ref = match_top2(q, g)
            for got, want in zip((d1[p, :ql], d2[p, :ql], i1[p, :ql], i2[p, :ql]), ref):
                assert torch.equal(got, want), (p, qs, ql, gs, gl)
            if mu is not None:
                _, m, r, f, a, b = mutual_nn_ratio(q, g, return_pairs=False)
                assert torch.equal(mu[0][p, :ql], m) and torch.equal(mu[1][p, :ql], r) and torch.equal(mu[2][p, :ql], f), p
                assert torch.equal(mu[3][p, :ql], a) and torch.equal(mu[4][p, :ql], b), p
            if oracle_every and p % oracle_every == 0:
                _oracle_parity(q.cpu(), g.cpu(), d1[p, :ql], d2[p, :ql], i1[p, :ql])
        _fill_ok(d1, d2, i1, i2, p, ql if gl else 0)
        if mu is not None:
            assert not mu[0][p, ql if gl else 0:].any()
    return (d1, d2, i1, i2), mu


def _table(rows):
    return torch.tensor(rows, dtype=torch.int32)


def _mixed_case():
    lq = LENS + [1000, 129]
    lg = LENS[::-1] + [1003, 257]
    Q, sq, nq, G, sg, ng = _two_sets(lq, lg, seed=10)
    rows = [[sq[i], nq[i], sg[i], ng[i]] for i in range(len(lq))]                         # the natural pairs
    rows += [[sq[i], nq[i], sg[(i * 5 + 3) % len(lg)], ng[(i * 5 + 3) % len(lg)]] for i in range(len(lq))]   # images reused
    rows += [[sq[-2], nq[-2], G.size(0) - 700, 700]]                                       # gallery range ends at the last row
    rows += [[Q.size(0) - 129, 129, sg[-2], ng[-2]]]                                       # query range ends at the last row
    rows += [[sq[-2] + 1, 333, sg[-2] + 3, 517]]                                           # odd starts inside an image
    return Q, G, _table(rows), max(lq), max(lg)


def test_per_pair_equality_mixed_lengths_and_reused_images():
    Q, G, table, max_q, max_g = _mixed_case()
    _check_pairs(Q, G, table, max_q, max_g, oracle_every=3)


def test_self_pairs_same_set():
    """g is q: (i, i) self pairs and (i, j) pairs inside one set, packed once."""
    blocks = [synth.make_match_set(n, 8, seed=20 + n)[0] for n in (300, 129, 1000, 1, 256)]
    X, s, n = _concat(blocks, 1, seed=21)
    rows = [[s[i], n[i], s[i], n[i]] for i in range(len(n))] + [[s[i], n[i], s[j], n[j]] for i in range(len(n)) for j in range(len(n)) if i != j]
    _check_pairs(X, X, _table(rows), 1000, 1000, same=True)


def test_equal_to_padded_form():
    from hardnetnas_b200.matching import match_top2_batched, match_top2_pairs, mutual_nn_ratio_batched, mutual_nn_ratio_pairs
    Q, G, table, max_q, max_g = _mixed_case()
    cl = _clamp(table, Q.size(0), G.size(0), max_q, max_g)
    P = table.size(0)
    Qp = torch.full((P, max_q, 128), float("nan"))
    Gp = torch.full((P, max_g, 128), float("nan"))
    for p, (qs, ql, gs, gl) in enumerate(cl):
        Qp[p, :ql] = Q[qs:qs + ql]
        Gp[p, :gl] = G[gs:gs + gl]
    L1 = torch.tensor([c[1] for c in cl], dtype=torch.int32, device="cuda")
    L2 = torch.tensor([c[3] for c in cl], dtype=torch.int32, device="cuda")
    Qc, Gc, T = Q.cuda(), G.cuda(), table.cuda()
    for got, want in zip(match_top2_pairs(Qc, Gc, T, max_q, max_g), match_top2_batched(Qp.cuda(), Gp.cuda(), L1, L2)):
        assert torch.equal(got, want)
    for got, want in zip(mutual_nn_ratio_pairs(Qc, Gc, T, max_q, max_g), mutual_nn_ratio_batched(Qp.cuda(), Gp.cuda(), L1, L2)):
        assert torch.equal(got, want)


def test_rows_outside_every_pair_never_matter():
    from hardnetnas_b200.matching import match_top2_pairs, mutual_nn_ratio_pairs
    Q, sq, nq, G, sg, ng = _two_sets([200, 300, 129, 257], [500, 128, 400, 300], seed=30)
    # pairs use only parts of the images: rows 20.. of image 0, the first 100 rows of image 1, ...
    table = _table([[sq[0] + 20, 180, sg[0], 400], [sq[1], 100, sg[1] + 28, 100], [sq[2], 129, sg[2], 400], [sq[3], 257, sg[3], 250]])
    used_q = torch.zeros(Q.size(0), dtype=torch.bool)
    used_g = torch.zeros(G.size(0), dtype=torch.bool)
    for qs, ql, gs, gl in table.tolist():
        used_q[qs:qs + ql] = True
        used_g[gs:gs + gl] = True
    Qn, Gn = Q.clone(), G.clone()
    Qn[~used_q] = float("nan")
    Gn[~used_g] = float("nan")
    T = table.cuda()
    a = match_top2_pairs(Q.cuda(), G.cuda(), T, 257, 400) + mutual_nn_ratio_pairs(Q.cuda(), G.cuda(), T, 257, 400)
    b = match_top2_pairs(Qn.cuda(), Gn.cuda(), T, 257, 400) + mutual_nn_ratio_pairs(Qn.cuda(), Gn.cuda(), T, 257, 400)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    # an exact copy of a query row right after a pair's gallery range (the next image, or unused rows) is never returned
    Gc = G.clone()
    for p, (qs, ql, gs, gl) in enumerate(table.tolist()):
        Gc[gs + gl] = Q[qs]
        Gc[gs + gl + 1] = Q[qs + 1]
    (d1, _, i1, _), _ = _check_pairs(Q, Gc, table, 257, 400)
    assert torch.all(i1[:, :2] >= 0) and torch.all(d1[:, :2] > 1e-3)


def test_table_clamping():
    Q, sq, nq, G, sg, ng = _two_sets([300, 200], [400, 250], seed=40)
    nqr, ngr = Q.size(0), G.size(0)
    rows = [[nqr + 5, 10, sg[0], 100],          # query start past the set: no rows
            [sq[0], 50, ngr + 100, 20],         # gallery start past the set: every row is fill
            [nqr - 40, 300, sg[1], 250],        # start + len past the set: 40 rows
            [sq[1], 200, ngr - 7, 100],         # 7 gallery rows
            [sq[0], -5, sg[0], 400],            # negative lengths
            [sq[0], 300, sg[0], -1],
            [-9, 300, -2, 400],                 # negative starts: clamped to row 0
            [sq[0], 300, sg[0], 400],           # len > max on both sides: clamped to max_q = 256, max_g = 300
            [sq[1], 1, sg[1], 1]]
    _check_pairs(Q, G, _table(rows), 256, 300)


def test_packed_operands_and_split_calls():
    from hardnetnas_b200._ops import pack_descriptors
    from hardnetnas_b200.matching import match_top2_pairs, mutual_nn_ratio_pairs
    Q, G, table, max_q, max_g = _mixed_case()
    Qc, Gc, T = Q.cuda(), G.cuda(), table.cuda()
    q16, g16 = pack_descriptors(Qc), pack_descriptors(Gc)
    inside = match_top2_pairs(Qc, Gc, T, max_q, max_g)
    given = match_top2_pairs(Qc, Gc, T, max_q, max_g, q16, g16)
    half = table.size(0) // 2
    first = match_top2_pairs(Qc, Gc, T[:half], max_q, max_g, q16, g16)
    second = match_top2_pairs(Qc, Gc, T[half:], max_q, max_g, q16, g16)
    for a, b, c, d in zip(inside, given, first, second):
        assert torch.equal(a, b) and torch.equal(a, torch.cat([c, d]))
    m_inside = mutual_nn_ratio_pairs(Qc, Gc, T, max_q, max_g)
    m_given = mutual_nn_ratio_pairs(Qc, Gc, T, max_q, max_g, des1_16=q16, des2_16=g16)
    for a, b in zip(m_inside, m_given):
        assert torch.equal(a, b)


def test_max_lengths_from_the_table():
    """max_len* = None reads the largest clamped lengths from the table; the result equals the call with them given."""
    from hardnetnas_b200.matching import match_top2_pairs
    Q, G, table, max_q, max_g = _mixed_case()
    a = match_top2_pairs(Q.cuda(), G.cuda(), table.cuda())
    b = match_top2_pairs(Q.cuda(), G.cuda(), table.cuda(), max_q, max_g)
    assert a[0].shape == (table.size(0), max_q)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def test_no_host_sync_and_graph_follows_table_edits():
    from hardnetnas_b200 import _ops
    Q, sq, nq, G, sg, ng = _two_sets([500, 129, 1024, 7], [1024, 600, 1, 300], seed=50)
    Qc, Gc = Q.cuda(), G.cuda()
    q16, g16 = _ops.pack_descriptors(Qc), _ops.pack_descriptors(Gc)
    T = _table([[sq[i], nq[i], sg[i], ng[i]] for i in range(4)]).cuda()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        eager = _ops.match_pairs(Qc, Gc, T, 1024, 1024, q16, g16, mutual=True)   # warm-up: workspace, kernel attributes
        torch.cuda.set_sync_debug_mode("error")
        try:
            again = _ops.match_pairs(Qc, Gc, T, 1024, 1024, q16, g16, mutual=True)
        finally:
            torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    for x, y in zip(eager, again):
        assert torch.equal(x, y)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        captured = _ops.match_pairs(Qc, Gc, T, 1024, 1024, q16, g16, mutual=True)
    for t in captured:
        t.fill_(0)
    graph.replay()
    torch.cuda.synchronize()
    for x, y in zip(eager, captured):
        assert torch.equal(x, y)
    # edit the device table in place: other images, other lengths; the replayed graph follows it
    new = _table([[sq[2], 700, sg[0], 1024], [sq[0], 500, sg[3], 300], [sq[1], 129, sg[1], 0], [sq[3], 7, sg[2], 1]])
    T.copy_(new.cuda())
    graph.replay()
    torch.cuda.synchronize()
    want = _ops.match_pairs(Qc, Gc, new.cuda(), 1024, 1024, q16, g16, mutual=True)
    for x, y in zip(want, captured):
        assert torch.equal(x, y)


def test_argument_errors():
    from hardnetnas_b200 import _lib
    from hardnetnas_b200.matching import match_top2_pairs
    x = synth.unit_vectors(100, 128, 1).cuda()
    t = _table([[0, 50, 50, 50]]).cuda()
    with pytest.raises(ValueError):
        match_top2_pairs(x, x, t[:, :3], 50, 50)                     # not [P, 4]
    with pytest.raises(ValueError):
        match_top2_pairs(x, x, t.float(), 50, 50)                    # not an integer table
    with pytest.raises(ValueError):
        match_top2_pairs(x, x, t, 50, 50, des1_16=torch.zeros(99, 128, dtype=torch.float16, device="cuda"))
    with pytest.raises(_lib.HardnetB200Error):
        match_top2_pairs(x, x, t[:0], 50, 50)                        # no pairs
    d1, _, i1, _ = match_top2_pairs(x, x, _table([[0, 50, 50, 50]]).long(), 64, 64)   # CPU int64 tables are copied to the device
    assert d1.shape == (1, 64) and torch.all(i1[0, 50:] == -1) and torch.all(i1[0, :50] >= 0)


def test_start_past_row_2_25():
    """A pair that starts past row 2^25: the row index fits 32 bits, the element offset row * 128 does not."""
    from hardnetnas_b200._ops import pack_descriptors
    from hardnetnas_b200.matching import match_top2, match_top2_pairs, mutual_nn_ratio, mutual_nn_ratio_pairs
    n = (1 << 25) + 4096                     # 17 GB of fp32 rows, 8.6 GB packed; one set on both sides
    if torch.cuda.mem_get_info()[0] < (48 << 30):
        pytest.skip("needs 48 GB of free device memory")
    gen = torch.Generator(device="cuda").manual_seed(13)
    X = torch.empty(n, 128, device="cuda")
    for c in range(0, n, 1 << 22):
        v = torch.randn(min(1 << 22, n - c), 128, device="cuda", generator=gen)
        X[c:c + v.size(0)] = v / v.norm(dim=1, keepdim=True)
    x16 = pack_descriptors(X)
    big = 1 << 25
    rows = [[0, 300, big + 100, 700], [big + 1001, 257, big + 2000, 2096], [big + 3, 1000, 17, 129], [n - 200, 200, n - 1000, 1000]]
    T = _table(rows).cuda()
    out = match_top2_pairs(X, X, T, 1000, 2096, x16, x16)
    mu = mutual_nn_ratio_pairs(X, X, T, 1000, 2096, des1_16=x16, des2_16=x16)
    for p, (qs, ql, gs, gl) in enumerate(rows):
        q, g = X[qs:qs + ql], X[gs:gs + gl]
        for got, want in zip(out, match_top2(q, g)):
            assert torch.equal(got[p, :ql], want), p
        _, m, _, f, _, _ = mutual_nn_ratio(q, g, return_pairs=False)
        assert torch.equal(mu[0][p, :ql], m) and torch.equal(mu[2][p, :ql], f), p
    del X, x16, out, mu
    torch.cuda.empty_cache()


def test_score_counters_golden_and_per_pair_equality(golden_dir):
    from hardnetnas_b200 import matching
    from oracle.make_golden_match_scores import COO_THRSH, DES_THRSH, inputs
    gold = np.load(golden_dir / "match_scores.npz")
    q0, g0, kp1w0, kp20, vis0 = inputs()
    gen = torch.Generator().manual_seed(6)
    qs, gs, kq, kg, vis, truth = [q0], [g0], [kp1w0], [kp20], [vis0], []
    for i, (a, c) in enumerate([(500, 1000), (129, 2048), (100, 1), (0, 30), (40, 0)]):
        q, g, t = synth.make_match_set(a, c, seed=60 + i)
        k1, k2, v = _keypoints(a, c, t, gen)
        qs.append(q)
        gs.append(g)
        kq.append(k1)
        kg.append(k2)
        vis.append(v)
    Q, sq, nq = _concat(qs, 3, seed=61)
    G, sg, ng = _concat(gs, 5, seed=62)
    KP2 = torch.cat([torch.full((5, 3), float("nan"))] + kg)          # keypoints of the gallery set, row for row
    n_img = len(qs)
    pairs = [(i, i) for i in range(n_img)] + [(1, 2), (2, 1)]            # the golden pair first; image 1 and 2 reused
    table = _table([[sq[i], nq[i], sg[j], ng[j]] for i, j in pairs])
    max_q = max(nq)
    KP1 = torch.full((len(pairs), max_q, 3), float("nan"))
    VIS = torch.ones(len(pairs), max_q, dtype=torch.bool)               # padding rows "visible": the lengths must exclude them
    for p, (i, j) in enumerate(pairs):
        # kp1w of a pair is the query image's keypoints warped into the gallery image; for the reused pairs any warp will do
        KP1[p, :nq[i]] = kq[i]
        VIS[p, :nq[i]] = vis[i]
    Qc, Gc, T, KP1, KP2, VIS = Q.cuda(), G.cuda(), table.cuda(), KP1.cuda(), KP2.cuda(), VIS.cuda()
    got = {
        "nn": matching.nearest_neighbor_match_score_pairs(Qc, Gc, T, KP1, KP2, VIS, COO_THRSH),
        "nn_thresh": matching.nearest_neighbor_threshold_match_score_pairs(Qc, Gc, T, KP1, KP2, VIS, DES_THRSH, COO_THRSH),
        "nn_ratio": matching.nearest_neighbor_distance_ratio_match_score_pairs(Qc, Gc, T, KP1, KP2, VIS, COO_THRSH, 0.7),
    }
    for key, (correct, predicted) in got.items():
        assert correct.is_cuda and correct.dtype == torch.int64 and correct.shape == (len(pairs),)
        assert [correct[0].item(), predicted[0].item()] == gold[key].tolist(), key
    for p, (i, j) in enumerate(pairs):
        if not (nq[i] and ng[j]):
            assert all(got[k][0][p].item() == 0 and got[k][1][p].item() == 1 for k in got)
            continue
        q, g = Qc[sq[i]:sq[i] + nq[i]], Gc[sg[j]:sg[j] + ng[j]]
        k1, k2, v = KP1[p, :nq[i]], KP2[sg[j]:sg[j] + ng[j]], VIS[p, :nq[i]]
        want = {
            "nn": matching.nearest_neighbor_match_score(q, g, k1, k2, v, COO_THRSH),
            "nn_thresh": matching.nearest_neighbor_threshold_match_score(q, g, k1, k2, v, DES_THRSH, COO_THRSH),
            "nn_ratio": matching.nearest_neighbor_distance_ratio_match_score(q, g, k1, k2, v, COO_THRSH),
        }
        for key in got:
            assert (got[key][0][p].item(), got[key][1][p].item()) == tuple(want[key]), (p, key)

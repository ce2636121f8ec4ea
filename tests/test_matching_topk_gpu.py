"""k-nearest-neighbour matching on the GPU: exact against a float64 oracle for k = 1..8, consistent bit for bit with the top-2
calls and across k, exact on planted ties and on rows whose approximate dot order inverts the exact one across more than eight
chunks of one list, the same on every row type, and the pair-table form (per pair, padded batches, CUDA graphs)."""
import pytest
import torch

from oracle import knn_oracle, synth

pytestmark = pytest.mark.gpu

INF = float("inf")


def _dist64(q, g, idx):
    """float64 FDLNet distances of the columns idx [n, k] (-1: +inf)."""
    qd, gd = q.double(), g.double()
    dot = torch.einsum("nd,nkd->nk", qd, gd[idx.clamp(min=0)])
    d = torch.sqrt((2 - 2 * dot).clamp(1e-8, 4.0))
    return torch.where(idx >= 0, d, torch.full_like(d, INF))


def _check_sorted(D, I):
    """Ascending by (distance, index), no repeated index, +inf / -1 only in trailing slots."""
    assert torch.all((I == -1) == (D == INF))
    lo, hi, ilo, ihi = D[:, :-1], D[:, 1:], I[:, :-1], I[:, 1:]
    assert torch.all((lo < hi) | ((lo == hi) & ((ilo < ihi) | (ihi == -1))))
    for row in I.tolist():
        v = [x for x in row if x >= 0]
        assert len(v) == len(set(v))


def _check_oracle(q, g, D, I, k):
    """Against the float64 oracle: the same indices except at near ties, distances through d^2 within 5e-6."""
    D64, I64 = knn_oracle.knn_match(q, g, k, chunk=512)
    assert D.shape == I.shape == (q.size(0), k)
    assert torch.equal(I == -1, I64 == -1)
    got64 = _dist64(q, g, I)
    valid = I >= 0
    diff = I != I64
    assert torch.all((got64[diff] - D64[diff]).abs() <= 1e-5), "an index differs from the oracle beyond a near tie"
    assert torch.all(((D.double() ** 2 - got64 ** 2).abs() <= 5e-6)[valid])
    _check_sorted(D, I)


SHAPES = [(5, 3), (9, 8), (300, 1001), (257, 130), (1000, 4097), (3, 20000), (511, 640), (700, 128), (2000, 2050)]


@pytest.mark.parametrize("nq,ng", SHAPES)
def test_against_float64_oracle(nq, ng):
    from hardnetnas_b200.matching import match_topk
    q, g, _ = synth.make_match_set(nq, ng, seed=nq + ng)
    q, g = q.cuda(), g.cuda()
    for k in range(1, 9):
        D, I = match_topk(q, g, k)
        _check_oracle(q, g, D, I, k)


def test_64k_sample_and_prefixes():
    from hardnetnas_b200.matching import match_topk
    q, g, _ = synth.make_match_set(65536, 65536, seed=11)
    q, g = q.cuda(), g.cuda()
    D8, I8 = match_topk(q, g, 8)
    rows = torch.randperm(65536, generator=torch.Generator().manual_seed(0))[:256].cuda()
    _check_oracle(q[rows], g, D8[rows], I8[rows], 8)
    for k in range(1, 8):
        D, I = match_topk(q, g, k)
        assert torch.equal(D, D8[:, :k]) and torch.equal(I, I8[:, :k])


@pytest.mark.parametrize("nq,ng", [(300, 1001), (4096, 8192), (1000, 4097)])
def test_consistent_with_top2_and_nearest_neighbour(nq, ng):
    from hardnetnas_b200.matching import match_top2, match_topk, nearest_neighbor_match
    q, g, _ = synth.make_match_set(nq, ng, seed=3 * nq)
    q, g = q.cuda(), g.cuda()
    da, db, ia, ib = match_top2(q, g)
    D2, I2 = match_topk(q, g, 2)
    assert torch.equal(D2[:, 0], da) and torch.equal(D2[:, 1], db) and torch.equal(I2[:, 0], ia) and torch.equal(I2[:, 1], ib)
    d1, i1 = nearest_neighbor_match(q, g)
    D1, I1 = match_topk(q, g, 1)
    assert torch.equal(D1[:, 0], d1) and torch.equal(I1[:, 0], i1)
    D8, I8 = match_topk(q, g, 8)
    for k in range(1, 8):
        D, I = match_topk(q, g, k)
        assert torch.equal(D, D8[:, :k]) and torch.equal(I, I8[:, :k])


def test_copies_spread_over_many_chunks():
    """24 exact copies of each query in 24 chunks of one segment: the answer is the k lowest copy indices."""
    from hardnetnas_b200.matching import match_topk
    ng = 4096   # 32 tiles: 16 segments of 256 columns
    g = synth.unit_vectors(ng, 128, 9)
    q = synth.unit_vectors(16, 128, 10)
    want = []
    for s in range(16):
        cols = [s * 256 + 8 * c + (c % 8) for c in range(24)]
        g[cols] = q[s]
        want.append(cols[:8])
    D, I = match_topk(q.cuda(), g.cuda(), 8)
    assert I.tolist() == want
    assert torch.all(D == D[:, :1])
    _check_oracle(q.cuda(), g.cuda(), D, I, 8)


def _inverted_set(dtype=torch.float32, n_clusters=16, per=24, step=5e-6, seed=0):
    """Per query, `per` gallery rows around it in `per` chunks of one segment, with exact dots 1 - (0.005 + j * step) and the
    best ones in the last chunks, so the approximate dot order differs from the exact one across more than eight chunks of one
    list: the k nearest can only be found through the list's dropped maximum."""
    gen = torch.Generator().manual_seed(seed)
    ng = 4096
    g = synth.unit_vectors(ng, 128, seed + 1)
    q = synth.unit_vectors(n_clusters, 128, seed + 2)
    for s in range(n_clusters):
        u = torch.randn(per, 128, generator=gen, dtype=torch.float64)
        qd = q[s].double()
        u -= (u @ qd)[:, None] * qd[None]
        u /= u.norm(dim=1, keepdim=True)
        c = 1 - (0.005 + step * torch.arange(per, dtype=torch.float64))
        rows = c[:, None] * qd[None] + torch.sqrt(1 - c * c)[:, None] * u
        cols = [s * 256 + 8 * (per - 1 - j) + (j % 8) for j in range(per)]
        g[cols] = rows.float()
    if dtype != torch.float32:
        q, g = q.to(dtype), g.to(dtype)
    return q.cuda(), g.cuda()


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16, torch.float8_e4m3fn])
def test_inverted_approximate_order(dtype):
    from hardnetnas_b200.matching import match_topk
    q, g = _inverted_set(dtype)
    for k in (1, 2, 5, 8):
        D, I = match_topk(q, g, k)
        _check_oracle(q.float(), g.float(), D, I, k)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16, torch.float8_e4m3fn])
def test_row_types_equal_the_fp32_call(dtype):
    from hardnetnas_b200._ops import pack_descriptors
    from hardnetnas_b200.matching import match_topk
    q, g, _ = synth.make_match_set(1000, 4097, seed=17)
    q, g = q.cuda().to(dtype), g.cuda().to(dtype)
    for k in (1, 3, 8):
        D, I = match_topk(q, g, k)
        Df, If = match_topk(q.float(), g.float(), k)
        assert torch.equal(D, Df) and torch.equal(I, If)
    from hardnetnas_b200._ops import match_topk as ops_topk
    Dp, Ip = ops_topk(q, g, 8, q16=pack_descriptors(q), g16=pack_descriptors(g))
    D, I = match_topk(q, g, 8)
    assert torch.equal(Dp, D) and torch.equal(Ip.long(), I)


def _table(rows):
    return torch.tensor(rows, dtype=torch.int32)


def _pairs_case(seed=40):
    lq, lg = [500, 129, 1024, 7, 0, 300], [1024, 600, 1, 300, 50, 0]
    qs, gs = [], []
    for i, (a, c) in enumerate(zip(lq, lg)):
        q, g, _ = synth.make_match_set(max(a, 1), max(c, 1), seed=seed + 7 * i)
        qs.append(q[:a])
        gs.append(g[:c])
    lead_q, lead_g = synth.unit_vectors(3, 128, seed + 1), synth.unit_vectors(5, 128, seed + 2)
    Q, G = torch.cat([lead_q] + qs), torch.cat([lead_g] + gs)
    sq = [3 + sum(lq[:i]) for i in range(len(lq))]
    sg = [5 + sum(lg[:i]) for i in range(len(lg))]
    rows = [[sq[i], lq[i], sg[i], lg[i]] for i in range(len(lq))]
    rows += [[sq[2], 1024, sg[0], 1024], [sq[0], 500, sg[2], 1], [Q.size(0) + 10, 5, 0, 5], [sq[1], 129, G.size(0) - 3, 100]]
    return Q.cuda(), G.cuda(), _table(rows)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.float8_e4m3fn])
def test_pairs_equal_per_pair_calls(dtype):
    """Every pair equals match_topk on its (clamped) slices; empty pairs, zero-length galleries and clamped starts fill."""
    from hardnetnas_b200.matching import match_topk, match_topk_pairs
    Q, G, T = _pairs_case()
    Q, G = Q.to(dtype), G.to(dtype)
    for k in (1, 4, 8):
        D, I = match_topk_pairs(Q, G, T.cuda(), k, 1024, 1024)
        assert D.shape == (T.size(0), 1024, k)
        for p, (qs, ql, gs, gl) in enumerate(T.tolist()):
            qs, gs = min(max(qs, 0), Q.size(0)), min(max(gs, 0), G.size(0))
            ql, gl = max(0, min(ql, 1024, Q.size(0) - qs)), max(0, min(gl, 1024, G.size(0) - gs))
            assert torch.all(D[p, ql:] == INF) and torch.all(I[p, ql:] == -1)
            if ql == 0:
                continue
            if gl == 0:
                assert torch.all(D[p] == INF) and torch.all(I[p] == -1)
                continue
            d, i = match_topk(Q[qs:qs + ql], G[gs:gs + gl], k)
            assert torch.equal(D[p, :ql], d) and torch.equal(I[p, :ql], i), p


def test_padded_batch_as_pair_table():
    from hardnetnas_b200.matching import match_topk, match_topk_pairs
    B, N1, N2 = 5, 300, 700
    q = torch.stack([synth.make_match_set(N1, N2, seed=b)[0] for b in range(B)]).cuda()
    g = torch.stack([synth.make_match_set(N1, N2, seed=b)[1] for b in range(B)]).cuda()
    len1, len2 = torch.tensor([300, 0, 17, 299, 128]), torch.tensor([700, 5, 0, 3, 640])
    T = torch.stack([torch.arange(B) * N1, len1, torch.arange(B) * N2, len2], 1).to(torch.int32).cuda()
    D, I = match_topk_pairs(q.flatten(0, 1), g.flatten(0, 1), T, 6, N1, N2)
    for b in range(B):
        a, c = int(len1[b]), int(len2[b])
        if a and c:
            d, i = match_topk(q[b, :a], g[b, :c], 6)
            assert torch.equal(D[b, :a], d) and torch.equal(I[b, :a], i)
            _check_oracle(q[b, :a], g[b, :c], D[b, :a], I[b, :a], 6)
        assert torch.all(I[b, a:] == -1) and torch.all(D[b, a:] == INF)
        if not c:
            assert torch.all(I[b] == -1)


def test_pairs_graph_capture_follows_table_edits():
    from hardnetnas_b200 import _ops
    Q, G, T = _pairs_case(seed=60)
    T = T[:4].contiguous().cuda()
    q16, g16 = _ops.pack_descriptors(Q), _ops.pack_descriptors(G)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        eager = _ops.match_pairs_topk(Q, G, T, 8, 1024, 1024, q16, g16)   # warm-up: workspace, kernel attributes
        torch.cuda.set_sync_debug_mode("error")
        try:
            again = _ops.match_pairs_topk(Q, G, T, 8, 1024, 1024, q16, g16)
        finally:
            torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    for x, y in zip(eager, again):
        assert torch.equal(x, y)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        captured = _ops.match_pairs_topk(Q, G, T, 8, 1024, 1024, q16, g16)
    for t in captured:
        t.fill_(0)
    graph.replay()
    torch.cuda.synchronize()
    for x, y in zip(eager, captured):
        assert torch.equal(x, y)
    new = T[[2, 0, 3, 1]].clone()
    new[1, 3] = 0
    T.copy_(new)
    graph.replay()
    torch.cuda.synchronize()
    want = _ops.match_pairs_topk(Q, G, new, 8, 1024, 1024, q16, g16)
    for x, y in zip(want, captured):
        assert torch.equal(x, y)


def test_profile_hooks_and_fallback_count():
    import ctypes as C

    from hardnetnas_b200 import _lib
    from hardnetnas_b200.matching import match_topk
    lib = _lib.load()
    q, g = _inverted_set()
    match_topk(q, g, 8)   # warm-up
    assert lib.hn_match_profile_enable(1) == 0 and lib.hn_match_topk_fallback_enable(1) == 0
    try:
        match_topk(q, g, 8)
        ms, n = (C.c_double * 3)(), (C.c_longlong * 3)()
        assert lib.hn_match_profile_read(ms, n) == 0
        assert list(n) == [1, 1, 1] and all(x > 0 for x in ms)
        rows = C.c_longlong(-1)
        assert lib.hn_match_topk_fallback_read(C.byref(rows)) == 0
        assert 0 < rows.value <= q.size(0)   # the planted clusters need their lists scanned
    finally:
        lib.hn_match_profile_enable(0)
        lib.hn_match_topk_fallback_enable(0)

"""Radius matching on the GPU: exact against a float64 oracle, consistent bit for bit with the top-2 and top-k calls, strict at
the boundary, exact on rows that must scan a whole list, the dense and empty limits, every row type, truncation at a capacity,
pair tables (per pair, padded batches, CUDA graphs) and threshold_matches."""
import math

import pytest
import torch

from oracle import radius_oracle, synth

pytestmark = pytest.mark.gpu

RADII = [0.5, 1.0, 1.3]
SHAPES = [(5, 3), (9, 8), (300, 1001), (257, 130), (1000, 4097), (3, 20000), (511, 640), (700, 128)]


def _rows_of(row_ptr):
    return torch.repeat_interleave(torch.arange(row_ptr.numel() - 1, device=row_ptr.device), row_ptr.diff())


def _d64(q, g, rows, cols):
    dot = (q.double()[rows] * g.double()[cols]).sum(1)
    return torch.sqrt((2 - 2 * dot).clamp(1e-8, 4.0))


def _check_csr(row_ptr, col, dist, nq, ng):
    assert row_ptr.dtype == torch.int64 and row_ptr.numel() == nq + 1 and int(row_ptr[0]) == 0
    assert int(row_ptr[-1]) == col.numel() == dist.numel() and bool((row_ptr.diff() >= 0).all())
    if col.numel():
        assert int(col.min()) >= 0 and int(col.max()) < ng
        rows = _rows_of(row_ptr)
        key = rows * ng + col
        assert bool((key[1:] > key[:-1]).all()), "not in row-major nonzero() order"


def _check_oracle(q, g, r, row_ptr, col, dist):
    """Column sets equal to the float64 oracle's except for columns within 1e-6 of r; distances within 5e-6 of float64 through
    d^2 (as in the top-k test: near d = 0 the sqrt turns the fp32 dot error of ~1e-7 into ~3e-4 of d)."""
    _check_csr(row_ptr, col, dist, q.size(0), g.size(0))
    rp64, c64, _ = radius_oracle.radius_match(q.cpu(), g.cpu(), r, chunk=512)
    got = set(zip(_rows_of(row_ptr).tolist(), col.tolist()))
    want = set(zip(_rows_of(rp64).tolist(), c64.tolist()))
    for i, j in got ^ want:
        d = float(_d64(q, g, torch.tensor([i], device=q.device), torch.tensor([j], device=q.device)))
        assert abs(d - r) <= 1e-6, (i, j, d)
    if col.numel():
        assert float((dist.double() ** 2 - _d64(q, g, _rows_of(row_ptr), col.long()) ** 2).abs().max()) <= 5e-6


@pytest.mark.parametrize("nq,ng", SHAPES)
def test_against_float64_oracle(nq, ng):
    from hardnetnas_b200.matching import match_radius
    q, g, _ = synth.make_match_set(nq, ng, seed=nq + ng)
    qr, gr = synth.unit_vectors(nq, 128, nq), synth.unit_vectors(ng, 128, ng + 1)
    for a, b in ((q, g), (qr, gr)):
        a, b = a.cuda(), b.cuda()
        for r in RADII:
            _check_oracle(a, b, r, *match_radius(a, b, r))


@pytest.mark.parametrize("nq,ng", [(300, 1001), (1000, 4097), (4096, 8192)])
def test_consistent_with_top2_and_topk(nq, ng):
    from hardnetnas_b200.matching import match_radius, match_top2, match_topk
    q, g, _ = synth.make_match_set(nq, ng, seed=5 * nq)
    q, g = q.cuda(), g.cuda()
    d1, _, i1, _ = match_top2(q, g)
    D8, I8 = match_topk(q, g, 8)
    for r in RADII:
        row_ptr, col, dist = match_radius(q, g, r)
        cnt = row_ptr.diff()
        assert torch.equal(cnt > 0, d1 < r)
        rows = _rows_of(row_ptr)
        nonempty = cnt > 0
        row_min = torch.full((nq,), math.inf, device=q.device).scatter_reduce(0, rows, dist, "amin")
        assert torch.equal(row_min[nonempty], d1[nonempty])
        # every entry among the top-k columns carries match_topk's distance; the top-k entries below r are the row's k smallest
        k_in = (D8 < r).sum(1)
        for i in torch.nonzero(nonempty).flatten()[:400].tolist():
            c, d = col[row_ptr[i]:row_ptr[i + 1]], dist[row_ptr[i]:row_ptr[i + 1]]
            for j, dj in zip(I8[i].tolist(), D8[i].tolist()):
                hit = (c == j).nonzero()
                if dj < r:
                    assert hit.numel() == 1 and float(d[hit[0, 0]]) == dj
                else:
                    assert hit.numel() == 0
            order = torch.sort(d, stable=True).indices[: int(k_in[i])]   # c ascends: (distance, index) order
            assert torch.equal(c[order].long(), I8[i, : int(k_in[i])])
        assert int(k_in.sum()) <= int(row_ptr[-1])


def test_strict_boundary():
    from hardnetnas_b200.matching import match_radius, match_top2
    q, g, _ = synth.make_match_set(200, 700, seed=9)
    q, g = q.cuda(), g.cuda()
    d1, _, i1, _ = match_top2(q, g)
    for i in (0, 17, 199):
        r = float(d1[i])
        rp, col, _ = match_radius(q, g, r)
        assert int(i1[i]) not in col[rp[i]:rp[i + 1]].tolist()
        rn = float(torch.nextafter(d1[i:i + 1], torch.tensor([math.inf], device=q.device)))
        rp, col, dist = match_radius(q, g, rn)
        row = col[rp[i]:rp[i + 1]].tolist()
        assert int(i1[i]) in row and float(dist[rp[i] + row.index(int(i1[i]))]) == r


def _inverted_set(dtype=torch.float32, n_clusters=16, per=24, step=5e-6, seed=0):
    """Per query, `per` gallery rows around it in `per` chunks of one segment, exact dots 1 - (0.005 + j * step), the best in the
    last chunks (the construction of test_matching_topk_gpu.py): more than eight chunks of one list reach the threshold of a
    radius just above their distances, so every cluster row has to scan that list."""
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
    return q.to(dtype).cuda(), g.to(dtype).cuda()


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16, torch.float8_e4m3fn])
def test_scan_path_is_exact(dtype):
    from hardnetnas_b200 import _lib
    from hardnetnas_b200.matching import match_radius
    lib = _lib.load()
    q, g = _inverted_set(dtype)
    r = 0.11   # d of the planted fp32 rows: sqrt(2 * (0.005 + j * 5e-6)) <= 0.1012; random columns are near sqrt(2)
    match_radius(q, g, r)   # warm-up
    assert lib.hn_match_topk_fallback_enable(1) == 0
    try:
        row_ptr, col, dist = match_radius(q, g, r)
        import ctypes as C
        n = C.c_longlong(-1)
        assert lib.hn_match_topk_fallback_read(C.byref(n)) == 0
    finally:
        lib.hn_match_topk_fallback_enable(0)
    if dtype == torch.float32:   # rounding to the other types spreads the planted dots
        assert n.value == q.size(0)   # every cluster row scanned its list
        assert bool((row_ptr.diff() >= 24).all())
    _check_oracle(q.float(), g.float(), r, row_ptr, col, dist)


def test_dense_and_empty_limits():
    from hardnetnas_b200.matching import match_radius, match_top2
    q, g, _ = synth.make_match_set(130, 300, seed=2)
    q, g = q.cuda(), g.cuda()
    q[5] = 0
    g[7] = 0
    row_ptr, col, dist = match_radius(q, g, 2.001)
    assert torch.equal(row_ptr, torch.arange(131, device=q.device) * 300)
    assert torch.equal(col.view(130, 300), torch.arange(300, device=q.device).expand(130, 300))
    d1, _, _, _ = match_top2(q, g)
    assert torch.equal(dist.view(130, 300).min(1).values, d1)
    for r in (float(torch.tensor(1e-8).sqrt()), 1e-5, 0.0, -1.0, -math.inf):   # sqrtf(1e-8f): the clamp's floor
        rp, c, d = match_radius(q, g, r)
        assert int(rp[-1]) == 0 and c.numel() == 0 and bool((rp == 0).all())
    # all-zero rows: d = sqrt(2) to every column, so they are entries exactly when sqrt(2) < r
    s2 = float(torch.tensor(2.0).sqrt())
    for r, want in ((s2, 0), (float(torch.nextafter(torch.tensor(s2), torch.tensor(3.0))), 300)):
        rp, c, d = match_radius(q, g, r)
        assert int(rp[6] - rp[5]) == want and bool((d[rp[5]:rp[6]] == s2).all())
        zero_col = [int(i) for i in range(130) if 7 in c[rp[i]:rp[i + 1]].tolist()]
        assert (5 in zero_col) == (want > 0) and len(zero_col) == (130 if want else 0)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16, torch.float8_e4m3fn])
def test_row_types_equal_the_fp32_call(dtype):
    from hardnetnas_b200._ops import match_radius as ops_radius
    from hardnetnas_b200._ops import pack_descriptors
    from hardnetnas_b200.matching import match_radius
    q, g, _ = synth.make_match_set(1000, 4097, seed=17)
    q, g = q.cuda().to(dtype), g.cuda().to(dtype)
    for r in RADII:
        got = match_radius(q, g, r)
        want = match_radius(q.float(), g.float(), r)
        for a, b in zip(got, want):
            assert torch.equal(a, b)
    packed = ops_radius(q, g, 1.0, q16=pack_descriptors(q), g16=pack_descriptors(g))
    for a, b in zip(packed, match_radius(q, g, 1.0)):
        assert torch.equal(a.long() if a.dtype == torch.int32 else a, b)


def test_capacity_truncation_and_sentinel():
    from hardnetnas_b200 import _lib, _ops
    q, g, _ = synth.make_match_set(500, 2000, seed=23)
    q, g = q.cuda(), g.cuda()
    full = _ops.match_radius(q, g, 1.2)
    nnz = int(full[0][-1])
    assert nnz > 100
    lib = _lib.load()
    ws = _ops._workspace(q.device, lib.hn_match_radius_workspace_bytes(500, 2000))
    for cap in (0, 1, 37, nnz - 1, nnz, nnz + 5):
        row_ptr = torch.empty(501, dtype=torch.int64, device=q.device)
        col = torch.full((nnz + 16,), -7, dtype=torch.int32, device=q.device)
        dist = torch.full((nnz + 16,), -7.0, device=q.device)
        st = _ops._stream_ptr()
        assert lib.hn_match_radius_count_typed(_ops._ptr(q), _ops._ptr(g), _lib.HN_F32, None, None, 500, 2000, 1.2, _ops._ptr(row_ptr),
                                               _ops._ptr(ws), ws.numel(), st) == 0
        assert lib.hn_match_radius_fill_typed(_ops._ptr(q), _ops._ptr(g), _lib.HN_F32, 500, 2000, 1.2, _ops._ptr(row_ptr), cap,
                                              _ops._ptr(col) if cap else None, _ops._ptr(dist), _ops._ptr(ws), ws.numel(), st) == 0
        assert torch.equal(row_ptr, full[0])
        w = min(cap, nnz)
        assert torch.equal(col[:w], full[1][:w]) and torch.equal(dist[:w], full[2][:w])
        assert bool((col[w:] == -7).all()) and bool((dist[w:] == -7.0).all())
    # without dist
    col = torch.empty(nnz, dtype=torch.int32, device=q.device)
    assert lib.hn_match_radius_fill_typed(_ops._ptr(q), _ops._ptr(g), _lib.HN_F32, 500, 2000, 1.2, _ops._ptr(full[0]), nnz, _ops._ptr(col),
                                          None, _ops._ptr(ws), ws.numel(), _ops._stream_ptr()) == 0
    assert torch.equal(col, full[1])
    # the Python capacity form: buffers of `capacity` entries, the written prefix equal to the exact-size call
    row_ptr, col, dist = _ops.match_radius(q, g, 1.2, capacity=50)
    assert col.numel() == dist.numel() == 50 and torch.equal(row_ptr, full[0]) and torch.equal(col, full[1][:50])


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


def _per_pair(row_ptr, col, dist, p, max_q):
    a, b = int(row_ptr[p * max_q]), int(row_ptr[(p + 1) * max_q])
    return row_ptr[p * max_q:(p + 1) * max_q + 1] - a, col[a:b], dist[a:b]


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.float8_e4m3fn])
def test_pairs_equal_per_pair_calls(dtype):
    from hardnetnas_b200.matching import match_radius, match_radius_pairs
    Q, G, T = _pairs_case()
    Q, G = Q.to(dtype), G.to(dtype)
    for r in (1.0, 1.3):
        row_ptr, col, dist = match_radius_pairs(Q, G, T.cuda(), r, 1024, 1024)
        assert row_ptr.numel() == T.size(0) * 1024 + 1
        for p, (qs, ql, gs, gl) in enumerate(T.tolist()):
            qs, gs = min(max(qs, 0), Q.size(0)), min(max(gs, 0), G.size(0))
            ql, gl = max(0, min(ql, 1024, Q.size(0) - qs)), max(0, min(gl, 1024, G.size(0) - gs))
            rp, c, d = _per_pair(row_ptr, col, dist, p, 1024)
            assert bool((rp[ql:] == rp[ql]).all())
            if ql == 0 or gl == 0:
                assert c.numel() == 0
                continue
            want = match_radius(Q[qs:qs + ql], G[gs:gs + gl], r)
            assert torch.equal(rp[:ql + 1], want[0]) and torch.equal(c, want[1]) and torch.equal(d, want[2]), p


def test_padded_batch_as_pair_table():
    from hardnetnas_b200.matching import match_radius, match_radius_pairs
    B, N1, N2 = 5, 300, 700
    q = torch.stack([synth.make_match_set(N1, N2, seed=b)[0] for b in range(B)]).cuda()
    g = torch.stack([synth.make_match_set(N1, N2, seed=b)[1] for b in range(B)]).cuda()
    len1, len2 = torch.tensor([300, 0, 17, 299, 128]), torch.tensor([700, 5, 0, 3, 640])
    T = torch.stack([torch.arange(B) * N1, len1, torch.arange(B) * N2, len2], 1).to(torch.int32).cuda()
    row_ptr, col, dist = match_radius_pairs(q.flatten(0, 1), g.flatten(0, 1), T, 1.1, N1, N2)
    for b in range(B):
        a, c = int(len1[b]), int(len2[b])
        rp, cc, dd = _per_pair(row_ptr, col, dist, b, N1)
        if a and c:
            want = match_radius(q[b, :a], g[b, :c], 1.1)
            assert torch.equal(rp[:a + 1], want[0]) and torch.equal(cc, want[1]) and torch.equal(dd, want[2])
            _check_oracle(q[b, :a], g[b, :c], 1.1, *want)
        else:
            assert cc.numel() == 0


def test_pairs_graph_capture_follows_table_edits():
    from hardnetnas_b200 import _ops
    Q, G, T = _pairs_case(seed=60)
    T = T[:4].contiguous().cuda()
    q16, g16 = _ops.pack_descriptors(Q), _ops.pack_descriptors(G)
    cap = 1 << 20
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        eager = _ops.match_pairs_radius(Q, G, T, 1.2, 1024, 1024, cap, q16, g16)   # warm-up: workspace, kernel attributes
        torch.cuda.set_sync_debug_mode("error")
        try:
            again = _ops.match_pairs_radius(Q, G, T, 1.2, 1024, 1024, cap, q16, g16)
        finally:
            torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    nnz = int(eager[0][-1])
    assert 0 < nnz < cap
    assert torch.equal(eager[0], again[0]) and torch.equal(eager[1][:nnz], again[1][:nnz])
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        captured = _ops.match_pairs_radius(Q, G, T, 1.2, 1024, 1024, cap, q16, g16)
    for t in captured:
        t.fill_(0)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(eager[0], captured[0])
    assert torch.equal(eager[1][:nnz], captured[1][:nnz]) and torch.equal(eager[2][:nnz], captured[2][:nnz])
    new = T[[2, 0, 3, 1]].clone()
    new[1, 3] = 0
    T.copy_(new)
    graph.replay()
    torch.cuda.synchronize()
    want = _ops.match_pairs_radius(Q, G, new, 1.2, 1024, 1024, None, q16, g16)
    n = int(want[0][-1])
    assert torch.equal(want[0], captured[0]) and torch.equal(want[1], captured[1][:n]) and torch.equal(want[2], captured[2][:n])


def test_threshold_matches_is_nonzero_order():
    from hardnetnas_b200.matching import threshold_matches
    q, g, _ = synth.make_match_set(700, 1500, seed=31)
    q, g = q.cuda(), g.cuda()
    pairs, dist = threshold_matches(q, g, 1.0)
    rp64, c64, _ = radius_oracle.radius_match(q.cpu(), g.cpu(), 1.0)
    assert pairs.dtype == torch.int64 and pairs.size(0) > 0 and dist.numel() == pairs.size(0)
    assert torch.equal(pairs.cpu(), torch.stack([_rows_of(rp64), c64], 1))
    assert float((dist.double() ** 2 - _d64(q, g, pairs[:, 0], pairs[:, 1]) ** 2).abs().max()) <= 5e-6


def test_profile_hooks():
    import ctypes as C

    from hardnetnas_b200 import _lib
    from hardnetnas_b200.matching import match_radius
    lib = _lib.load()
    q, g, _ = synth.make_match_set(1000, 3000, seed=4)
    q, g = q.cuda(), g.cuda()
    match_radius(q, g, 1.0)
    assert lib.hn_match_profile_enable(1) == 0
    try:
        match_radius(q, g, 1.0)
        ms, n = (C.c_double * 3)(), (C.c_longlong * 3)()
        assert lib.hn_match_profile_read(ms, n) == 0
        assert list(n) == [1, 1, 2] and all(x > 0 for x in ms)
    finally:
        lib.hn_match_profile_enable(0)

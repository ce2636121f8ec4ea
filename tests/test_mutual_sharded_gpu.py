"""Sharded mutual nearest neighbours on ONE GPU: R ranks of distributed.mutual_nn_ratio_sharded simulated in one process
(hn_match_ex with block maxima, hn_mutual_claims at each rank's global row offset, the MIN reduction of the claims,
hn_mutual_verify, the MAX reduction of the beaten flags), compared with the full-set kernels and a float64 oracle. Also
hn_match's gallery offset, and the Python wrappers' checks of the tensors these calls read and write through bare pointers."""
import pytest
import torch

from hardnetnas_b200 import _lib, _ops
from hardnetnas_b200.distributed import shard_range
from oracle import mutual_oracle, synth
from oracle.losses_oracle import distance_matrix_vector_fdl

pytestmark = pytest.mark.gpu

# the two "unclaimed" fills: what mutual_nn_ratio_sharded writes, and the 0x7f bytes hn_match_mutual memsets
INITS = {"int64_max": torch.iinfo(torch.int64).max, "bytes_7f": 0x7F7F7F7F7F7F7F7F}
NEAR_TIE = 1e-6


@pytest.fixture
def force_kernel():
    """hn_match_force_kernel(mode): -1 by size, 0 single-CTA GEMM, 1 CTA-pair GEMM; restored afterwards."""
    lib = _lib.load()
    yield lambda mode: _lib.check(lib.hn_match_force_kernel(int(mode)), "hn_match_force_kernel")
    lib.hn_match_force_kernel(-1)


def sharded_mutual(q, g, bounds, base, init):
    """distributed.mutual_nn_ratio_sharded step by step, one rank per (lo, hi) of `bounds` holding query rows q[lo:hi] with
    global ids base + lo ...: match_top2 with the block maxima, mutual_claims into a claim vector filled with `init`; then
    the all_reduce(MIN) of the claims as an amin over the ranks' vectors, mutual_verify per rank against the reduced claims,
    the all_reduce(MAX) of the beaten flags as an amax, and the mutual mask of every rank's rows."""
    ng, dev = g.size(0), q.device
    ranks = []
    for lo, hi in bounds:
        bm = torch.empty(_ops.block_max_elems(hi - lo, ng), dtype=torch.float32, device=dev)
        d1, d2, i1, i2 = _ops.match_top2(q[lo:hi], g, block_max=bm)
        claim = torch.full((ng,), init, dtype=torch.int64, device=dev)
        rbmin = _ops.mutual_claims(i1, d1, d2, base + lo, claim)
        ranks.append(dict(top2=(d1, d2, i1, i2), bm=bm, claim=claim, rbmin=rbmin))
    claim = torch.stack([r["claim"] for r in ranks]).amin(0)
    beaten = []
    for (lo, hi), r in zip(bounds, ranks):
        b = torch.zeros(ng, dtype=torch.uint8, device=dev)
        _ops.mutual_verify(q[lo:hi], base + lo, g, claim, r["bm"], r["rbmin"], b)
        beaten.append(b)
    beaten = torch.stack(beaten).amax(0)
    fwd = torch.cat([r["top2"][2] for r in ranks]).long()
    i = torch.arange(q.size(0), device=dev) + base
    mutual = ((claim[fwd] & 0xFFFFFFFF) == i) & (beaten[fwd] == 0)
    return ranks, claim, mutual


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _near_tie_gap(q64, g64, i, j_kernel, j_oracle):
    """The float64 gap between the two distances whose order decides row i's mutual flag: its two candidate columns when
    the row side differs, else d(i, j) against the nearest other query of column j."""
    if j_kernel != j_oracle:
        d = distance_matrix_vector_fdl(q64[i:i + 1], g64[[j_kernel, j_oracle]])[0]
        return (d[0] - d[1]).abs().item()
    col = distance_matrix_vector_fdl(q64, g64[j_oracle:j_oracle + 1])[:, 0]
    di = col[i].item()
    col[i] = float("inf")
    return abs(di - col.min().item())


def check_sharded(q, g, bounds, base, exact_oracle):
    """Every check of one shard layout, for both claim fills; returns the mutual mask and the number of rows on which it
    differs from the float64 oracle at a near tie (always 0 with exact_oracle)."""
    from hardnetnas_b200.matching import mutual_nn_ratio, mutual_nn_ratio_two_pass
    nq, ng = q.size(0), g.size(0)
    assert bounds[0][0] == 0 and bounds[-1][1] == nq and all(a[1] == b[0] for a, b in zip(bounds, bounds[1:]))
    full = _ops.match_top2(q, g)
    _, want_mutual, *_ = mutual_nn_ratio(q, g, return_pairs=False)
    _, two_pass, *_ = mutual_nn_ratio_two_pass(q, g, return_pairs=False)
    fwd_o, _, _, mutual_o = mutual_oracle.mutual_match(q, g)
    rows = torch.arange(nq, device=q.device)
    key = (full[0].view(torch.int32).long() << 32) | (rows + base)
    result = None
    for name, init in INITS.items():
        ranks, claim, mutual = sharded_mutual(q, g, bounds, base, init)
        for (lo, hi), r in zip(bounds, ranks):
            for got, want in zip(r["top2"], full):
                assert torch.equal(_bits(got), _bits(want[lo:hi])), (name, lo, hi)
            d2 = torch.cat([full[1][lo:hi], full[1].new_full(((lo - hi) % 32,), float("inf"))])
            assert torch.equal(_bits(r["rbmin"]), _bits(d2.view(-1, 32).amin(1))), (name, lo, hi)
        want_claim = torch.full((ng,), init, dtype=torch.int64, device=q.device).scatter_reduce(0, full[2].long(), key, "amin")
        assert torch.equal(claim, want_claim), name
        assert torch.equal(mutual, want_mutual) and torch.equal(mutual, two_pass), name
        result = mutual
    diff = (result != mutual_o).nonzero().flatten().tolist()
    if exact_oracle:
        assert not diff, f"mutual differs from the float64 oracle on rows {diff[:20]}"
        return result, 0
    q64, g64 = q.double(), g.double()
    fwd = full[2].long()
    for i in diff:
        gap = _near_tie_gap(q64, g64, i, int(fwd[i]), int(fwd_o[i]))
        assert gap <= NEAR_TIE, f"row {i}: mutual {bool(result[i])}, oracle {bool(mutual_o[i])}, float64 gap {gap:.3e}"
    return result, len(diff)


def _bounds(nq, layout):
    """Shard layout: ("equal", R), ("range", R) = distributed.shard_range, or an explicit list of shard sizes."""
    if isinstance(layout, tuple):
        kind, r = layout
        if kind == "equal":
            assert nq % r == 0
            return [(k * nq // r, (k + 1) * nq // r) for k in range(r)]
        return [shard_range(nq, k, r) for k in range(r)]
    ends = torch.tensor(layout).cumsum(0).tolist()
    assert ends[-1] == nq
    return list(zip([0] + ends[:-1], ends))


def _random_set(kind, nq, ng, seed):
    if kind == "match":
        q, g, _ = synth.make_match_set(nq, ng, seed=seed)
        return q, g
    return synth.unit_vectors(nq, 128, seed), synth.unit_vectors(ng, 128, seed + 1)   # unstructured: many weak claims


RANDOM_CASES = [
    # (set, Nq, Ng, layout, base of the global row ids)
    ("match", 1000, 1500, ("equal", 1), 0),
    ("match", 2048, 3000, ("equal", 2), 7),
    ("unit", 3001, 4000, ("range", 3), (1 << 31) - 1500),
    ("match", 5003, 6000, ("range", 5), 0),
    ("match", 8297, 5000, [1, 31, 32, 33, 8200], 0),
    ("unit", 8297, 5000, [8200, 33, 32, 31, 1], 12345),
    ("match", 16384, 24576, ("equal", 8), 0),
    ("unit", 16003, 24000, ("range", 8), (1 << 32) - 1 - 16003),
]


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("kind,nq,ng,layout,base", RANDOM_CASES)
def test_sharded_random_sets(kind, nq, ng, layout, base, mode, force_kernel):
    force_kernel(mode)
    q, g = _random_set(kind, nq, ng, seed=nq + ng)
    _, near = check_sharded(q.cuda(), g.cuda(), _bounds(nq, layout), base, exact_oracle=False)
    print(f"\n[{kind} {nq}x{ng} {layout} base={base} mode={mode}] rows differing from the float64 oracle at a near tie: {near}")


# ---- planted cross-shard cases ------------------------------------------------------------------------------------------
# Planted rows live on dimensions 0..11 of the gallery's leading basis rows; the random rows have zeros there, so every dot
# product of a planted row is a sum of exact products x * 1 and x * 0, and ties are bit for bit in every path (GEMM operands,
# re-rank, verification, float64). X = fl(1/sqrt(2)).
X = float(torch.tensor(0.5 ** 0.5, dtype=torch.float32))
NQ_PLANT, NG_RANDOM = 640, 1000
BASIS = 14        # gallery columns 0..13: e_127, e_0 .. e_11, e_3 again
P = dict(zero=(5, 140, 300), dup_lo=99, dup_hi=100, force=101, c_b=20, k_b=400, k_c=270, c_c=500, c_d=180, k_d=600)
PLANT_LAYOUT = [100, 160, 200, 180]   # ranks [0,100) [100,260) [260,460) [460,640): the duplicates straddle the first boundary


def _col(p):
    return 1 + p   # gallery column of e_p


def planted_set(seed=3):
    q, g, _ = synth.make_match_set(NQ_PLANT, NG_RANDOM, seed=seed)
    g[:, :12] = 0.0
    g[:, 127] = 0.0
    g = torch.nn.functional.normalize(g, dim=1)
    q[:, :12] = 0.0
    q[:, 127] = 0.0
    q = torch.nn.functional.normalize(q, dim=1) * (0.99 ** 0.5)
    q[:, 127] = -0.1     # random queries are sqrt(2.2) from column 0, planted and zero rows exactly sqrt(2)
    basis = torch.zeros(BASIS, 128)
    basis[0, 127] = 1.0
    basis[torch.arange(1, 13), torch.arange(12)] = 1.0
    basis[13, 3] = 1.0
    g = torch.cat([basis, g])

    def row(**comp):
        r = torch.zeros(128)
        for p, v in comp.items():
            r[int(p[1:])] = v
        return r

    for z in P["zero"]:
        q[z] = 0.0       # all distances exactly sqrt(2): nearest column 0; the lowest such row wins it
    # identical queries on two ranks (nearest column 1, tied with column 2): the lower global row holds the claim; the row
    # after the higher one has d1 = d2 = 1e-4 (two copies of e_3), so verification must evaluate the higher one's block
    q[P["dup_lo"]] = q[P["dup_hi"]] = row(e0=X, e1=X)
    q[P["force"]] = row(e3=1.0)
    # beaten from another rank: k_b's nearest is column e_2, and it is nearer to column e_4 than c_b, who claims e_4
    q[P["k_b"]] = row(e2=0.8, e4=0.6)
    q[P["c_b"]] = row(e4=0.55)
    q[P["c_b"], 12:127] = (1 - 0.55 ** 2) ** 0.5 / 115 ** 0.5
    # exact-tie beat: k_c (lower id) is exactly as near to c_c's column e_6 as c_c, its own nearest is e_5 at the same
    # distance; k_c's 32-row block has no smaller d2, so its minimum d2 EQUALS the claim distance
    q[P["k_c"]] = row(e5=X, e6=X)
    q[P["c_c"]] = row(e6=X, e7=X)
    # the same tie with the higher id on the other side: c_d keeps column e_9
    q[P["c_d"]] = row(e9=X, e10=X)
    q[P["k_d"]] = row(e8=X, e9=X)
    return q, g


PLANT_BASES = [0, (1 << 31) - PLANT_LAYOUT[0], (1 << 32) - 1 - NQ_PLANT]   # boundary at global id 2^31; last id 2^32 - 2


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("base", PLANT_BASES)
@pytest.mark.parametrize("layout", ["ranks4", "ranks1"])
def test_sharded_planted(layout, base, mode, force_kernel):
    force_kernel(mode)
    q, g = planted_set()
    bounds = _bounds(NQ_PLANT, PLANT_LAYOUT if layout == "ranks4" else ("equal", 1))
    mutual, _ = check_sharded(q.cuda(), g.cuda(), bounds, base, exact_oracle=True)
    fwd = _ops.match_top2(q.cuda(), g.cuda())[2].cpu()
    m = mutual.cpu()
    z = list(P["zero"])
    assert fwd[z].tolist() == [0] * len(z) and m[z[0]] and not m[z[1:]].any()
    assert fwd[P["dup_lo"]] == fwd[P["dup_hi"]] == _col(0) and m[P["dup_lo"]] and not m[P["dup_hi"]]
    assert fwd[P["force"]] == _col(3) and m[P["force"]]
    assert fwd[P["c_b"]] == _col(4) and fwd[P["k_b"]] == _col(2) and not m[P["c_b"]] and m[P["k_b"]]
    assert fwd[P["c_c"]] == _col(6) and fwd[P["k_c"]] == _col(5) and not m[P["c_c"]] and m[P["k_c"]]
    assert fwd[P["c_d"]] == _col(9) and fwd[P["k_d"]] == _col(8) and m[P["c_d"]] and m[P["k_d"]]
    if layout == "ranks4" and base == PLANT_BASES[1]:
        assert base + P["dup_lo"] == (1 << 31) - 1 and base + P["dup_hi"] == 1 << 31


# ---- hn_match's gallery offset -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("ng,g_offset", [(3000, 12345), (1, 77), (1000, (1 << 31) - 1 - 1000), (1, (1 << 31) - 2)])
def test_g_offset_shifts_indices_only(ng, g_offset, mode, force_kernel):
    force_kernel(mode)
    q, g, _ = synth.make_match_set(2000, ng, seed=ng + 4)
    q, g = q.cuda(), g.cuda()
    d1, d2, i1, i2 = _ops.match_top2(q, g)
    e1, e2, j1, j2 = _ops.match_top2(q, g, g_offset=g_offset)
    assert torch.equal(_bits(e1), _bits(d1)) and torch.equal(_bits(e2), _bits(d2))
    assert torch.equal(j1.long(), i1.long() + g_offset)
    assert torch.equal(j2.long(), torch.where(i2 < 0, -1, i2.long() + g_offset))
    if ng == 1:
        assert torch.all(j2 == -1) and torch.all(j1 == g_offset)
    assert int(j1.max()) < 1 << 31


# ---- the wrappers check every tensor before any launch -------------------------------------------------------------------
def test_wrappers_reject_bad_tensors_before_launch():
    lib = _lib.load()
    q, g, _ = synth.make_match_set(100, 300, seed=1)
    q, g = q.cuda(), g.cuda()
    nq, ng = 100, 300
    bm = torch.empty(_ops.block_max_elems(nq, ng), dtype=torch.float32, device="cuda")
    d1, d2, i1, _ = _ops.match_top2(q, g, block_max=bm)
    claim = torch.full((ng,), INITS["int64_max"], dtype=torch.int64, device="cuda")
    rbmin = _ops.mutual_claims(i1, d1, d2, 0, claim)
    beaten = torch.full((ng,), 7, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    claim0 = claim.clone()
    launches = lib.hn_launch_count()

    def rejected(call):
        with pytest.raises((ValueError, _lib.HardnetB200Error)):
            call()

    verify = dict(q=q, q_offset=0, g=g, claim=claim, block_max=bm, rb_min_d2=rbmin, beaten=beaten)
    bad_verify = [
        dict(claim=claim[:-1]), dict(claim=claim.int()), dict(claim=claim.cpu()), dict(beaten=beaten[:-1]),
        dict(beaten=beaten.bool()), dict(beaten=torch.full((2 * ng,), 7, dtype=torch.uint8, device="cuda")[::2]),
        dict(block_max=bm[:-1]), dict(block_max=bm.half()), dict(rb_min_d2=rbmin[:-1]), dict(rb_min_d2=rbmin.double()),
        dict(q=q.half()), dict(g=g.half()), dict(g=g.cpu()), dict(q=q[:, :64]),
    ]
    for bad in bad_verify:
        rejected(lambda: _ops.mutual_verify(**{**verify, **bad}))
    claims = dict(i1=i1, d1=d1, d2=d2, q_offset=0, claim=claim)
    for bad in [dict(i1=i1.long()), dict(d1=d1[:-1]), dict(d2=d2.half()), dict(d2=d2.cpu()), dict(claim=claim.int()),
                dict(claim=torch.full((2 * ng,), 0, dtype=torch.int64, device="cuda")[::2]), dict(i1=i1.cpu())]:
        rejected(lambda: _ops.mutual_claims(**{**claims, **bad}))
    for bad in [bm[:-1], bm.double(), bm.cpu(), torch.empty(2 * bm.numel(), device="cuda")[::2]]:
        rejected(lambda: _ops.match_top2(q, g, block_max=bad))
    torch.cuda.synchronize()
    assert lib.hn_launch_count() == launches
    assert torch.all(beaten == 7) and torch.equal(claim, claim0)
    # the same calls with valid tensors go through
    _ops.mutual_verify(**verify)
    assert lib.hn_launch_count() > launches

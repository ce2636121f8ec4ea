"""Radius matching (hn_match_radius_*, hn_match_pairs_radius_*) without a GPU: argument validation before any device work, the
workspace sizes, the Python wrappers' checks and the float64 oracle."""
import ctypes as C
import math

import pytest
import torch

from hardnetnas_b200 import _lib

HN_ERR_INVALID = -1
FAKE = C.c_void_p(1 << 20)   # never dereferenced: every case below fails validation first
NULL = C.c_void_p(0)
ALIGN2 = C.c_void_p((1 << 20) + 2)
ALIGN4 = C.c_void_p((1 << 20) + 4)
COUNT = ["hn_match_radius_count_typed", "hn_match_pairs_radius_count_typed"]
FILL = ["hn_match_radius_fill_typed", "hn_match_pairs_radius_fill_typed"]
FNS = COUNT + FILL


@pytest.fixture(scope="module")
def lib():
    if not _lib.LIB_PATH.exists():
        from hardnetnas_b200 import build
        build.build()
    return _lib.load()


def _call(lib, fn, radius=1.0, dt=_lib.HN_F32, q=FAKE, g=FAKE, row_ptr=FAKE, capacity=16, col=FAKE, dist=FAKE, ws=FAKE,
          ws_bytes=1 << 40):
    """One call on 100 x 120 rows (pair form: 4 pairs over sets of 1000 rows)."""
    r = C.c_float(radius)
    if fn == "hn_match_radius_count_typed":
        return lib.hn_match_radius_count_typed(q, g, dt, NULL, NULL, 100, 120, r, row_ptr, ws, ws_bytes, NULL)
    if fn == "hn_match_radius_fill_typed":
        return lib.hn_match_radius_fill_typed(q, g, dt, 100, 120, r, row_ptr, capacity, col, dist, ws, ws_bytes, NULL)
    if fn == "hn_match_pairs_radius_count_typed":
        return lib.hn_match_pairs_radius_count_typed(q, FAKE, 1000, g, FAKE, 1000, dt, FAKE, 4, 100, 120, r, row_ptr, ws, ws_bytes, NULL)
    return lib.hn_match_pairs_radius_fill_typed(q, FAKE, 1000, g, FAKE, 1000, dt, FAKE, 4, 100, 120, r, row_ptr, capacity, col, dist,
                                                ws, ws_bytes, NULL)


def _rejected(lib, fn, status, what):
    assert status == HN_ERR_INVALID
    msg = lib.hn_last_error().decode()
    assert msg.startswith(fn + ":") and what in msg, msg


@pytest.mark.parametrize("fn", FNS)
@pytest.mark.parametrize("arg", ["q", "g", "row_ptr", "ws"])
def test_null_arguments(lib, fn, arg):
    _rejected(lib, fn, _call(lib, fn, **{arg: NULL}), "NULL argument")


@pytest.mark.parametrize("fn", FNS)
def test_nan_radius(lib, fn):
    _rejected(lib, fn, _call(lib, fn, radius=math.nan), "radius is NaN")


@pytest.mark.parametrize("fn", FILL)
def test_capacity_and_col(lib, fn):
    _rejected(lib, fn, _call(lib, fn, capacity=-1), "capacity must be >= 0 (got -1)")
    _rejected(lib, fn, _call(lib, fn, col=NULL), "col is NULL with capacity 16 > 0")
    _rejected(lib, fn, _call(lib, fn, col=ALIGN2), "col and dist must be 4-byte aligned")
    _rejected(lib, fn, _call(lib, fn, dist=ALIGN2), "col and dist must be 4-byte aligned")


@pytest.mark.parametrize("fn", FNS)
def test_misaligned_row_ptr(lib, fn):
    _rejected(lib, fn, _call(lib, fn, row_ptr=ALIGN4), "row_ptr must be 8-byte aligned")


@pytest.mark.parametrize("fn", FNS)
def test_unknown_dtype(lib, fn):
    _rejected(lib, fn, _call(lib, fn, dt=4), "desc_dtype must be HN_F32, HN_F16 or HN_BF16, or HN_F8E4M3 (got 4)")
    _rejected(lib, fn, _call(lib, fn, dt=_lib.HN_U8), "desc_dtype must be")


@pytest.mark.parametrize("fn", FNS)
@pytest.mark.parametrize("dt,what", [(_lib.HN_F16, "8-byte aligned"), (_lib.HN_BF16, "8-byte aligned"), (_lib.HN_F8E4M3, "4-byte aligned")])
def test_misaligned_rows(lib, fn, dt, what):
    _rejected(lib, fn, _call(lib, fn, dt=dt, g=ALIGN2), what)


@pytest.mark.parametrize("fn", FNS)
def test_workspace_too_small_and_misaligned(lib, fn):
    pairs = "pairs" in fn
    need = lib.hn_match_pairs_radius_workspace_bytes(4, 100, 120) if pairs else lib.hn_match_radius_workspace_bytes(100, 120)
    _rejected(lib, fn, _call(lib, fn, ws_bytes=need - 1), "workspace too small")
    _rejected(lib, fn, _call(lib, fn, ws=C.c_void_p((1 << 20) + 16)), "256-byte aligned")


def _tiles(rows):
    return 256 * ((8 * -(-rows // 8192) + 255) // 256)   # the scan's tile sums, 8 bytes per 8192 rows, 256-byte aligned


@pytest.mark.parametrize("nq,ng", [(1, 1), (100, 120), (8192, 300), (8193, 4097), (65536, 65536), (1 << 22, 1000)])
def test_workspace_is_the_topk_layout_plus_the_scan(lib, nq, ng):
    got = lib.hn_match_radius_workspace_bytes(nq, ng)
    assert got == lib.hn_match_topk_workspace_bytes(nq, ng) + _tiles(nq) and got % 256 == 0


@pytest.mark.parametrize("b,mq,mg", [(1, 1, 1), (4, 100, 120), (57, 1500, 2000), (300, 4096, 4096)])
def test_pairs_workspace_is_the_topk_layout_plus_the_scan(lib, b, mq, mg):
    got = lib.hn_match_pairs_radius_workspace_bytes(b, mq, mg)
    assert got == lib.hn_match_pairs_topk_workspace_bytes(b, mq, mg) + _tiles(b * mq) and got % 256 == 0


def test_workspace_of_negative_sizes(lib):
    assert lib.hn_match_radius_workspace_bytes(-1, 5) == 0 and lib.hn_match_pairs_radius_workspace_bytes(1, -1, 5) == 0


@pytest.mark.parametrize("radius", [float("nan"), "1.0", None, True, torch.tensor(1.0)])
def test_python_wrappers_reject_radius(radius):
    from hardnetnas_b200 import matching
    x = torch.zeros(4, 128)
    with pytest.raises(ValueError, match="radius must be a real number"):
        matching.match_radius(x, x, radius)
    with pytest.raises(ValueError, match="radius must be a real number"):
        matching.match_radius_pairs(x, x, torch.zeros(1, 4, dtype=torch.int32), radius, 4, 4)


@pytest.mark.parametrize("capacity", [-1, 2.0, True, "3"])
def test_python_wrappers_reject_capacity(capacity):
    from hardnetnas_b200 import matching
    x = torch.zeros(4, 128)
    with pytest.raises(ValueError, match="capacity must be None or an integer >= 0"):
        matching.match_radius(x, x, 1.0, capacity=capacity)
    with pytest.raises(ValueError, match="capacity must be None or an integer >= 0"):
        matching.match_radius_pairs(x, x, torch.zeros(1, 4, dtype=torch.int32), 1.0, 4, 4, capacity=capacity)


def test_python_wrappers_reject_cpu_tensors():
    from hardnetnas_b200 import matching
    x = torch.nn.functional.normalize(torch.randn(4, 128), dim=1)
    with pytest.raises(_lib.HardnetB200Error, match="CUDA tensors only"):
        matching.match_radius(x, x, 1.0)
    with pytest.raises(_lib.HardnetB200Error, match="CUDA tensors only"):
        matching.threshold_matches(x, x, 1.0)
    with pytest.raises(_lib.HardnetB200Error, match="CUDA tensors only"):
        matching.match_radius_pairs(x, x, torch.tensor([[0, 4, 0, 4]], dtype=torch.int32), 1.0, 4, 4)


@pytest.mark.parametrize("r", [0.5, 1.0, 1.3])
def test_radius_oracle_agrees_with_knn_and_ratio_oracles(r):
    """Each row's entries are exactly its knn_oracle columns below r (the whole sorted row), and the row minimum is ratio_match's."""
    from oracle import knn_oracle, losses_oracle, radius_oracle, synth
    q, g, _ = synth.make_match_set(200, 300, seed=7)
    row_ptr, col, dist = radius_oracle.radius_match(q, g, r, chunk=64)
    D, I = knn_oracle.knn_match(q, g, g.size(0), chunk=64)
    _, ia, da, _ = losses_oracle.ratio_match(q.double(), g.double(), chunk=64)
    assert row_ptr[0] == 0 and row_ptr[-1] == col.numel() == dist.numel() and dist.dtype == torch.float64
    for i in range(q.size(0)):
        c, d = col[row_ptr[i]:row_ptr[i + 1]], dist[row_ptr[i]:row_ptr[i + 1]]
        want = I[i][D[i] < r]
        assert torch.equal(c, want.sort().values)
        assert bool((d < r).all())
        if c.numel():
            assert d.min() == da[i] and ia[i] in c.tolist()
        else:
            assert da[i] >= r


def test_radius_oracle_is_nonzero_order():
    from oracle import radius_oracle, synth
    q, g, _ = synth.make_match_set(70, 90, seed=3)
    row_ptr, col, _ = radius_oracle.radius_match(q, g, 1.2, chunk=16)
    D = torch.sqrt((2 - 2 * q.double() @ g.double().t()).clamp(1e-8, 4.0))
    nz = D.lt(1.2).nonzero()
    rows = torch.repeat_interleave(torch.arange(70), row_ptr.diff())
    assert torch.equal(torch.stack([rows, col], 1), nz)

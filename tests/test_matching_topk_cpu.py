"""k-nearest-neighbour matching (hn_match_topk_typed, hn_match_pairs_topk_typed) without a GPU: argument validation before any
device work, the Python wrappers' checks, the float64 oracle, and the workspace sizes of the pre-existing matching calls."""
import ctypes as C

import pytest
import torch

from hardnetnas_b200 import _lib

HN_ERR_INVALID = -1
FAKE = C.c_void_p(1 << 20)   # never dereferenced: every case below fails validation first
NULL = C.c_void_p(0)
ALIGN2 = C.c_void_p((1 << 20) + 2)
FNS = ["hn_match_topk_typed", "hn_match_pairs_topk_typed"]


@pytest.fixture(scope="module")
def lib():
    if not _lib.LIB_PATH.exists():
        from hardnetnas_b200 import build
        build.build()
    return _lib.load()


def _call(lib, fn, k=4, dt=_lib.HN_F32, q=FAKE, g=FAKE, out=FAKE, ws=FAKE, ws_bytes=1 << 40):
    """One call on 100 x 120 rows (pair form: 4 pairs over sets of 1000 rows)."""
    if fn == "hn_match_topk_typed":
        return lib.hn_match_topk_typed(q, g, dt, NULL, NULL, 100, 120, k, out, FAKE, ws, ws_bytes, NULL)
    return lib.hn_match_pairs_topk_typed(q, FAKE, 1000, g, FAKE, 1000, dt, FAKE, 4, 100, 120, k, out, FAKE, ws, ws_bytes, NULL)


def _rejected(lib, fn, status, what):
    assert status == HN_ERR_INVALID
    msg = lib.hn_last_error().decode()
    assert msg.startswith(fn + ":") and what in msg, msg


@pytest.mark.parametrize("fn", FNS)
@pytest.mark.parametrize("k", [0, 9, -1])
def test_k_out_of_range(lib, fn, k):
    _rejected(lib, fn, _call(lib, fn, k=k), f"k must be in [1, 8] (got {k})")


@pytest.mark.parametrize("fn", FNS)
@pytest.mark.parametrize("arg", ["q", "g", "out", "ws"])
def test_null_arguments(lib, fn, arg):
    _rejected(lib, fn, _call(lib, fn, **{arg: NULL}), "NULL argument")


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
    need = lib.hn_match_topk_workspace_bytes(100, 120) if fn == FNS[0] else lib.hn_match_pairs_topk_workspace_bytes(4, 100, 120)
    assert need > 0
    _rejected(lib, fn, _call(lib, fn, ws_bytes=need - 1), "workspace too small")
    _rejected(lib, fn, _call(lib, fn, ws=C.c_void_p((1 << 20) + 16)), "256-byte aligned")


def test_topk_workspace_covers_the_lists():
    lib = _lib.load()
    # 16 segments x 8 chunks of (id, maximum) per row and 16 dropped maxima, plus the packed operands
    assert lib.hn_match_topk_workspace_bytes(65536, 65536) >= 65536 * (2 * 16 * 8 * 4 + 16 * 4 + 2 * 256)
    assert lib.hn_match_pairs_topk_workspace_bytes(10, 1000, 1000) >= 10 * 1000 * (2 * 8 * 8 * 4 + 8 * 4)
    assert lib.hn_match_topk_workspace_bytes(-1, 5) == 0 and lib.hn_match_pairs_topk_workspace_bytes(1, -1, 5) == 0


# Values of the parent commit: the top-k lists reuse the layout functions, which must size the existing calls as before.
OLD_SINGLE = [(1, 1), (100, 120), (1000, 4097), (65536, 65536)]
OLD_DIST = [3072, 172800, 3993344, 102498560]
OLD_MUTUAL = [4352, 174848, 4097024, 170205696]
OLD_BATCHED = [(1, 1, 1), (4, 100, 120), (57, 1500, 2000), (300, 4096, 4096)]
OLD_BATCHED_BYTES = {0: [1024, 238080, 94848000, 1258291200], 1: [2048, 243712, 98564096, 1348147200]}
OLD_PAIRS_BYTES = {0: [512, 12800, 43776000, 629145600], 1: [1536, 18432, 47492096, 719001600]}


def test_existing_workspace_sizes_unchanged(lib):
    assert [lib.hn_dist_workspace_bytes(a, b, 0) for a, b in OLD_SINGLE] == OLD_DIST
    assert [lib.hn_mutual_workspace_bytes(a, b) for a, b in OLD_SINGLE] == OLD_MUTUAL
    for m in (0, 1):
        assert [lib.hn_match_batched_workspace_bytes(*s, m) for s in OLD_BATCHED] == OLD_BATCHED_BYTES[m]
        assert [lib.hn_match_pairs_workspace_bytes(*s, m) for s in OLD_BATCHED] == OLD_PAIRS_BYTES[m]


def test_fallback_count_needs_enabling(lib):
    n = C.c_longlong(-1)
    _rejected(lib, "hn_match_topk_fallback_read", lib.hn_match_topk_fallback_read(C.byref(n)), "not enabled")
    assert lib.hn_match_topk_fallback_enable(0) == 0


@pytest.mark.parametrize("k", [0, 9, 2.0, True, None])
def test_python_wrappers_reject_k(k):
    from hardnetnas_b200 import matching
    x = torch.zeros(4, 128)
    with pytest.raises(ValueError, match="k must be an integer in \\[1, 8\\]"):
        matching.match_topk(x, x, k)
    with pytest.raises(ValueError, match="k must be an integer in \\[1, 8\\]"):
        matching.match_topk_pairs(x, x, torch.zeros(1, 4, dtype=torch.int32), k, 4, 4)


def test_python_wrappers_reject_cpu_tensors():
    from hardnetnas_b200 import matching
    x = torch.nn.functional.normalize(torch.randn(4, 128), dim=1)
    with pytest.raises(_lib.HardnetB200Error, match="CUDA tensors only"):
        matching.match_topk(x, x, 2)
    with pytest.raises(_lib.HardnetB200Error, match="CUDA tensors only"):
        matching.match_topk_pairs(x, x, torch.tensor([[0, 4, 0, 4]], dtype=torch.int32), 2, 4, 4)


def test_knn_oracle_agrees_with_ratio_match_for_k2():
    from oracle import knn_oracle, losses_oracle, synth
    q, g, _ = synth.make_match_set(300, 700, seed=5)
    D, I = knn_oracle.knn_match(q, g, 2, chunk=128)
    _, ia, da, db = losses_oracle.ratio_match(q.double(), g.double(), chunk=128)
    assert D.dtype == torch.float64 and I.shape == (300, 2)
    assert torch.equal(I[:, 0], ia) and torch.equal(D[:, 0], da) and torch.equal(D[:, 1], db)


def test_knn_oracle_order_and_padding():
    from oracle import knn_oracle, synth
    g = synth.unit_vectors(5, 128, 3)
    q = torch.cat([g[2:3], g[2:3]])
    g = torch.cat([g, g[2:3]])   # column 5 ties column 2: the lower index comes first
    D, I = knn_oracle.knn_match(q, g, 8)
    assert I[0, :2].tolist() == [2, 5] and I[0, 6:].tolist() == [-1, -1]
    assert torch.all(D[:, 6:] == float("inf")) and torch.all(D[:, 1:6] >= D[:, :5])

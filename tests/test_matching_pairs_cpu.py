"""Argument validation of hn_match_pairs and the pair-table builder: rejected before any device work, so it runs without a GPU."""
import ctypes as C

import pytest
import torch

from hardnetnas_b200 import _lib

HN_ERR_INVALID = -1
FAKE = C.c_void_p(1 << 20)   # never dereferenced: every case below fails validation first


@pytest.fixture(scope="module")
def lib():
    if not _lib.LIB_PATH.exists():
        from hardnetnas_b200 import build
        build.build()
    return _lib.load()


def _call(lib, B=4, max_q=100, max_g=120, nq_rows=1000, ng_rows=900, q=FAKE, q16=FAKE, g=FAKE, g16=FAKE, pairs=FAKE, d1=FAKE,
          i2=FAKE, ws=FAKE, ws_bytes=None, mutual=None):
    if ws_bytes is None:
        ws_bytes = lib.hn_match_pairs_workspace_bytes(B, max_q, max_g, int(mutual is not None))
    null = C.c_void_p(0)
    return lib.hn_match_pairs(q, q16, nq_rows, g, g16, ng_rows, pairs, B, max_q, max_g, d1, FAKE, FAKE, i2,
                              mutual if mutual is not None else null, ws, ws_bytes, null)


def _rejected(lib, status, what):
    assert status == HN_ERR_INVALID
    msg = lib.hn_last_error().decode()
    assert "hn_match_pairs" in msg and what in msg, msg


def test_workspace_bytes_grow_with_the_column_side(lib):
    plain = lib.hn_match_pairs_workspace_bytes(8, 1000, 1000, 0)
    assert plain > 0 and plain % 256 == 0
    assert lib.hn_match_pairs_workspace_bytes(8, 1000, 1000, 1) > plain
    assert lib.hn_match_pairs_workspace_bytes(8, 1000, 4000, 1) > lib.hn_match_pairs_workspace_bytes(8, 1000, 1000, 1)
    # packing is the caller's: no room for packed rows, unlike the padded form
    assert plain < lib.hn_match_batched_workspace_bytes(8, 1000, 1000, 0)
    for args in ((-1, 10, 10), (4, -1, 10), (4, 10, -1)):
        assert lib.hn_match_pairs_workspace_bytes(*args, 0) == 0


@pytest.mark.parametrize("arg", ["q", "q16", "g", "g16", "pairs", "d1", "i2", "ws"])
def test_null_pointer(lib, arg):
    _rejected(lib, _call(lib, **{arg: C.c_void_p(0)}), "NULL")


@pytest.mark.parametrize("B,max_q,max_g,nq_rows,ng_rows", [(0, 10, 10, 50, 50), (3, 0, 10, 50, 50), (3, 10, 0, 50, 50),
                                                           (3, 10, 10, 0, 50), (3, 10, 10, 50, 0), (-2, 10, 10, 50, 50)])
def test_empty_input(lib, B, max_q, max_g, nq_rows, ng_rows):
    _rejected(lib, _call(lib, B=B, max_q=max_q, max_g=max_g, nq_rows=nq_rows, ng_rows=ng_rows, ws_bytes=1 << 30), "empty")


@pytest.mark.parametrize("side", ["q", "g"])
def test_set_of_2_31_rows(lib, side):
    rows = {"nq_rows": 1 << 31} if side == "q" else {"ng_rows": 1 << 31}
    _rejected(lib, _call(lib, **rows), "2^31 rows or more")


@pytest.mark.parametrize("max_q,max_g", [(1 << 19, 16), (16, 1 << 19)])
def test_more_than_2_31_output_rows(lib, max_q, max_g):
    _rejected(lib, _call(lib, B=1 << 12, max_q=max_q, max_g=max_g, ws_bytes=1 << 62), "B*max_q and B*max_g")


@pytest.mark.parametrize("arg", ["q16", "g16"])
def test_misaligned_packed_operands(lib, arg):
    _rejected(lib, _call(lib, **{arg: C.c_void_p((1 << 20) + 8)}), "16-byte aligned")


def test_undersized_workspace(lib):
    need = lib.hn_match_pairs_workspace_bytes(4, 100, 120, 1)
    _rejected(lib, _call(lib, ws_bytes=need - 1, mutual=FAKE), "too small")
    # the column side needs more than the row side alone
    _rejected(lib, _call(lib, ws_bytes=lib.hn_match_pairs_workspace_bytes(4, 100, 120, 0), mutual=FAKE), "too small")


def test_misaligned_workspace(lib):
    _rejected(lib, _call(lib, ws=C.c_void_p((1 << 20) + 64)), "aligned")


def test_cpu_descriptors_raise():
    from hardnetnas_b200.matching import match_top2_pairs, mutual_nn_ratio_pairs
    x = torch.zeros(6, 128)
    table = torch.tensor([[0, 3, 3, 3]], dtype=torch.int32)
    with pytest.raises(_lib.HardnetB200Error):
        match_top2_pairs(x, x, table, 3, 3)
    with pytest.raises(_lib.HardnetB200Error):
        mutual_nn_ratio_pairs(x, x, table)


def test_pair_table_offsets():
    from hardnetnas_b200.matching import pair_table
    counts = torch.tensor([5, 0, 7, 3])
    t = pair_table(counts, [0, 0, 2, 3, 1], [2, 3, 3, 3, 0])
    assert t.dtype == torch.int32 and t.shape == (5, 4)
    starts = [0, 5, 5, 12]
    want = [[starts[a], int(counts[a]), starts[b], int(counts[b])] for a, b in [(0, 2), (0, 3), (2, 3), (3, 3), (1, 0)]]
    assert t.tolist() == want


def test_pair_table_two_sets():
    from hardnetnas_b200.matching import pair_table
    t = pair_table(torch.tensor([4, 6]), torch.tensor([1, 0]), torch.tensor([2, 0]), counts2=torch.tensor([1, 2, 3]))
    assert t.tolist() == [[4, 6, 3, 3], [0, 4, 0, 1]]
    with pytest.raises(ValueError):
        pair_table(torch.tensor([1.0, 2.0]), [0], [1])
    with pytest.raises(ValueError):
        pair_table(torch.tensor([1, 2]), [0, 1], [1])


def test_max_lengths_follow_the_clamping():
    """With max_len* = None the maxima are the largest lengths after the device-side clamping of the table."""
    from hardnetnas_b200.matching import _max_lens
    table = torch.tensor([[0, 5, 90, 50],      # gallery length clamped by the set end: 100 - 90 = 10
                          [95, 30, -4, 7],     # query length clamped to 80 - 80 = 0 (start 95 -> 80); start -4 -> 0
                          [10, -3, 0, 2]])     # negative length -> 0
    assert _max_lens(table, 80, 100, None, None) == (5, 10)
    assert _max_lens(table[1:2], 80, 100, None, None) == (1, 7)   # never below 1
    assert _max_lens(table, 80, 100, 64, None) == (64, 10)
    assert _max_lens(table, 80, 100, 3, 4) == (3, 4)

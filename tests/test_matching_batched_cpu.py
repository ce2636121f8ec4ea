"""Argument validation of hn_match_batched: rejected before any device work, so it runs without a GPU."""
import ctypes as C

import pytest

from hardnetnas_b200 import _lib

HN_ERR_INVALID = -1
FAKE = C.c_void_p(1 << 20)   # never dereferenced: every case below fails validation first


@pytest.fixture(scope="module")
def lib():
    if not _lib.LIB_PATH.exists():
        from hardnetnas_b200 import build
        build.build()
    return _lib.load()


def _call(lib, B=4, nq=100, ng=120, q=FAKE, g=FAKE, d1=FAKE, ws=FAKE, ws_bytes=None, mutual=None):
    if ws_bytes is None:
        ws_bytes = lib.hn_match_batched_workspace_bytes(B, nq, ng, int(mutual is not None))
    null = C.c_void_p(0)
    return lib.hn_match_batched(q, g, B, nq, ng, null, null, d1, FAKE, FAKE, FAKE, mutual if mutual is not None else null, ws,
                                ws_bytes, null)


def _rejected(lib, status, what):
    assert status == HN_ERR_INVALID
    msg = lib.hn_last_error().decode()
    assert "hn_match_batched" in msg and what in msg, msg


def test_workspace_bytes_grow_with_the_column_side(lib):
    plain = lib.hn_match_batched_workspace_bytes(8, 1000, 1000, 0)
    assert plain > 8 * 1000 * 128 * 2 * 2 and plain % 256 == 0
    assert lib.hn_match_batched_workspace_bytes(8, 1000, 1000, 1) > plain
    assert lib.hn_match_batched_workspace_bytes(-1, 10, 10, 0) == 0


@pytest.mark.parametrize("arg", ["q", "g", "d1", "ws"])
def test_null_pointer(lib, arg):
    _rejected(lib, _call(lib, **{arg: C.c_void_p(0)}), "NULL")


@pytest.mark.parametrize("B,nq,ng", [(0, 10, 10), (3, 0, 10), (3, 10, 0), (-2, 10, 10)])
def test_empty_batch_or_rows(lib, B, nq, ng):
    _rejected(lib, _call(lib, B=B, nq=nq, ng=ng, ws_bytes=1 << 30), "empty")


def test_more_than_2_31_rows(lib):
    _rejected(lib, _call(lib, B=1 << 12, nq=1 << 19, ng=16, ws_bytes=1 << 62), "2^31")


def test_undersized_workspace(lib):
    need = lib.hn_match_batched_workspace_bytes(4, 100, 120, 1)
    _rejected(lib, _call(lib, ws_bytes=need - 1, mutual=FAKE), "too small")
    # the column side needs more than the row side alone
    _rejected(lib, _call(lib, ws_bytes=lib.hn_match_batched_workspace_bytes(4, 100, 120, 0), mutual=FAKE), "too small")


def test_misaligned_workspace(lib):
    _rejected(lib, _call(lib, ws=C.c_void_p((1 << 20) + 64)), "aligned")


def test_cpu_descriptors_raise():
    import torch
    from hardnetnas_b200.matching import match_top2_batched
    with pytest.raises(_lib.HardnetB200Error):
        match_top2_batched(torch.zeros(2, 3, 128), torch.zeros(2, 3, 128))

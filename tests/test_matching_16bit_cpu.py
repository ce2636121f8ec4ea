"""Argument validation of the typed matching entry points (fp32 / fp16 / bf16 descriptor rows) and the row-dtype rule of the
Python wrappers: rejected before any device work, so it runs without a GPU."""
import ctypes as C

import pytest
import torch

from hardnetnas_b200 import _lib

HN_ERR_INVALID = -1
FAKE = C.c_void_p(1 << 20)   # never dereferenced: every case below fails validation first
NULL = C.c_void_p(0)
MISALIGNED = C.c_void_p((1 << 20) + 4)   # 4-byte aligned: enough for fp32 rows, not for the 8-byte loads of 16-bit rows


@pytest.fixture(scope="module")
def lib():
    if not _lib.LIB_PATH.exists():
        from hardnetnas_b200 import build
        build.build()
    return _lib.load()


def _pack(lib, dt=_lib.HN_F16, x=FAKE, n=100, out=FAKE, **_):
    return lib.hn_pack_descriptors_typed(x, dt, n, out, NULL)


def _match(lib, dt=_lib.HN_F16, q=FAKE, g=FAKE, nq=100, ng=120, ws=FAKE, ws_bytes=None, q16=NULL, **_):
    if ws_bytes is None:
        ws_bytes = lib.hn_dist_workspace_bytes(nq, ng, 0)
    return lib.hn_match_typed(q, g, dt, q16, NULL, nq, ng, 0, FAKE, FAKE, FAKE, FAKE, NULL, ws, ws_bytes, NULL, NULL)


def _mutual(lib, dt=_lib.HN_F16, q=FAKE, g=FAKE, nq=100, ng=120, ws=FAKE, ws_bytes=None, q16=NULL, **_):
    if ws_bytes is None:
        ws_bytes = lib.hn_mutual_workspace_bytes(nq, ng)
    return lib.hn_match_mutual_typed(q, g, dt, q16, NULL, nq, ng, FAKE, FAKE, FAKE, FAKE, FAKE, ws, ws_bytes, NULL)


def _batched(lib, dt=_lib.HN_F16, q=FAKE, g=FAKE, nq=100, ng=120, B=4, ws=FAKE, ws_bytes=None, **_):
    if ws_bytes is None:
        ws_bytes = lib.hn_match_batched_workspace_bytes(B, nq, ng, 1)
    return lib.hn_match_batched_typed(q, g, dt, B, nq, ng, NULL, NULL, FAKE, FAKE, FAKE, FAKE, FAKE, ws, ws_bytes, NULL)


def _pairs(lib, dt=_lib.HN_F16, q=FAKE, g=FAKE, nq=100, ng=120, B=4, ws=FAKE, ws_bytes=None, q16=FAKE, rows=1000, **_):
    if ws_bytes is None:
        ws_bytes = lib.hn_match_pairs_workspace_bytes(B, nq, ng, 1)
    return lib.hn_match_pairs_typed(q, q16, rows, g, FAKE, rows, dt, FAKE, B, nq, ng, FAKE, FAKE, FAKE, FAKE, FAKE, ws, ws_bytes, NULL)


CALLS = {"hn_pack_descriptors_typed": _pack, "hn_match_typed": _match, "hn_match_mutual_typed": _mutual,
         "hn_match_batched_typed": _batched, "hn_match_pairs_typed": _pairs}
MATCHING = [k for k in CALLS if k != "hn_pack_descriptors_typed"]


def _rejected(lib, fn, status, what):
    assert status == HN_ERR_INVALID
    msg = lib.hn_last_error().decode()
    assert msg.startswith(fn + ":") and what in msg, msg


@pytest.mark.parametrize("fn", list(CALLS))
@pytest.mark.parametrize("dt", [_lib.HN_U8, -1, 4, 1 << 20])
def test_unknown_or_u8_dtype(lib, fn, dt):
    _rejected(lib, fn, CALLS[fn](lib, dt=dt), "desc_dtype must be HN_F32, HN_F16 or HN_BF16")


@pytest.mark.parametrize("fn", list(CALLS))
@pytest.mark.parametrize("arg", ["q", "g", "ws"])
def test_null_pointer(lib, fn, arg):
    if fn == "hn_pack_descriptors_typed":
        arg = {"q": "x", "g": "out", "ws": "x"}[arg]
    _rejected(lib, fn, CALLS[fn](lib, **{arg: NULL}), "NULL")


@pytest.mark.parametrize("fn", list(CALLS))
@pytest.mark.parametrize("dt", [_lib.HN_F16, _lib.HN_BF16])
@pytest.mark.parametrize("side", ["q", "g"])
def test_misaligned_16bit_rows(lib, fn, dt, side):
    if fn == "hn_pack_descriptors_typed":
        side = "x"
    _rejected(lib, fn, CALLS[fn](lib, dt=dt, **{side: MISALIGNED}), "8-byte aligned")


@pytest.mark.parametrize("fn", MATCHING)
def test_fp32_rows_keep_their_alignment_rules(lib, fn):
    """fp32 rows through a typed twin are validated as by the fp32 function: no 8-byte rule (the call then fails on the
    next check, here the undersized workspace)."""
    _rejected(lib, fn, CALLS[fn](lib, dt=_lib.HN_F32, q=MISALIGNED, ws_bytes=1), "too small")


@pytest.mark.parametrize("fn", list(CALLS))
def test_empty_input(lib, fn):
    if fn == "hn_pack_descriptors_typed":
        _rejected(lib, fn, _pack(lib, n=0), "out of range")
    else:
        _rejected(lib, fn, CALLS[fn](lib, nq=0, ws_bytes=1 << 40), "empty")


def test_pack_of_2_31_rows(lib):
    _rejected(lib, "hn_pack_descriptors_typed", _pack(lib, n=1 << 31), "out of range")


def test_more_than_2_31_rows(lib):
    _rejected(lib, "hn_match_typed", _match(lib, nq=1 << 31, ws_bytes=1 << 62), "2^31")
    _rejected(lib, "hn_match_batched_typed", _batched(lib, B=1 << 12, nq=1 << 19, ng=16, ws_bytes=1 << 62), "2^31")
    _rejected(lib, "hn_match_pairs_typed", _pairs(lib, rows=1 << 31), "2^31 rows or more")
    _rejected(lib, "hn_match_pairs_typed", _pairs(lib, B=1 << 12, nq=1 << 19, ng=16, ws_bytes=1 << 62), "B*max_q and B*max_g")


@pytest.mark.parametrize("fn", MATCHING)
def test_undersized_workspace(lib, fn):
    _rejected(lib, fn, CALLS[fn](lib, ws_bytes=1), "too small")


@pytest.mark.parametrize("fn", ["hn_match_typed", "hn_match_batched_typed", "hn_match_pairs_typed"])
def test_misaligned_workspace(lib, fn):
    _rejected(lib, fn, CALLS[fn](lib, ws=C.c_void_p((1 << 20) + 64)), "aligned")


@pytest.mark.parametrize("fn", ["hn_match_typed", "hn_match_pairs_typed"])
def test_misaligned_packed_operands(lib, fn):
    _rejected(lib, fn, CALLS[fn](lib, q16=C.c_void_p((1 << 20) + 8)), "16-byte aligned")


def test_fp32_functions_still_name_themselves(lib):
    """The fp32 entry points are the typed calls with HN_F32 and keep their messages."""
    st = lib.hn_match_batched(FAKE, FAKE, 0, 10, 10, NULL, NULL, FAKE, FAKE, FAKE, FAKE, NULL, FAKE, 1 << 30, NULL)
    _rejected(lib, "hn_match_batched", st, "empty")
    _rejected(lib, "hn_pack_descriptors", lib.hn_pack_descriptors(NULL, 10, FAKE, NULL), "NULL")
    _rejected(lib, "hn_match", lib.hn_match(FAKE, FAKE, 0, 10, 0, FAKE, FAKE, FAKE, FAKE, FAKE, 1 << 30, NULL), "empty")


@pytest.mark.parametrize("fn", MATCHING)
@pytest.mark.parametrize("dt", [_lib.HN_F16, _lib.HN_BF16])
def test_workspace_is_sized_by_the_fp32_functions(lib, fn, dt):
    """The typed twins take the workspace the *_workspace_bytes functions give for the fp32 call: one byte less is too small."""
    need = {"hn_match_typed": lambda: lib.hn_dist_workspace_bytes(100, 120, 0),
            "hn_match_mutual_typed": lambda: lib.hn_mutual_workspace_bytes(100, 120),
            "hn_match_batched_typed": lambda: lib.hn_match_batched_workspace_bytes(4, 100, 120, 1),
            "hn_match_pairs_typed": lambda: lib.hn_match_pairs_workspace_bytes(4, 100, 120, 1)}[fn]()
    _rejected(lib, fn, CALLS[fn](lib, dt=dt, ws_bytes=need - 1), "too small")


def test_row_dtype_rule():
    from hardnetnas_b200._ops import _desc_rows
    h = torch.zeros(4, 128, dtype=torch.float16)
    b = torch.zeros(4, 128, dtype=torch.bfloat16)
    f = torch.zeros(4, 128)
    q, g, dt = _desc_rows(h, h)
    assert dt == _lib.HN_F16 and q is h and g is h
    q, g, dt = _desc_rows(b)
    assert dt == _lib.HN_BF16 and q is b and g is None
    for x, y in ((h, b), (h, f), (f, f), (b, f), (f.double(), f.double())):
        q, g, dt = _desc_rows(x, y)
        assert dt == _lib.HN_F32 and q.dtype == torch.float32 and g.dtype == torch.float32
    t = torch.zeros(128, 4, dtype=torch.float16).t()
    q, _, dt = _desc_rows(t)
    assert dt == _lib.HN_F16 and q.is_contiguous() and torch.equal(q, t)

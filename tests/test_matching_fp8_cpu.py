"""fp8 e4m3 descriptor rows (HN_F8E4M3) without a GPU: the dtype code, the validation of the typed matching entry points and
of hn_forward's out_dtype, and the row-dtype rule of the Python wrappers. Everything here is rejected before device work."""
import ctypes as C
import re
from pathlib import Path

import pytest
import torch

from hardnetnas_b200 import _lib

HN_ERR_INVALID = -1
FAKE = C.c_void_p(1 << 20)   # never dereferenced: every case below fails validation first
NULL = C.c_void_p(0)
ALIGN2 = C.c_void_p((1 << 20) + 2)   # not 4-byte aligned: e4m3 rows are read 4 bytes per lane
ALIGN4 = C.c_void_p((1 << 20) + 4)   # 4-byte aligned: enough for e4m3 rows, not for 16-bit rows
F8 = _lib.HN_F8E4M3


@pytest.fixture(scope="module")
def lib():
    if not _lib.LIB_PATH.exists():
        from hardnetnas_b200 import build
        build.build()
    return _lib.load()


def test_dtype_code_matches_the_header():
    hdr = (Path(__file__).resolve().parents[1] / "include" / "hardnet_b200.h").read_text()
    enum = re.search(r"typedef enum hn_dtype \{([^}]*)\}", hdr).group(1)
    codes = {k: int(v) for k, v in re.findall(r"(HN_\w+)\s*=\s*(\d+)", enum)}
    assert codes["HN_F8E4M3"] == _lib.HN_F8E4M3 == 5
    assert 4 not in codes.values()


def _calls(lib, dt, q=FAKE, g=FAKE, ws_bytes=1 << 40):
    """Every typed entry point on 100 x 120 rows, with a workspace large enough to pass its size check."""
    return {
        "hn_pack_descriptors_typed": lambda: lib.hn_pack_descriptors_typed(q, dt, 100, FAKE, NULL),
        "hn_match_typed": lambda: lib.hn_match_typed(q, g, dt, NULL, NULL, 100, 120, 0, FAKE, FAKE, FAKE, FAKE, NULL, FAKE, ws_bytes,
                                                     NULL, NULL),
        "hn_match_mutual_typed": lambda: lib.hn_match_mutual_typed(q, g, dt, NULL, NULL, 100, 120, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE,
                                                                   ws_bytes, NULL),
        "hn_match_batched_typed": lambda: lib.hn_match_batched_typed(q, g, dt, 4, 100, 120, NULL, NULL, FAKE, FAKE, FAKE, FAKE, FAKE,
                                                                     FAKE, ws_bytes, NULL),
        "hn_match_pairs_typed": lambda: lib.hn_match_pairs_typed(q, FAKE, 1000, g, FAKE, 1000, dt, FAKE, 4, 100, 120, FAKE, FAKE, FAKE,
                                                                 FAKE, FAKE, FAKE, ws_bytes, NULL),
    }


FNS = list(_calls(None, 0))


def _rejected(lib, fn, status, what):
    assert status == HN_ERR_INVALID
    msg = lib.hn_last_error().decode()
    assert msg.startswith(fn + ":") and what in msg, msg


@pytest.mark.parametrize("fn,side", [(f, s) for f in FNS for s in "qg" if f != "hn_pack_descriptors_typed" or s == "q"])
def test_misaligned_e4m3_rows(lib, fn, side):
    _rejected(lib, fn, _calls(lib, F8, **{side: ALIGN2})[fn](), "4-byte aligned")


@pytest.mark.parametrize("fn", FNS[1:])
def test_e4m3_rows_need_only_4_byte_alignment(lib, fn):
    """4-byte-aligned e4m3 rows pass the row checks (the call then fails on the next check, here the undersized workspace),
    while the same pointer is rejected for 16-bit rows."""
    _rejected(lib, fn, _calls(lib, F8, q=ALIGN4, ws_bytes=1)[fn](), "too small")
    _rejected(lib, fn, _calls(lib, _lib.HN_F16, q=ALIGN4, ws_bytes=1)[fn](), "8-byte aligned")


@pytest.mark.parametrize("fn", FNS)
def test_unknown_dtype_message_names_e4m3(lib, fn):
    _rejected(lib, fn, _calls(lib, 4)[fn](), "desc_dtype must be HN_F32, HN_F16 or HN_BF16, or HN_F8E4M3 (got 4)")


@pytest.mark.parametrize("fn", FNS[1:])
def test_e4m3_workspace_is_sized_by_the_fp32_functions(lib, fn):
    need = {"hn_match_typed": lambda: lib.hn_dist_workspace_bytes(100, 120, 0),
            "hn_match_mutual_typed": lambda: lib.hn_mutual_workspace_bytes(100, 120),
            "hn_match_batched_typed": lambda: lib.hn_match_batched_workspace_bytes(4, 100, 120, 1),
            "hn_match_pairs_typed": lambda: lib.hn_match_pairs_workspace_bytes(4, 100, 120, 1)}[fn]()
    _rejected(lib, fn, _calls(lib, F8, ws_bytes=need - 1)[fn](), "too small")


def test_forward_out_dtype_check_in_source():
    """hn_forward, hn_forward_clip and hn_forward_nas accept out_dtype HN_F8E4M3 and size its output rows at one byte per
    element. Their argument checks sit behind the handle, which needs a device, so without one they are read from the source
    (tests/test_matching_fp8_gpu.py runs them)."""
    root = Path(__file__).resolve().parents[1] / "hardnetnas_b200" / "csrc"
    fwd, nas = (root / "hardnet_forward.cu").read_text(), (root / "nas.cu").read_text()
    for src, fn in ((fwd, "hn_forward"), (fwd, "hn_forward_clip"), (nas, "hn_forward_nas")):
        body = src[src.index(f'extern "C" int {fn}('):]
        check = re.search(r"HN_REQUIRE\(([^;]*)\"" + fn + r": bad out_dtype\"", body).group(1)
        assert "out_dtype == HN_F8E4M3" in check, fn
    assert fwd.count("out_dtype == HN_F8E4M3 ? 1 : 2") == 1 and nas.count("out_dtype == HN_F8E4M3 ? 1 : 2") == 1


def test_row_dtype_rule():
    from hardnetnas_b200._ops import _desc_rows
    e = torch.zeros(4, 128, dtype=torch.float8_e4m3fn)
    h = torch.zeros(4, 128, dtype=torch.float16)
    q, g, dt = _desc_rows(e, e)
    assert dt == F8 and q is e and g is e
    q, g, dt = _desc_rows(e)
    assert dt == F8 and q is e and g is None
    e5 = torch.zeros(4, 128, dtype=torch.float8_e5m2)
    for x, y in ((e, h), (h, e), (e5, e5), (e, e5)):
        q, g, dt = _desc_rows(x, y)
        assert dt == _lib.HN_F32 and q.dtype == torch.float32 and g.dtype == torch.float32
    q, _, dt = _desc_rows(e5)
    assert dt == _lib.HN_F32 and q.dtype == torch.float32


@pytest.mark.parametrize("dt,wrong", [(F8, torch.float16), (_lib.HN_F16, torch.float8_e4m3fn), (_lib.HN_F32, torch.float8_e4m3fn),
                                      (_lib.HN_BF16, torch.float8_e4m3fn)])
def test_packed_operands_of_the_other_kind_are_rejected(dt, wrong):
    """e4m3 rows take e4m3 packed operands and every other row type fp16 ones; the wrong kind is refused by its dtype before
    anything else is looked at (the C entry points receive bare pointers and cannot tell them apart)."""
    from hardnetnas_b200._ops import _packed
    with pytest.raises(ValueError, match="e4m3 for e4m3 rows, fp16 otherwise"):
        _packed("match", torch.zeros(10, 128, dtype=wrong), 10, dt)

"""The sharded mutual-NN steps (hn_mutual_claims, hn_mutual_verify) and hn_match's gallery offset without a GPU: offsets out
of range are rejected before any device work, and the float64 mutual-NN oracle agrees with losses_oracle.mutual_nn."""
import ctypes as C

import pytest
import torch

from hardnetnas_b200 import _lib

HN_ERR_INVALID = -1
FAKE = C.c_void_p(1 << 20)   # never dereferenced: every call below fails validation first
NULL = C.c_void_p(0)

# A call that passed validation would launch on the fake pointers; on a machine with a GPU it is not made at all.
no_device = pytest.mark.skipif(torch.cuda.is_available(), reason="fake-pointer calls run only where no CUDA device is visible")


@pytest.fixture(scope="module")
def lib():
    if not _lib.LIB_PATH.exists():
        from hardnetnas_b200 import build
        build.build()
    return _lib.load()


def _rejected(lib, fn, status, what):
    assert status == HN_ERR_INVALID
    msg = lib.hn_last_error().decode()
    assert msg.startswith(fn + ":") and what in msg, msg


def _claims(lib, nq, q_offset, ng=120):
    return lib.hn_mutual_claims(FAKE, FAKE, FAKE, nq, q_offset, FAKE, ng, FAKE, NULL)


def _verify(lib, nq, q_offset, ng=120):
    return lib.hn_mutual_verify(FAKE, nq, q_offset, FAKE, ng, FAKE, FAKE, FAKE, FAKE, NULL)


def _match(lib, ng, g_offset, nq=100):
    return lib.hn_match_typed(FAKE, FAKE, _lib.HN_F32, NULL, NULL, nq, ng, g_offset, FAKE, FAKE, FAKE, FAKE, NULL, FAKE, 1 << 40,
                              NULL, NULL)


@no_device
@pytest.mark.parametrize("q_offset", [-1, -5, -(1 << 31), -(1 << 40)])
def test_negative_q_offset_rejected(lib, q_offset):
    _rejected(lib, "hn_mutual_claims", _claims(lib, 100, q_offset), f"q_offset must be >= 0 (got {q_offset})")
    _rejected(lib, "hn_mutual_verify", _verify(lib, 100, q_offset), f"q_offset must be >= 0 (got {q_offset})")


@no_device
@pytest.mark.parametrize("g_offset", [-1, -7, -(1 << 31)])
def test_negative_g_offset_rejected(lib, g_offset):
    _rejected(lib, "hn_match_typed", _match(lib, 120, g_offset), f"g_offset must be >= 0 (got {g_offset})")
    status = lib.hn_match(FAKE, FAKE, 100, 120, g_offset, FAKE, FAKE, FAKE, FAKE, FAKE, 1 << 40, NULL)
    _rejected(lib, "hn_match", status, f"g_offset must be >= 0 (got {g_offset})")


@no_device
def test_upper_bounds_rejected(lib):
    _rejected(lib, "hn_match_typed", _match(lib, 120, (1 << 31) - 120), "more than 2^31 rows")
    _rejected(lib, "hn_mutual_claims", _claims(lib, 100, (1 << 32) - 100), "size out of range")
    _rejected(lib, "hn_mutual_verify", _verify(lib, 100, (1 << 32) - 100), "size out of range")


def test_mutual_oracle_agrees_with_losses_oracle():
    from oracle import losses_oracle, mutual_oracle, synth
    q, g, _ = synth.make_match_set(500, 700, seed=5)
    q = torch.cat([q, q[:40], torch.zeros(3, 128)])   # duplicate queries and all-zero rows: exact ties on both sides
    g = torch.cat([g, g[:30]])
    fwd, col_min, col_arg, mutual = mutual_oracle.mutual_match(q, g, chunk=128)
    i = torch.arange(q.size(0))
    assert torch.equal(torch.stack([i[mutual], fwd[mutual]], dim=1), losses_oracle.mutual_nn(q.double(), g.double()))
    _, fwd_ref = losses_oracle.nn_match(q.double(), g.double())
    col_ref, bwd_ref = losses_oracle.nn_match(g.double(), q.double())
    assert torch.equal(fwd, fwd_ref) and torch.equal(col_arg, bwd_ref) and torch.equal(col_min, col_ref)
    assert mutual[:40].sum() < 40 and not mutual[-2:].any()   # of two identical rows only the lower one can be mutual

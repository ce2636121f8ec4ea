"""ctypes binding of libhardnet_b200.so (the C ABI declared in include/hardnet_b200.h).

There is no fallback: if the shared library is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "libhardnet_b200.so"

HN_F32, HN_F16, HN_BF16, HN_U8, HN_F8E4M3 = 0, 1, 2, 3, 5
HN_FORM_HARDNET, HN_FORM_FDL = 0, 1
HN_FLAG_LOSS_MASK, HN_FLAG_SWAP, HN_FLAG_NEI_MASK = 1, 2, 4

# name -> (restype, argtypes); kept in sync with include/hardnet_b200.h (tests/test_abi.py checks it)
_P = C.c_void_p
_FPP = C.POINTER(C.c_void_p)
SIGNATURES = {
    "hn_version": (C.c_int, []),
    "hn_last_error": (C.c_char_p, []),
    "hn_launch_count": (C.c_longlong, []),
    "hn_set_hardnet_eps": (C.c_int, [_P, C.c_float, C.c_float]),
    "hn_profile_enable": (C.c_int, [_P, C.c_uint]),
    "hn_profile_read": (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(C.c_longlong)]),
    "hn_create": (C.c_int, [C.POINTER(_P), C.c_int, C.c_longlong]),
    "hn_destroy": (C.c_int, [_P]),
    "hn_pack_hardnet": (C.c_int, [_P, _FPP, _FPP, _FPP, C.c_float, C.c_int]),
    "hn_forward": (C.c_int, [_P, _P, C.c_int, C.c_longlong, _P, C.c_int, _P]),
    "hn_forward_dump": (C.c_int, [_P, _P, C.c_int, C.c_longlong, C.c_int, _P, _P]),
    "hn_pack_nas": (C.c_int, [_P, _P, C.c_int, _P, C.c_longlong, C.c_int]),
    "hn_forward_nas": (C.c_int, [_P, _P, C.c_int, C.c_longlong, _P, C.c_int, _P]),
    "hn_nas_plan": (C.c_int, [_P, C.POINTER(C.c_int), C.c_int]),
    "hn_forward_nas_dump": (C.c_int, [_P, _P, C.c_int, C.c_longlong, C.c_int, _P, _P]),
    "hn_dist_workspace_bytes": (C.c_longlong, [C.c_longlong, C.c_longlong, C.c_int]),
    "hn_dist_min": (C.c_int, [_P, _P, C.c_longlong, C.c_longlong, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P,
                              C.c_longlong, _P]),
    "hn_dist_min_ex": (C.c_int, [_P, _P, C.c_longlong, C.c_longlong, C.c_int, C.c_int, _P, _P, C.c_float, _P, _P, _P, _P, _P, _P,
                                 C.c_longlong, _P]),
    "hn_loss_hardnet": (C.c_int, [_P, _P, C.c_longlong, C.c_float, C.c_int, _P, _P, C.c_longlong, _P]),
    "hn_match": (C.c_int, [_P, _P, C.c_longlong, C.c_longlong, C.c_longlong, _P, _P, _P, _P, _P, C.c_longlong, _P]),
    "hn_pack_descriptors": (C.c_int, [_P, C.c_longlong, _P, _P]),
    "hn_pack_descriptors_multicast": (C.c_int, [_P, C.c_longlong, _P, _P, _P]),
    "hn_match_ex": (C.c_int, [_P, _P, _P, _P, C.c_longlong, C.c_longlong, C.c_longlong, _P, _P, _P, _P, _P, _P, C.c_longlong, _P, _P]),
    "hn_mutual_workspace_bytes": (C.c_longlong, [C.c_longlong, C.c_longlong]),
    "hn_match_mutual": (C.c_int, [_P, _P, _P, _P, C.c_longlong, C.c_longlong, _P, _P, _P, _P, _P, _P, C.c_longlong, _P]),
    "hn_block_max_elems": (C.c_longlong, [C.c_longlong, C.c_longlong]),
    "hn_mutual_claims": (C.c_int, [_P, _P, _P, C.c_longlong, C.c_longlong, _P, C.c_longlong, _P, _P]),
    "hn_mutual_verify": (C.c_int, [_P, C.c_longlong, C.c_longlong, _P, C.c_longlong, _P, _P, _P, _P, _P]),
    "hn_match_batched_workspace_bytes": (C.c_longlong, [C.c_longlong, C.c_longlong, C.c_longlong, C.c_int]),
    "hn_match_batched": (C.c_int, [_P, _P, C.c_longlong, C.c_longlong, C.c_longlong, _P, _P, _P, _P, _P, _P, _P, _P, C.c_longlong, _P]),
    "hn_match_pairs_workspace_bytes": (C.c_longlong, [C.c_longlong, C.c_longlong, C.c_longlong, C.c_int]),
    "hn_match_pairs": (C.c_int, [_P, _P, C.c_longlong, _P, _P, C.c_longlong, _P, C.c_longlong, C.c_longlong, C.c_longlong, _P, _P, _P,
                                 _P, _P, _P, C.c_longlong, _P]),
    "hn_match_force_kernel": (C.c_int, [C.c_int]),
    "hn_pack_descriptors_typed": (C.c_int, [_P, C.c_int, C.c_longlong, _P, _P]),
    "hn_match_typed": (C.c_int, [_P, _P, C.c_int, _P, _P, C.c_longlong, C.c_longlong, C.c_longlong, _P, _P, _P, _P, _P, _P,
                                 C.c_longlong, _P, _P]),
    "hn_match_mutual_typed": (C.c_int, [_P, _P, C.c_int, _P, _P, C.c_longlong, C.c_longlong, _P, _P, _P, _P, _P, _P, C.c_longlong,
                                        _P]),
    "hn_match_batched_typed": (C.c_int, [_P, _P, C.c_int, C.c_longlong, C.c_longlong, C.c_longlong, _P, _P, _P, _P, _P, _P, _P, _P,
                                         C.c_longlong, _P]),
    "hn_match_pairs_typed": (C.c_int, [_P, _P, C.c_longlong, _P, _P, C.c_longlong, C.c_int, _P, C.c_longlong, C.c_longlong,
                                       C.c_longlong, _P, _P, _P, _P, _P, _P, C.c_longlong, _P]),
    "hn_match_topk_workspace_bytes": (C.c_longlong, [C.c_longlong, C.c_longlong]),
    "hn_match_topk_typed": (C.c_int, [_P, _P, C.c_int, _P, _P, C.c_longlong, C.c_longlong, C.c_int, _P, _P, _P, C.c_longlong, _P]),
    "hn_match_pairs_topk_workspace_bytes": (C.c_longlong, [C.c_longlong, C.c_longlong, C.c_longlong]),
    "hn_match_pairs_topk_typed": (C.c_int, [_P, _P, C.c_longlong, _P, _P, C.c_longlong, C.c_int, _P, C.c_longlong, C.c_longlong,
                                            C.c_longlong, C.c_int, _P, _P, _P, C.c_longlong, _P]),
    "hn_match_radius_workspace_bytes": (C.c_longlong, [C.c_longlong, C.c_longlong]),
    "hn_match_radius_count_typed": (C.c_int, [_P, _P, C.c_int, _P, _P, C.c_longlong, C.c_longlong, C.c_float, _P, _P, C.c_longlong,
                                              _P]),
    "hn_match_radius_fill_typed": (C.c_int, [_P, _P, C.c_int, C.c_longlong, C.c_longlong, C.c_float, _P, C.c_longlong, _P, _P, _P,
                                             C.c_longlong, _P]),
    "hn_match_pairs_radius_workspace_bytes": (C.c_longlong, [C.c_longlong, C.c_longlong, C.c_longlong]),
    "hn_match_pairs_radius_count_typed": (C.c_int, [_P, _P, C.c_longlong, _P, _P, C.c_longlong, C.c_int, _P, C.c_longlong, C.c_longlong,
                                                    C.c_longlong, C.c_float, _P, _P, C.c_longlong, _P]),
    "hn_match_pairs_radius_fill_typed": (C.c_int, [_P, _P, C.c_longlong, _P, _P, C.c_longlong, C.c_int, _P, C.c_longlong, C.c_longlong,
                                                   C.c_longlong, C.c_float, _P, C.c_longlong, _P, _P, _P, C.c_longlong, _P]),
    "hn_match_topk_fallback_enable": (C.c_int, [C.c_int]),
    "hn_match_topk_fallback_read": (C.c_int, [C.POINTER(C.c_longlong)]),
    "hn_match_profile_enable": (C.c_int, [C.c_int]),
    "hn_match_profile_read": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_longlong)]),
    "hn_pair_distances": (C.c_int, [_P, _P, C.c_longlong, _P, _P]),
    "hn_fpr95": (C.c_int, [_P, _P, C.c_longlong, _P, _P]),
    "hn_clip_patches": (C.c_int, [_P, C.c_longlong, C.c_int, C.c_int, _P, _P, _P, _P, C.c_longlong, C.c_int, _P, _P]),
    "hn_forward_clip": (C.c_int, [_P, _P, C.c_int, C.c_longlong, C.c_int, C.c_int, _P, _P, _P, _P, C.c_longlong, _P, C.c_int, _P]),
}


class HardnetB200Error(RuntimeError):
    pass


_lib = None


def load(build_if_missing: bool | None = None) -> C.CDLL:
    """Load the extension. With HARDNET_B200_AUTOBUILD=1 (or build_if_missing=True) a missing library is
    compiled in-tree with nvcc first; otherwise a missing library is an error."""
    global _lib
    if _lib is not None:
        return _lib
    if build_if_missing is None:
        build_if_missing = os.environ.get("HARDNET_B200_AUTOBUILD", "0") == "1"
    lib_path = Path(os.environ["HARDNET_B200_LIB"]) if os.environ.get("HARDNET_B200_LIB") else LIB_PATH   # developer switch: A/B builds
    if not lib_path.exists():
        if not build_if_missing:
            raise HardnetB200Error(
                f"{lib_path} is missing: build it with `python -m hardnetnas_b200.build` "
                "(there is no CPU or PyTorch fallback for the accelerated path)")
        from . import build as _build
        _build.build()
    lib = C.CDLL(str(lib_path))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int, what: str) -> None:
    if status != 0:
        msg = load().hn_last_error()
        raise HardnetB200Error(f"{what} failed with status {status}: {msg.decode() if msg else ''}")


def float_ptr_array(tensors) -> C.Array:
    """Array of `const float*` from contiguous fp32 CPU tensors (keeps no reference: caller holds them)."""
    arr = (C.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        assert t.dtype.is_floating_point and t.element_size() == 4 and t.is_contiguous() and not t.is_cuda
        arr[i] = t.data_ptr()
    return arr

"""Tensor-level wrappers over the distance / matching entry points of the C ABI."""
from __future__ import annotations

import ctypes as C
import numbers

import torch

from . import _lib

_ws_cache: dict = {}


def _workspace(device: torch.device, nbytes: int) -> torch.Tensor:
    """Scratch reused across calls (grown on demand), so the hot calls never allocate. One buffer per (device, stream):
    calls on different streams may run concurrently and must not share packed operands or partial minima; a buffer that is
    outgrown is handed back to the caching allocator only after the work queued on its stream (record_stream)."""
    stream = torch.cuda.current_stream(device)
    key = (device.type, device.index, stream.cuda_stream)
    ws = _ws_cache.get(key)
    if ws is None or ws.numel() < nbytes:
        if ws is not None:
            ws.record_stream(stream)
        ws = torch.empty(int(nbytes * 1.25) + 256, dtype=torch.uint8, device=device)
        _ws_cache[key] = ws
    return ws


def _require_cuda_desc(name: str, t: torch.Tensor) -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise _lib.HardnetB200Error(f"{name}: the fused path runs on B200 CUDA tensors only (no CPU fallback)")
    assert t.dim() == 2, "Inputd must be a 2D matrix."
    if t.size(1) != 128:
        raise ValueError(f"{name}: descriptors must be 128-d, got {t.size(1)}")
    return t.detach()


def _require_cuda_f32(name: str, t: torch.Tensor) -> torch.Tensor:
    return _require_cuda_desc(name, t).float().contiguous()


_ROW_DTYPES = {torch.float16: _lib.HN_F16, torch.bfloat16: _lib.HN_BF16, torch.float8_e4m3fn: _lib.HN_F8E4M3}


def _desc_rows(q: torch.Tensor, g: torch.Tensor | None = None):
    """(q, g, desc_dtype) for the *_typed matching entry points: fp16, bf16 and fp8 e4m3 (torch.float8_e4m3fn) rows are read
    as they are (made contiguous) when both sides share the dtype, so no fp32 copy is made; anything else (fp32, fp64,
    float8_e5m2, mixed dtypes) is converted to fp32. The results are the same either way (include/hardnet_b200.h).
    g = None: a single set."""
    code = _ROW_DTYPES.get(q.dtype) if g is None or g.dtype == q.dtype else None
    if code is None:
        return q.float().contiguous(), (None if g is None else g.float().contiguous()), _lib.HN_F32
    return q.contiguous(), (None if g is None else g.contiguous()), code


def _stream_ptr() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def dist_min(a: torch.Tensor, p: torch.Tensor, form: int, loss_mask: bool, swap: bool, a_xy: torch.Tensor | None = None,
             p_xy: torch.Tensor | None = None, nei_c: float = 0.0):
    """Returns dict(pos, row_min, row_arg[, col_min, col_arg]) — see hn_dist_min / hn_dist_min_ex in include/hardnet_b200.h.
    a_xy / p_xy ([N,2] keypoint coordinates) switch on the neighbour mask of HardNetNeiMask.loss."""
    lib = _lib.load()
    a = _require_cuda_f32("dist_min", a)
    p = _require_cuda_f32("dist_min", p)
    na, npos = a.size(0), p.size(0)
    dev = a.device
    nei = a_xy is not None
    if nei:
        a_xy = a_xy.detach().to(dev, torch.float32).contiguous()
        p_xy = p_xy.detach().to(dev, torch.float32).contiguous()
        assert tuple(a_xy.shape) == (na, 2) and tuple(p_xy.shape) == (npos, 2), "keypoint coordinates must be [N,2]"
    with torch.cuda.device(dev):
        ws = _workspace(dev, lib.hn_dist_workspace_bytes(na, npos, 1))
        has_pos = loss_mask or nei
        out = {
            "pos": torch.empty(min(na, npos), dtype=torch.float32, device=dev) if has_pos else None,
            "row_min": torch.empty(na, dtype=torch.float32, device=dev),
            "row_arg": torch.empty(na, dtype=torch.int32, device=dev),
            "col_min": torch.empty(npos, dtype=torch.float32, device=dev) if swap else None,
            "col_arg": torch.empty(npos, dtype=torch.int32, device=dev) if swap else None,
        }
        flags = (_lib.HN_FLAG_LOSS_MASK if loss_mask else 0) | (_lib.HN_FLAG_SWAP if swap else 0) | (_lib.HN_FLAG_NEI_MASK if nei else 0)
        _lib.check(lib.hn_dist_min_ex(_ptr(a), _ptr(p), na, npos, form, flags, _ptr(a_xy), _ptr(p_xy), C.c_float(nei_c),
                                      _ptr(out["pos"]), _ptr(out["row_min"]), _ptr(out["row_arg"]), _ptr(out["col_min"]),
                                      _ptr(out["col_arg"]), _ptr(ws), ws.numel(), _stream_ptr()), "hn_dist_min")
    return out


def loss_hardnet(anchor: torch.Tensor, positive: torch.Tensor, margin: float, anchor_swap: bool) -> torch.Tensor:
    lib = _lib.load()
    a = _require_cuda_f32("loss_HardNet", anchor)
    p = _require_cuda_f32("loss_HardNet", positive)
    n = a.size(0)
    dev = a.device
    with torch.cuda.device(dev):
        ws = _workspace(dev, lib.hn_dist_workspace_bytes(n, n, 1))
        out = torch.empty((), dtype=torch.float32, device=dev)
        _lib.check(lib.hn_loss_hardnet(_ptr(a), _ptr(p), n, C.c_float(margin), int(bool(anchor_swap)), _ptr(out), _ptr(ws),
                                       ws.numel(), _stream_ptr()), "hn_loss_hardnet")
    return out


def _packed_dtype(desc_dtype: int) -> torch.dtype:
    """dtype of the packed operand rows of a matching call on rows of desc_dtype: e4m3 for e4m3 rows, fp16 otherwise."""
    return torch.float8_e4m3fn if desc_dtype == _lib.HN_F8E4M3 else torch.float16


def pack_descriptors(x: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
    """[n,128] unit rows (fp32, or fp16 / bf16 / fp8 e4m3 read as they are) -> the operand rows of the matching GEMM (x * 2^8),
    see hn_pack_descriptors_typed: fp16 rows, or e4m3 rows for e4m3 input (exact: |x| <= 1). `out`: optional destination
    (e.g. a symmetric-memory exchange buffer) of that dtype."""
    lib = _lib.load()
    x, _, dt = _desc_rows(_require_cuda_desc("pack_descriptors", x))
    pdt = _packed_dtype(dt)
    if out is None:
        out = torch.empty((x.size(0), 128), dtype=pdt, device=x.device)
    elif not (out.is_cuda and out.dtype == pdt and tuple(out.shape) == (x.size(0), 128) and out.is_contiguous()):
        raise ValueError(f"pack_descriptors: out must be a contiguous CUDA {pdt} [n,128] tensor")
    if x.size(0):
        with torch.cuda.device(x.device):
            _lib.check(lib.hn_pack_descriptors_typed(_ptr(x), dt, x.size(0), _ptr(out), _stream_ptr()), "hn_pack_descriptors_typed")
    return out


def pack_descriptors_multicast(x: torch.Tensor, mc16_ptr: int, mc32_ptr: int) -> None:
    """Pack x:[n,128] and push the fp16 and the fp32 rows to multicast addresses (hn_pack_descriptors_multicast)."""
    lib = _lib.load()
    x = _require_cuda_f32("pack_descriptors_multicast", x)
    with torch.cuda.device(x.device):
        _lib.check(lib.hn_pack_descriptors_multicast(_ptr(x), x.size(0), C.c_void_p(mc16_ptr), C.c_void_p(mc32_ptr), _stream_ptr()),
                   "hn_pack_descriptors_multicast")


def match_top2(q: torch.Tensor, g: torch.Tensor, g_offset: int = 0, q16: torch.Tensor | None = None,
               g16: torch.Tensor | None = None, g_ready_event: torch.cuda.Event | None = None,
               block_max: torch.Tensor | None = None):
    """(d1, d2, i1, i2): nearest / second-nearest gallery row per query in the FDLNet distance form.
    q16 / g16: operands already packed by `pack_descriptors` (skips the packing kernels); g_ready_event: the exact re-rank
    (the only reader of the fp32 gallery `g`) waits for it, so `g` may still be arriving while the GEMM runs.
    block_max: optional fp32 tensor of `block_max_elems(nq, ng)` elements that receives the GEMM's per-cell maxima (column side
    of mutual NN, see hn_match_mutual). fp16 / bf16 / fp8 e4m3 rows of one dtype are read as they are (hn_match_typed); packed
    operands are then of the dtype pack_descriptors gives for them (e4m3 for e4m3 rows, fp16 otherwise)."""
    lib = _lib.load()
    q, g, dt = _desc_rows(_require_cuda_desc("match", q), _require_cuda_desc("match", g))
    nq, ng = q.size(0), g.size(0)
    for t, n in ((q16, nq), (g16, ng)):
        if t is not None:
            _packed("match", t, n, dt)
    dev = q.device
    if block_max is not None:
        _buffer("match", "block_max", block_max, torch.float32, dev, min_numel=block_max_elems(nq, ng))
    with torch.cuda.device(dev):
        ws = _workspace(dev, lib.hn_dist_workspace_bytes(nq, ng, 0))
        d1 = torch.empty(nq, dtype=torch.float32, device=dev)
        d2 = torch.empty(nq, dtype=torch.float32, device=dev)
        i1 = torch.empty(nq, dtype=torch.int32, device=dev)
        i2 = torch.empty(nq, dtype=torch.int32, device=dev)
        ev = C.c_void_p(g_ready_event.cuda_event) if g_ready_event is not None else C.c_void_p(0)
        _lib.check(lib.hn_match_typed(_ptr(q), _ptr(g), dt, _ptr(q16), _ptr(g16), nq, ng, g_offset, _ptr(d1), _ptr(d2), _ptr(i1),
                                      _ptr(i2), _ptr(block_max), _ptr(ws), ws.numel(), ev, _stream_ptr()), "hn_match_typed")
    return d1, d2, i1, i2


def block_max_elems(nq: int, ng: int) -> int:
    return int(_lib.load().hn_block_max_elems(nq, ng))


def match_mutual(q: torch.Tensor, g: torch.Tensor, q16: torch.Tensor | None = None, g16: torch.Tensor | None = None):
    """(d1, d2, i1, i2, mutual bool[Nq]) from ONE matching GEMM: hn_match_mutual_typed (rows as in match_top2)."""
    lib = _lib.load()
    q, g, dt = _desc_rows(_require_cuda_desc("match_mutual", q), _require_cuda_desc("match_mutual", g))
    nq, ng = q.size(0), g.size(0)
    dev = q.device
    with torch.cuda.device(dev):
        ws = _workspace(dev, lib.hn_mutual_workspace_bytes(nq, ng))
        d1 = torch.empty(nq, dtype=torch.float32, device=dev)
        d2 = torch.empty(nq, dtype=torch.float32, device=dev)
        i1 = torch.empty(nq, dtype=torch.int32, device=dev)
        i2 = torch.empty(nq, dtype=torch.int32, device=dev)
        mutual = torch.empty(nq, dtype=torch.bool, device=dev)
        _lib.check(lib.hn_match_mutual_typed(_ptr(q), _ptr(g), dt, _ptr(q16), _ptr(g16), nq, ng, _ptr(d1), _ptr(d2), _ptr(i1),
                                             _ptr(i2), _ptr(mutual), _ptr(ws), ws.numel(), _stream_ptr()), "hn_match_mutual_typed")
    return d1, d2, i1, i2, mutual


def _require_cuda_desc_batched(name: str, t: torch.Tensor) -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise _lib.HardnetB200Error(f"{name}: the fused path runs on B200 CUDA tensors only (no CPU fallback)")
    if t.dim() != 3:
        raise ValueError(f"{name}: descriptors must be a padded batch [B, N, 128], got shape {tuple(t.shape)}")
    if t.size(2) != 128:
        raise ValueError(f"{name}: descriptors must be 128-d, got {t.size(2)}")
    return t.detach()


def _lengths(name: str, t, batch: int, device: torch.device):
    if t is None:
        return None
    if not isinstance(t, torch.Tensor) or t.dtype.is_floating_point or t.dtype.is_complex or t.dtype == torch.bool:
        raise ValueError(f"{name}: lengths must be an integer tensor of shape [{batch}]")
    if tuple(t.shape) != (batch,):
        raise ValueError(f"{name}: lengths must have shape [{batch}], got {tuple(t.shape)}")
    return t.to(device=device, dtype=torch.int32).contiguous()


def match_batched(q: torch.Tensor, g: torch.Tensor, q_len: torch.Tensor | None = None, g_len: torch.Tensor | None = None,
                  mutual: bool = False):
    """(d1, d2, i1, i2[, mutual]), each [B, Nq]: hn_match_batched over the padded batches q [B, Nq, 128] and g [B, Ng, 128].
    q_len / g_len: integer [B] tensors of valid rows per pair (None = all). Lengths on q's device keep the call free of host
    synchronisation (and CUDA-graph capturable); a CPU lengths tensor is copied to the device first. Indices are local to the
    pair; rows past q_len get d = +inf, i = -1 (and mutual = False). Rows as in match_top2 (hn_match_batched_typed)."""
    lib = _lib.load()
    q, g, dt = _desc_rows(_require_cuda_desc_batched("match_batched", q), _require_cuda_desc_batched("match_batched", g))
    if q.size(0) != g.size(0):
        raise ValueError(f"match_batched: q and g hold {q.size(0)} and {g.size(0)} pairs")
    b, nq, ng = q.size(0), q.size(1), g.size(1)
    dev = q.device
    ql = _lengths("match_batched q_len", q_len, b, dev)
    gl = _lengths("match_batched g_len", g_len, b, dev)
    with torch.cuda.device(dev):
        ws = _workspace(dev, max(lib.hn_match_batched_workspace_bytes(b, nq, ng, int(mutual)), 1))
        d1 = torch.empty((b, nq), dtype=torch.float32, device=dev)
        d2 = torch.empty((b, nq), dtype=torch.float32, device=dev)
        i1 = torch.empty((b, nq), dtype=torch.int32, device=dev)
        i2 = torch.empty((b, nq), dtype=torch.int32, device=dev)
        mu = torch.empty((b, nq), dtype=torch.bool, device=dev) if mutual else None
        _lib.check(lib.hn_match_batched_typed(_ptr(q), _ptr(g), dt, b, nq, ng, _ptr(ql), _ptr(gl), _ptr(d1), _ptr(d2), _ptr(i1),
                                              _ptr(i2), _ptr(mu), _ptr(ws), ws.numel(), _stream_ptr()), "hn_match_batched_typed")
    return (d1, d2, i1, i2, mu) if mutual else (d1, d2, i1, i2)


def _packed(name: str, t: torch.Tensor, n: int, desc_dtype: int) -> torch.Tensor:
    """Checks packed operand rows against the rows they were made from: the C ABI receives a bare pointer and cannot tell an
    fp16 operand from an e4m3 one."""
    pdt = _packed_dtype(desc_dtype)
    if not (isinstance(t, torch.Tensor) and t.dtype == pdt and t.is_cuda and tuple(t.shape) == (n, 128) and t.is_contiguous()):
        raise ValueError(f"{name}: packed operands must be contiguous CUDA {pdt} [n,128] tensors from pack_descriptors "
                         f"(e4m3 for e4m3 rows, fp16 otherwise)")
    return t


def _pair_operands(name: str, q: torch.Tensor, g: torch.Tensor, pairs: torch.Tensor, q16: torch.Tensor | None,
                   g16: torch.Tensor | None):
    """(q, g, desc_dtype, device int32 table, q16, g16) of a pair-table call: rows as _desc_rows, the sets packed here unless
    their packed rows are given (once when g is q), packed rows checked against the rows."""
    same = g is q
    if same:
        q, _, dt = _desc_rows(_require_cuda_desc(name, q))
        g = q
    else:
        q, g, dt = _desc_rows(_require_cuda_desc(name, q), _require_cuda_desc(name, g))
    if not isinstance(pairs, torch.Tensor) or pairs.dtype not in (torch.int32, torch.int64) or pairs.dim() != 2 or pairs.size(1) != 4:
        raise ValueError(f"{name}: pairs must be an int32 or int64 [P, 4] tensor of (q_start, q_len, g_start, g_len)")
    dev = q.device
    if g.device != dev:
        raise ValueError(f"{name}: q and g must be on the same device")
    table = pairs.to(device=dev, dtype=torch.int32).contiguous()
    if q16 is None:
        q16 = g16 if same and g16 is not None else pack_descriptors(q)
    if g16 is None:
        g16 = q16 if same else pack_descriptors(g)
    return q, g, dt, table, _packed(name, q16, q.size(0), dt), _packed(name, g16, g.size(0), dt)


def match_pairs(q: torch.Tensor, g: torch.Tensor, pairs: torch.Tensor, max_q: int, max_g: int, q16: torch.Tensor | None = None,
                g16: torch.Tensor | None = None, mutual: bool = False):
    """(d1, d2, i1, i2[, mutual]), each [P, max_q]: hn_match_pairs over the concatenated sets q [Nq_rows, 128] and
    g [Ng_rows, 128]. pairs: integer [P, 4] table of (q_start, q_len, g_start, g_len), copied to q's device as int32 (a table
    already there keeps the call free of host synchronisation). q16 / g16: the sets' rows packed by `pack_descriptors`; a set
    whose packed rows are not given is packed here (per row dtype, see pack_descriptors), once when g is q. Indices are local to the pair's gallery range; rows past
    q_len get d = +inf, i = -1 (and mutual = False). Rows as in match_top2 (hn_match_pairs_typed)."""
    lib = _lib.load()
    q, g, dt, table, q16, g16 = _pair_operands("match_pairs", q, g, pairs, q16, g16)
    nq, ng, b = q.size(0), g.size(0), table.size(0)
    dev = q.device
    with torch.cuda.device(dev):
        ws = _workspace(dev, max(lib.hn_match_pairs_workspace_bytes(b, max_q, max_g, int(mutual)), 1))
        d1 = torch.empty((b, max_q), dtype=torch.float32, device=dev)
        d2 = torch.empty((b, max_q), dtype=torch.float32, device=dev)
        i1 = torch.empty((b, max_q), dtype=torch.int32, device=dev)
        i2 = torch.empty((b, max_q), dtype=torch.int32, device=dev)
        mu = torch.empty((b, max_q), dtype=torch.bool, device=dev) if mutual else None
        _lib.check(lib.hn_match_pairs_typed(_ptr(q), _ptr(q16), nq, _ptr(g), _ptr(g16), ng, dt, _ptr(table), b, max_q, max_g,
                                            _ptr(d1), _ptr(d2), _ptr(i1), _ptr(i2), _ptr(mu), _ptr(ws), ws.numel(), _stream_ptr()),
                   "hn_match_pairs_typed")
    return (d1, d2, i1, i2, mu) if mutual else (d1, d2, i1, i2)


TOPK_MAX = 8


def _check_k(name: str, k) -> int:
    if isinstance(k, bool) or not isinstance(k, int) or not 1 <= k <= TOPK_MAX:
        raise ValueError(f"{name}: k must be an integer in [1, {TOPK_MAX}], got {k!r}")
    return k


def match_topk(q: torch.Tensor, g: torch.Tensor, k: int, q16: torch.Tensor | None = None, g16: torch.Tensor | None = None):
    """(dist [Nq, k] fp32, idx [Nq, k] int32): the k nearest gallery rows per query, sorted by (distance, index), exact
    (hn_match_topk_typed). Rows and packed operands as in match_top2; missing slots (Ng < k) are +inf / -1."""
    k = _check_k("match_topk", k)
    lib = _lib.load()
    q, g, dt = _desc_rows(_require_cuda_desc("match_topk", q), _require_cuda_desc("match_topk", g))
    nq, ng = q.size(0), g.size(0)
    for t, n in ((q16, nq), (g16, ng)):
        if t is not None:
            _packed("match_topk", t, n, dt)
    dev = q.device
    with torch.cuda.device(dev):
        ws = _workspace(dev, lib.hn_match_topk_workspace_bytes(nq, ng))
        dist = torch.empty((nq, k), dtype=torch.float32, device=dev)
        idx = torch.empty((nq, k), dtype=torch.int32, device=dev)
        _lib.check(lib.hn_match_topk_typed(_ptr(q), _ptr(g), dt, _ptr(q16), _ptr(g16), nq, ng, k, _ptr(dist), _ptr(idx), _ptr(ws),
                                           ws.numel(), _stream_ptr()), "hn_match_topk_typed")
    return dist, idx


def match_pairs_topk(q: torch.Tensor, g: torch.Tensor, pairs: torch.Tensor, k: int, max_q: int, max_g: int,
                     q16: torch.Tensor | None = None, g16: torch.Tensor | None = None):
    """(dist, idx), each [P, max_q, k]: hn_match_pairs_topk_typed over the pair table (arguments as in match_pairs)."""
    k = _check_k("match_pairs_topk", k)
    lib = _lib.load()
    q, g, dt, table, q16, g16 = _pair_operands("match_pairs_topk", q, g, pairs, q16, g16)
    nq, ng, b = q.size(0), g.size(0), table.size(0)
    dev = q.device
    with torch.cuda.device(dev):
        ws = _workspace(dev, max(lib.hn_match_pairs_topk_workspace_bytes(b, max_q, max_g), 1))
        dist = torch.empty((b, max_q, k), dtype=torch.float32, device=dev)
        idx = torch.empty((b, max_q, k), dtype=torch.int32, device=dev)
        _lib.check(lib.hn_match_pairs_topk_typed(_ptr(q), _ptr(q16), nq, _ptr(g), _ptr(g16), ng, dt, _ptr(table), b, max_q, max_g, k,
                                                 _ptr(dist), _ptr(idx), _ptr(ws), ws.numel(), _stream_ptr()),
                   "hn_match_pairs_topk_typed")
    return dist, idx


def _check_radius(name: str, radius, capacity) -> tuple[float, int | None]:
    if isinstance(radius, bool) or not isinstance(radius, numbers.Real) or radius != radius:
        raise ValueError(f"{name}: radius must be a real number, got {radius!r}")
    if capacity is not None and (isinstance(capacity, bool) or not isinstance(capacity, int) or capacity < 0):
        raise ValueError(f"{name}: capacity must be None or an integer >= 0, got {capacity!r}")
    return float(radius), capacity


def _radius_csr(dev: torch.device, rows: int, capacity: int | None, count, fill):
    """Count into row_ptr [rows + 1], then fill col int32 / dist fp32 buffers of `capacity` entries, or, with capacity None, of the
    counted size (one host read of row_ptr[rows]). count(row_ptr) and fill(row_ptr, capacity, col, dist) launch the two phases."""
    with torch.cuda.device(dev):
        row_ptr = torch.empty(rows + 1, dtype=torch.int64, device=dev)
        count(row_ptr)
        n = int(row_ptr[rows]) if capacity is None else capacity
        col = torch.empty(n, dtype=torch.int32, device=dev)
        dist = torch.empty(n, dtype=torch.float32, device=dev)
        fill(row_ptr, n, col, dist)
    return row_ptr, col, dist


def match_radius(q: torch.Tensor, g: torch.Tensor, radius: float, capacity: int | None = None, q16: torch.Tensor | None = None,
                 g16: torch.Tensor | None = None):
    """(row_ptr int64 [Nq + 1], col int32, dist fp32): CSR of every (query, gallery) pair with d < radius, columns ascending per
    row (hn_match_radius_count_typed + hn_match_radius_fill_typed). Rows and packed operands as in match_topk. capacity=None:
    exact-size outputs after one host read of the total; capacity=n: buffers of n entries and no host synchronisation, entries at
    CSR positions >= n are not written (row_ptr[-1] > n tells the output was truncated)."""
    radius, capacity = _check_radius("match_radius", radius, capacity)
    lib = _lib.load()
    q, g, dt = _desc_rows(_require_cuda_desc("match_radius", q), _require_cuda_desc("match_radius", g))
    nq, ng = q.size(0), g.size(0)
    for t, n in ((q16, nq), (g16, ng)):
        if t is not None:
            _packed("match_radius", t, n, dt)
    dev = q.device
    with torch.cuda.device(dev):
        ws = _workspace(dev, lib.hn_match_radius_workspace_bytes(nq, ng))
    r = C.c_float(radius)

    def count(row_ptr):
        _lib.check(lib.hn_match_radius_count_typed(_ptr(q), _ptr(g), dt, _ptr(q16), _ptr(g16), nq, ng, r, _ptr(row_ptr), _ptr(ws),
                                                   ws.numel(), _stream_ptr()), "hn_match_radius_count_typed")

    def fill(row_ptr, n, col, dist):
        _lib.check(lib.hn_match_radius_fill_typed(_ptr(q), _ptr(g), dt, nq, ng, r, _ptr(row_ptr), n, _ptr(col), _ptr(dist), _ptr(ws),
                                                  ws.numel(), _stream_ptr()), "hn_match_radius_fill_typed")

    return _radius_csr(dev, nq, capacity, count, fill)


def match_pairs_radius(q: torch.Tensor, g: torch.Tensor, pairs: torch.Tensor, radius: float, max_q: int, max_g: int,
                       capacity: int | None = None, q16: torch.Tensor | None = None, g16: torch.Tensor | None = None):
    """(row_ptr int64 [P * max_q + 1], col int32, dist fp32): match_radius over the [P * max_q] padded rows of the pair table
    (hn_match_pairs_radius_*_typed; arguments as in match_pairs), columns local to the pair's gallery range."""
    radius, capacity = _check_radius("match_pairs_radius", radius, capacity)
    lib = _lib.load()
    q, g, dt, table, q16, g16 = _pair_operands("match_pairs_radius", q, g, pairs, q16, g16)
    nq, ng, b = q.size(0), g.size(0), table.size(0)
    dev = q.device
    with torch.cuda.device(dev):
        ws = _workspace(dev, max(lib.hn_match_pairs_radius_workspace_bytes(b, max_q, max_g), 1))
    r = C.c_float(radius)

    def count(row_ptr):
        _lib.check(lib.hn_match_pairs_radius_count_typed(_ptr(q), _ptr(q16), nq, _ptr(g), _ptr(g16), ng, dt, _ptr(table), b, max_q, max_g,
                                                         r, _ptr(row_ptr), _ptr(ws), ws.numel(), _stream_ptr()),
                   "hn_match_pairs_radius_count_typed")

    def fill(row_ptr, n, col, dist):
        _lib.check(lib.hn_match_pairs_radius_fill_typed(_ptr(q), _ptr(q16), nq, _ptr(g), _ptr(g16), ng, dt, _ptr(table), b, max_q, max_g,
                                                        r, _ptr(row_ptr), n, _ptr(col), _ptr(dist), _ptr(ws), ws.numel(), _stream_ptr()),
                   "hn_match_pairs_radius_fill_typed")

    return _radius_csr(dev, b * max_q, capacity, count, fill)


def _buffer(name: str, what: str, t, dtype: torch.dtype, device: torch.device, numel: int | None = None,
            min_numel: int | None = None) -> torch.Tensor:
    """Checks a tensor the C ABI reads or writes through a bare pointer at a length it derives from other arguments: a wrong
    dtype, device, layout or size would be read or written out of bounds."""
    if not (isinstance(t, torch.Tensor) and t.dtype == dtype and t.device == device and t.is_contiguous()):
        raise ValueError(f"{name}: {what} must be a contiguous {dtype} tensor on {device}")
    if (numel is not None and t.numel() != numel) or (min_numel is not None and t.numel() < min_numel):
        size = f"{numel}" if numel is not None else f"at least {min_numel}"
        raise ValueError(f"{name}: {what} must have {size} elements, got {t.numel()}")
    return t


def mutual_claims(i1: torch.Tensor, d1: torch.Tensor, d2: torch.Tensor, q_offset: int, claim: torch.Tensor) -> torch.Tensor:
    """atomicMin of (distance, global row) into claim[int64, Ng] (pre-filled with INT64_MAX = unclaimed); returns the per
    32-row-block minimum of d2 the verification needs."""
    lib = _lib.load()
    if not (isinstance(i1, torch.Tensor) and i1.is_cuda):
        raise ValueError("mutual_claims: i1 must be a CUDA tensor")
    dev, nq = i1.device, i1.numel()
    _buffer("mutual_claims", "i1", i1, torch.int32, dev)
    _buffer("mutual_claims", "d1", d1, torch.float32, dev, numel=nq)
    _buffer("mutual_claims", "d2", d2, torch.float32, dev, numel=nq)
    _buffer("mutual_claims", "claim", claim, torch.int64, dev)
    rbmin = torch.empty((nq + 31) // 32, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.hn_mutual_claims(_ptr(i1), _ptr(d1), _ptr(d2), nq, q_offset, _ptr(claim), claim.numel(), _ptr(rbmin),
                                        _stream_ptr()), "hn_mutual_claims")
    return rbmin


def mutual_verify(q: torch.Tensor, q_offset: int, g: torch.Tensor, claim: torch.Tensor, block_max: torch.Tensor,
                  rb_min_d2: torch.Tensor, beaten: torch.Tensor):
    """beaten[uint8, Ng] |= some local query row is nearer to g_j than the claimant of column j. q / g: fp32 [n,128] rows."""
    lib = _lib.load()
    q, g = _require_cuda_desc("mutual_verify", q), _require_cuda_desc("mutual_verify", g)
    dev, nq, ng = q.device, q.size(0), g.size(0)
    _buffer("mutual_verify", "q", q, torch.float32, dev)
    _buffer("mutual_verify", "g", g, torch.float32, dev)
    _buffer("mutual_verify", "claim", claim, torch.int64, dev, numel=ng)
    _buffer("mutual_verify", "block_max", block_max, torch.float32, dev, min_numel=block_max_elems(nq, ng))
    _buffer("mutual_verify", "rb_min_d2", rb_min_d2, torch.float32, dev, min_numel=(nq + 31) // 32)
    _buffer("mutual_verify", "beaten", beaten, torch.uint8, dev, numel=ng)
    with torch.cuda.device(dev):
        _lib.check(lib.hn_mutual_verify(_ptr(q), nq, q_offset, _ptr(g), ng, _ptr(claim), _ptr(block_max),
                                        _ptr(rb_min_d2), _ptr(beaten), _stream_ptr()), "hn_mutual_verify")

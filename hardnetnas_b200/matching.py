"""Drop-in mirror of the descriptor-matching part of FDLNet-master/utils/{math_utils,eval_utils}.py.

The reference materialises the full distance matrix and then takes `min` (eval_utils.py:113-114) or a full
row `sort` (:168-175). Here one fused pass (tensor-core GEMM + in-register shortlist, exact fp32 re-rank)
returns the nearest and second-nearest gallery row per query; nothing of size Nq x Ng is ever stored.
Descriptors may be fp32, fp16, bf16 or fp8 e4m3 (torch.float8_e4m3fn): fp16 / bf16 / e4m3 tensors of one dtype (e.g.
`HardNet.forward(x, out_dtype=torch.float16)`) are matched as they are, without an fp32 copy, with results bit-identical to the
same call on their `.float()`; e4m3 rows are matched on the fp8 tensor core. Mixed or other dtypes (float8_e5m2 included) are
converted to fp32 first.
"""
from __future__ import annotations

import torch

from . import _ops


def assert_unit_norm(des, tol: float = 1e-3):
    """Precondition of the fused matching kernels (include/hardnet_b200.h, hn_match): rows are L2-normalised descriptors, the
    only input the FDLNet distance form `sqrt(2 - 2 a.b)` is defined for. The kernels do not check it (their fp16 operand
    packing and the re-rank margin assume |x| <= 1); call this once on descriptors of unknown origin - one device
    synchronisation, raises ValueError naming the first offending row. Unit descriptors rounded to e4m3
    (torch.float8_e4m3fn) keep their norm within (2^-4 + sqrt(128) * 2^-10) < 0.074 of 1 (random unit rows: within about
    0.006), so check those with tol=0.075."""
    n = des.float().norm(dim=1)
    bad = ((n - 1.0).abs() > tol) & (n > 0)        # all-zero rows (constant patches) are legal and match nothing
    if bool(bad.any()):
        i = int(bad.nonzero()[0])
        raise ValueError(f"descriptor row {i} has L2 norm {float(n[i]):.6f}: the matching kernels need unit-norm rows "
                         f"(|norm - 1| <= {tol})")
    return des


def distance_matrix_vector(anchor, positive):
    """Materialising API for small inputs (FDLNet-master/utils/math_utils.py:8-19)."""
    m = 2 - 2 * torch.mm(anchor, positive.t())
    return torch.sqrt(m.clamp(min=1e-8, max=4.0))


def pairwise_distances(x, y=None):
    """L2 distances between the rows of x and y (y = x when omitted), FDLNet-master/utils/math_utils.py:22-40:
    sqrt(clamp(|x|^2 + |y|^2 - 2 x.y, min=1e-8)). Small coordinate sets only (keypoints); descriptors go through the fused
    matching kernel."""
    y = x if y is None else y
    d = (x * x).sum(1).view(-1, 1) + (y * y).sum(1).view(1, -1) - 2.0 * torch.mm(x, y.t())
    return torch.sqrt(d.clamp(min=1e-8))


def nearest_neighbor_match(des1, des2):
    """`des_dist_matrix.min(dim=-1)` of eval_utils.py:113-114 -> (nn_value [Nq] fp32, nn_idx [Nq] int64)."""
    d1, _, i1, _ = _ops.match_top2(des1, des2)
    return d1, i1.long()


def nearest_neighbor_threshold_match(des1, des2, des_thrsh):
    """nn_value.lt(DES_THRSH) of eval_utils.py:133-135 -> (predict_label, nn_idx)."""
    d1, _, i1, _ = _ops.match_top2(des1, des2)
    return d1.lt(des_thrsh), i1.long()


def nearest_neighbor_distance_ratio_match(des1, des2, kp2, threshold):
    """eval_utils.py:168-175 -> (predict_label bool[Nq], nn_kp2 = kp2[Ia])."""
    d1, d2, i1, _ = _ops.match_top2(des1, des2)
    predict_label = (d1 / d2).lt(threshold)
    nn_kp2 = kp2.index_select(dim=0, index=i1.long().view(-1))
    return predict_label, nn_kp2


def match_top2(des1, des2):
    """(Da, Db, Ia, Ib) = sorted[:,0], sorted[:,1], indices[:,0], indices[:,1] of eval_utils.py:170-171."""
    d1, d2, i1, i2 = _ops.match_top2(des1, des2)
    return d1, d2, i1.long(), i2.long()


def match_topk(des1, des2, k):
    """(D [Nq, k] fp32, I [Nq, k] int64) = sorted[:, :k], indices[:, :k] of eval_utils.py:170-171 for k in [1, 8]: the k nearest
    gallery rows of every query, ascending by (distance, index), exact (hn_match_topk_typed); without the Nq x Ng matrix.
    Rows with fewer than k gallery rows get +inf / -1 in the missing slots."""
    d, i = _ops.match_topk(des1, des2, k)
    return d, i.long()


def match_radius(des1, des2, radius, capacity=None):
    """(row_ptr int64 [Nq + 1], col int64, dist fp32): every pair with d < radius as CSR, exact (hn_match_radius_*_typed) - the
    entries of `distance_matrix_vector(des1, des2).lt(radius).nonzero()` (math_utils.py:8-19) without the Nq x Ng matrix,
    columns ascending within a row; (row_ptr, col) feed torch.sparse_csr_tensor as they are. capacity=None: one host read of the
    total, outputs of exactly that size; capacity=n: no host synchronisation, outputs of n entries, of which the first
    min(n, row_ptr[-1]) are written. radius is used as an fp32 value."""
    row_ptr, col, dist = _ops.match_radius(des1, des2, radius, capacity)
    return row_ptr, col.long(), dist


def threshold_matches(des1, des2, des_thrsh):
    """(pairs [M, 2] int64, dist [M] fp32) with pairs = D.lt(des_thrsh).nonzero() of the reference composition
    (D = distance_matrix_vector(des1, des2); DES_THRSH, config.py:47), in its row-major order: the threshold strategy of
    descriptor evaluation, one host synchronisation."""
    row_ptr, col, dist = match_radius(des1, des2, des_thrsh)
    rows = torch.repeat_interleave(torch.arange(row_ptr.numel() - 1, device=col.device), row_ptr.diff(), output_size=col.numel())
    return torch.stack([rows, col], dim=1), dist


def mutual_nn_ratio(des1, des2, threshold=0.7, return_pairs=True):
    """Mutual nearest neighbours AND the ratio test of BASELINE config 4 in one call:
    (pairs [M,2] int64 or None, mutual bool[Nq], ratio_label bool[Nq], Ia int64[Nq], Da, Db).
    (i, j) is mutual iff j = argmin_j D[i,:] and i = argmin_i D[:,j] - not in the reference; composed from its row / column
    minima (hardnet/Losses.py:105-108, eval_utils.py:24-32); ratio_label = Da / Db < threshold (eval_utils.py:168-175).
    ONE matching GEMM serves both directions (hn_match_mutual: the epilogue's per-cell maxima bound the column side, a small
    exact kernel verifies each column's best claimant). The masks come without any host synchronisation; compacting them into
    the `pairs` list needs its length on the host (return_pairs=False skips it)."""
    d1, d2, fwd, _, mutual = _ops.match_mutual(des1, des2)
    fwd = fwd.long()
    pairs = None
    if return_pairs:
        i = torch.arange(des1.size(0), device=fwd.device)
        pairs = torch.stack([i[mutual], fwd[mutual]], dim=1)
    return pairs, mutual, (d1 / d2).lt(threshold), fwd, d1, d2


def mutual_nn_ratio_two_pass(des1, des2, threshold=0.7, return_pairs=True):
    """The same result from two matching passes (queries x gallery, gallery x queries), operands packed once. Kept as the
    cross-check of the single-GEMM path (tests) and for A/B timing (bench.py)."""
    q16, g16 = _ops.pack_descriptors(des1), _ops.pack_descriptors(des2)
    d1, d2, fwd, _ = _ops.match_top2(des1, des2, q16=q16, g16=g16)
    _, _, bwd, _ = _ops.match_top2(des2, des1, q16=g16, g16=q16)
    fwd, bwd = fwd.long(), bwd.long()
    i = torch.arange(des1.size(0), device=fwd.device)
    mutual = bwd[fwd] == i
    pairs = torch.stack([i[mutual], fwd[mutual]], dim=1) if return_pairs else None
    return pairs, mutual, (d1 / d2).lt(threshold), fwd, d1, d2


def mutual_nearest_neighbors(des1, des2):
    """Mutual NN pairs [M,2]: (i, j) with j = argmin_j D[i,:] and i = argmin_i D[:,j] (see mutual_nn_ratio)."""
    return mutual_nn_ratio(des1, des2)[0]


# ---- many image pairs per call ------------------------------------------------------------------------------------------
# The reference's evaluation matches one image pair at a time (eval_utils.py:85-197). The batched forms take padded batches
# des1 [B, Nq, 128] / des2 [B, Ng, 128] plus optional integer [B] lengths len1 / len2 (valid rows per pair; device tensors keep
# the call free of host synchronisation) and run every pair in one launch sequence (hn_match_batched). Per pair and valid row
# the results equal the per-pair functions on des1[b, :len1[b]], des2[b, :len2[b]]; rows past len1[b], and all rows of a pair
# without gallery rows, get Da = Db = +inf, Ia = Ib = -1 and are never matched.

def match_top2_batched(des1, des2, len1=None, len2=None):
    """match_top2 for every pair of a padded batch -> (Da, Db, Ia, Ib), each [B, Nq]; indices int64, local to the pair."""
    d1, d2, i1, i2 = _ops.match_batched(des1, des2, len1, len2)
    return d1, d2, i1.long(), i2.long()


def mutual_nn_ratio_batched(des1, des2, len1=None, len2=None, threshold=0.7):
    """mutual_nn_ratio for every pair of a padded batch -> (mutual, ratio_label, Ia, Da, Db), all [B, Nq]. No pair list:
    compacting it needs its length on the host; mutual[b].nonzero() gives pair b's query rows."""
    d1, d2, i1, _, mutual = _ops.match_batched(des1, des2, len1, len2, mutual=True)
    return mutual, (d1 / d2).lt(threshold), i1.long(), d1, d2


# ---- pair tables over concatenated descriptor sets -----------------------------------------------------------------------
# Extraction over a set of images yields one [sum N_i, 128] tensor, and the pairs of an evaluation reuse images (a reference
# image against the others of its sequence, or every pair of a collection). The pair forms take those sets as they are: a
# [P, 4] table of (start1, len1, start2, len2) row ranges says which rows of des1 are matched against which rows of des2
# (hn_match_pairs). Each set is packed once per call, or not at all when its packed rows (pack_descriptors) are passed as
# des1_16 / des2_16. Outputs are padded per pair to [P, max_len1]; per pair and valid row they equal the per-pair functions on
# des1[start1:start1 + len1], des2[start2:start2 + len2], with indices local to the gallery range. Rows past len1, and all
# rows of a pair without gallery rows, get Da = Db = +inf, Ia = Ib = -1 and are never matched. A start is clamped to
# [0, rows], a length to [0, min(max_len, rows - start)]. max_len1 / max_len2 = None read the largest clamped lengths from the
# table: one host synchronisation. Passing them (and a table on the device) keeps the call free of host synchronisation and
# CUDA-graph capturable.

def pair_table(counts1, idx1, idx2, counts2=None):
    """[P, 4] int32 table for the pair forms, on the device of counts1: pair p matches image idx1[p] of the first set against
    image idx2[p] of the second. counts1 / counts2: keypoints per image of each set (the sets are the images' descriptors
    concatenated in image order); counts2 = None means both sides index the same set. Starts are the exclusive cumulative
    sums of the counts."""
    c1 = torch.as_tensor(counts1)
    c2 = c1 if counts2 is None else torch.as_tensor(counts2, device=c1.device)
    if c1.dim() != 1 or c2.dim() != 1 or c1.dtype.is_floating_point or c2.dtype.is_floating_point:
        raise ValueError("pair_table: counts must be 1-D integer tensors")
    i1 = torch.as_tensor(idx1, device=c1.device).long()
    i2 = torch.as_tensor(idx2, device=c1.device).long()
    if i1.shape != i2.shape or i1.dim() != 1:
        raise ValueError("pair_table: idx1 and idx2 must be 1-D of the same length")
    c1, c2 = c1.long(), c2.long()
    s1, s2 = torch.cumsum(c1, 0) - c1, torch.cumsum(c2, 0) - c2
    return torch.stack([s1[i1], c1[i1], s2[i2], c2[i2]], dim=1).to(torch.int32)


def _max_lens(pairs, n1, n2, max_len1, max_len2):
    """The per-pair maxima not given, from the table's clamped lengths (one host synchronisation)."""
    if max_len1 is not None and max_len2 is not None:
        return max_len1, max_len2
    t = pairs.long()
    m = []
    for k, n in ((0, n1), (2, n2)):
        start = t[:, k].clamp(0, n)
        m.append(torch.minimum(t[:, k + 1], n - start).clamp(min=0).max() if t.size(0) else t.new_zeros(()))
    m1, m2 = torch.stack(m).tolist()
    return (max(m1, 1) if max_len1 is None else max_len1), (max(m2, 1) if max_len2 is None else max_len2)


def match_top2_pairs(des1, des2, pairs, max_len1=None, max_len2=None, des1_16=None, des2_16=None):
    """match_top2 for every row-range pair of the table -> (Da, Db, Ia, Ib), each [P, max_len1]; indices int64, local to the
    pair's gallery range."""
    max_len1, max_len2 = _max_lens(pairs, des1.size(0), des2.size(0), max_len1, max_len2)
    d1, d2, i1, i2 = _ops.match_pairs(des1, des2, pairs, max_len1, max_len2, des1_16, des2_16)
    return d1, d2, i1.long(), i2.long()


def mutual_nn_ratio_pairs(des1, des2, pairs, max_len1=None, max_len2=None, threshold=0.7, des1_16=None, des2_16=None):
    """mutual_nn_ratio for every row-range pair of the table -> (mutual, ratio_label, Ia, Da, Db), all [P, max_len1]."""
    max_len1, max_len2 = _max_lens(pairs, des1.size(0), des2.size(0), max_len1, max_len2)
    d1, d2, i1, _, mutual = _ops.match_pairs(des1, des2, pairs, max_len1, max_len2, des1_16, des2_16, mutual=True)
    return mutual, (d1 / d2).lt(threshold), i1.long(), d1, d2


def match_topk_pairs(des1, des2, pairs, k, max_len1=None, max_len2=None, des1_16=None, des2_16=None):
    """match_topk for every row-range pair of the table -> (D, I), each [P, max_len1, k]; indices int64, local to the pair's
    gallery range; rows past len1 and pairs without gallery rows get +inf / -1. A padded batch des1 [B, N1, 128],
    des2 [B, N2, 128] with lengths len1 / len2 is the table (b * N1, len1[b], b * N2, len2[b]) over des1.flatten(0, 1) and
    des2.flatten(0, 1), with max_len1 = N1 and max_len2 = N2."""
    max_len1, max_len2 = _max_lens(pairs, des1.size(0), des2.size(0), max_len1, max_len2)
    d, i = _ops.match_pairs_topk(des1, des2, pairs, k, max_len1, max_len2, des1_16, des2_16)
    return d, i.long()


def match_radius_pairs(des1, des2, pairs, radius, max_len1=None, max_len2=None, capacity=None, des1_16=None, des2_16=None):
    """match_radius for every row-range pair of the table -> (row_ptr int64 [P * max_len1 + 1], col int64, dist fp32) over the
    padded rows (row r of pair p at p * max_len1 + r); columns local to the pair's gallery range; rows past len1 and pairs
    without gallery rows have no entries. With max_len1, max_len2 and capacity given (and the table on the device) the call is
    free of host synchronisation and CUDA-graph capturable."""
    max_len1, max_len2 = _max_lens(pairs, des1.size(0), des2.size(0), max_len1, max_len2)
    row_ptr, col, dist = _ops.match_pairs_radius(des1, des2, pairs, radius, max_len1, max_len2, capacity, des1_16, des2_16)
    return row_ptr, col.long(), dist


# ---- match-score counters (FDLNet-master/utils/eval_utils.py:112-197) -----------------------------------------------
# The callers right behind the hot path in the reference's evaluation: nearest neighbour (or ratio test) on the fused
# kernel, then "is the matched keypoint within COO_THRSH pixels of the warped keypoint" and two counters. The reference
# builds an Nq x Nq coordinate distance matrix and takes its diagonal; the same expression is evaluated row-wise here.

def _keypoint_distance(kp1w, nn_kp2):
    """diag(pairwise_distances(kp1w[..., 1:3], nn_kp2[..., 1:3])) of math_utils.py:22-40: sqrt(clamp(|x|^2 + |y|^2 - 2 x.y, 1e-8)),
    over the last keypoint dimension (one pair [N, >=3] or a batch of pairs [B, N, >=3])."""
    x, y = kp1w[..., 1:3].float(), nn_kp2[..., 1:3].float()
    sq = (x * x).sum(-1) + (y * y).sum(-1) - 2.0 * (x * y).sum(-1)
    return torch.sqrt(sq.clamp(min=1e-8))


def _counts(predict_label, kp1w, nn_kp2, visible, coo_thrsh, predicted):
    """(correct, max(#predicted, 1)) as device tensors, counted over the last dimension (per pair)."""
    correspondences = _keypoint_distance(kp1w, nn_kp2).le(coo_thrsh) & visible.bool()
    return (predict_label & correspondences).sum(-1), predicted.sum(-1).clamp(min=1)


def _score(predict_label, kp1w, nn_kp2, visible, coo_thrsh, predicted):
    correct, predict = _counts(predict_label, kp1w, nn_kp2, visible, coo_thrsh, predicted)
    return correct.item(), predict.item()


def nearest_neighbor_match_score(des1, des2, kp1w, kp2, visible, COO_THRSH):
    """eval_utils.py:112-127 -> (correct_matches, predict_matches = max(#visible, 1))."""
    _, nn_idx = nearest_neighbor_match(des1, des2)
    vis = visible.bool()
    return _score(vis, kp1w, kp2.index_select(0, nn_idx), vis, COO_THRSH, vis)


def nearest_neighbor_threshold_match_score(des1, des2, kp1w, kp2, visible, DES_THRSH, COO_THRSH):
    """eval_utils.py:130-150 -> (correct_matches, predict_matches = max(#(nn_value < DES_THRSH and visible), 1))."""
    label, nn_idx = nearest_neighbor_threshold_match(des1, des2, DES_THRSH)
    predict = label & visible.bool()
    return _score(predict, kp1w, kp2.index_select(0, nn_idx), visible, COO_THRSH, predict)


def nearest_neighbor_distance_ratio_match_score(des1, des2, kp1w, kp2, visible, COO_THRSH, threshold=0.7):
    """eval_utils.py:178-197 -> (correct_matches, predict_matches = max(#(Da / Db < threshold and visible), 1))."""
    label, nn_kp2 = nearest_neighbor_distance_ratio_match(des1, des2, kp2, threshold)
    predict = label & visible.bool()
    return _score(predict, kp1w, nn_kp2, visible, COO_THRSH, predict)


# Batched counters: kp1w [B, Nq, >=3], kp2 [B, Ng, >=3], visible [B, Nq] are the per-pair arguments with a batch dimension;
# each returns (correct [B], predicted [B]) int64 device tensors, without host synchronisation. A row without a match (past
# len1, or in a pair without gallery rows) is neither predicted nor correct.

def _batched_nn_kp2(kp2, ia):
    """kp2[b, Ia[b, i]] for every pair; rows without a match (Ia = -1) read row 0 and are masked by the caller."""
    return torch.gather(kp2, 1, ia.clamp(min=0).unsqueeze(-1).expand(-1, -1, kp2.size(-1)))


def nearest_neighbor_match_score_batched(des1, des2, kp1w, kp2, visible, COO_THRSH, len1=None, len2=None):
    """nearest_neighbor_match_score per pair -> (correct [B], predicted = max(#visible, 1) [B])."""
    _, _, ia, _ = match_top2_batched(des1, des2, len1, len2)
    vis = visible.bool() & (ia >= 0)
    return _counts(vis, kp1w, _batched_nn_kp2(kp2, ia), vis, COO_THRSH, vis)


def nearest_neighbor_threshold_match_score_batched(des1, des2, kp1w, kp2, visible, DES_THRSH, COO_THRSH, len1=None, len2=None):
    """nearest_neighbor_threshold_match_score per pair -> (correct [B], predicted = max(#(Da < DES_THRSH and visible), 1) [B])."""
    da, _, ia, _ = match_top2_batched(des1, des2, len1, len2)
    predict = da.lt(DES_THRSH) & visible.bool() & (ia >= 0)
    return _counts(predict, kp1w, _batched_nn_kp2(kp2, ia), visible, COO_THRSH, predict)


def nearest_neighbor_distance_ratio_match_score_batched(des1, des2, kp1w, kp2, visible, COO_THRSH, threshold=0.7, len1=None,
                                                        len2=None):
    """nearest_neighbor_distance_ratio_match_score per pair -> (correct [B], predicted = max(#(Da / Db < threshold and
    visible), 1) [B])."""
    da, db, ia, _ = match_top2_batched(des1, des2, len1, len2)
    predict = (da / db).lt(threshold) & visible.bool() & (ia >= 0)
    return _counts(predict, kp1w, _batched_nn_kp2(kp2, ia), visible, COO_THRSH, predict)


# Pair-table counters: kp1w [P, max_len1, >=3] (each pair's query keypoints warped by its homography) and visible [P, max_len1]
# are padded per pair, and max_len1 is their second dimension; kp2 [Ng_rows, >=3] holds the keypoints of the concatenated
# gallery set, read at row g_start + Ia. Each returns (correct [P], predicted [P]) int64 device tensors; a row without a match
# is neither predicted nor correct.

def _pairs_nn_kp2(kp2, pairs, ia):
    """kp2[g_start + Ia] for every pair and row; rows without a match (Ia = -1) read a valid row and are masked by the caller."""
    n = kp2.size(0)
    start = pairs.to(device=ia.device, dtype=torch.long)[:, 2].clamp(0, n)
    rows = (start.unsqueeze(1) + ia.clamp(min=0)).clamp(max=max(n - 1, 0))
    return kp2[rows]


def nearest_neighbor_match_score_pairs(des1, des2, pairs, kp1w, kp2, visible, COO_THRSH, max_len2=None, des1_16=None,
                                       des2_16=None):
    """nearest_neighbor_match_score per table pair -> (correct [P], predicted = max(#visible, 1) [P])."""
    _, _, ia, _ = match_top2_pairs(des1, des2, pairs, kp1w.size(1), max_len2, des1_16, des2_16)
    vis = visible.bool() & (ia >= 0)
    return _counts(vis, kp1w, _pairs_nn_kp2(kp2, pairs, ia), vis, COO_THRSH, vis)


def nearest_neighbor_threshold_match_score_pairs(des1, des2, pairs, kp1w, kp2, visible, DES_THRSH, COO_THRSH, max_len2=None,
                                                 des1_16=None, des2_16=None):
    """nearest_neighbor_threshold_match_score per table pair -> (correct [P], predicted = max(#(Da < DES_THRSH and visible), 1)
    [P])."""
    da, _, ia, _ = match_top2_pairs(des1, des2, pairs, kp1w.size(1), max_len2, des1_16, des2_16)
    predict = da.lt(DES_THRSH) & visible.bool() & (ia >= 0)
    return _counts(predict, kp1w, _pairs_nn_kp2(kp2, pairs, ia), visible, COO_THRSH, predict)


def nearest_neighbor_distance_ratio_match_score_pairs(des1, des2, pairs, kp1w, kp2, visible, COO_THRSH, threshold=0.7,
                                                      max_len2=None, des1_16=None, des2_16=None):
    """nearest_neighbor_distance_ratio_match_score per table pair -> (correct [P], predicted = max(#(Da / Db < threshold and
    visible), 1) [P])."""
    da, db, ia, _ = match_top2_pairs(des1, des2, pairs, kp1w.size(1), max_len2, des1_16, des2_16)
    predict = (da / db).lt(threshold) & visible.bool() & (ia >= 0)
    return _counts(predict, kp1w, _pairs_nn_kp2(kp2, pairs, ia), visible, COO_THRSH, predict)

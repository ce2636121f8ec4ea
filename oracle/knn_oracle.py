"""CPU / float64 restatement of k-nearest-neighbour matching — test infrastructure only.

The first k columns of the full row sort of FDLNet-master/utils/eval_utils.py:168-171 (`sorted, indices = D.sort(dim=-1)`),
with the distance form of oracle/losses_oracle.py (FDLNet-master/utils/math_utils.py:8-19).
"""
from __future__ import annotations

import torch

from oracle.losses_oracle import distance_matrix_vector_fdl


def knn_match(des1, des2, k: int, chunk: int = 2048):
    """sorted[:, :k], indices[:, :k] in float64, evaluated in query-row chunks like losses_oracle.ratio_match:
    (D [Nq, k] float64, I [Nq, k] int64), ascending by (distance, index) (stable sort). Rows with fewer than k gallery rows
    are padded with +inf / -1."""
    vals, idxs = [], []
    for s in range(0, des1.size(0), chunk):
        d = distance_matrix_vector_fdl(des1[s:s + chunk].double(), des2.double())
        v, i = torch.sort(d, dim=-1, stable=True)
        vals.append(v[:, :k])
        idxs.append(i[:, :k])
    v, i = torch.cat(vals), torch.cat(idxs)
    if v.size(1) < k:
        pad = k - v.size(1)
        v = torch.cat([v, v.new_full((v.size(0), pad), float("inf"))], 1)
        i = torch.cat([i, i.new_full((i.size(0), pad), -1)], 1)
    return v, i

"""CPU / float64 restatement of radius matching — test infrastructure only.

`D.lt(r).nonzero()` of the reference composition, D = distance_matrix_vector(des1, des2) (FDLNet-master/utils/math_utils.py:8-19,
oracle/losses_oracle.py), as CSR.
"""
from __future__ import annotations

import torch

from oracle.losses_oracle import distance_matrix_vector_fdl


def radius_match(des1, des2, r: float, chunk: int = 2048):
    """(row_ptr [Nq + 1] int64, col int64, dist float64): the entries of D.lt(r) in float64, evaluated in query-row chunks like
    losses_oracle.ratio_match, in the row-major order of nonzero()."""
    counts, cols, dists = [], [], []
    for s in range(0, des1.size(0), chunk):
        d = distance_matrix_vector_fdl(des1[s:s + chunk].double(), des2.double())
        nz = d.lt(r).nonzero()
        counts.append(torch.bincount(nz[:, 0], minlength=d.size(0)))
        cols.append(nz[:, 1])
        dists.append(d[nz[:, 0], nz[:, 1]])
    row_ptr = torch.zeros(des1.size(0) + 1, dtype=torch.int64)
    if counts:
        row_ptr[1:] = torch.cumsum(torch.cat(counts), 0)
    empty_col, empty_d = torch.zeros(0, dtype=torch.int64), torch.zeros(0, dtype=torch.float64)
    return row_ptr, torch.cat(cols) if cols else empty_col, torch.cat(dists) if dists else empty_d

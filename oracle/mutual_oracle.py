"""Float64 restatement of mutual nearest-neighbour matching — test infrastructure only.

One pass over query-row chunks computes both directions of losses_oracle.mutual_nn (D.min(1) and D.min(0) of the FDLNet
distance matrix, FDLNet-master/utils/math_utils.py:8-19). The column side is kept as a running minimum over the chunks, the
way sharded matching reduces it over the ranks' query rows.
"""
from __future__ import annotations

import torch

from oracle.losses_oracle import distance_matrix_vector_fdl


def _first_argmin(d: torch.Tensor, dim: int):
    """(min, lowest index attaining it) along dim: ties resolved explicitly rather than by torch.min's kernel."""
    v = d.min(dim=dim).values
    idx = torch.arange(d.size(dim), device=d.device).view((-1, 1) if dim == 0 else (1, -1))
    big = torch.iinfo(torch.int64).max
    arg = torch.where(d == v.unsqueeze(dim), idx, torch.full_like(idx, big)).min(dim=dim).values
    return v, arg


def mutual_match(des1, des2, chunk: int = 2048):
    """(fwd, col_min, col_arg, mutual) in float64 on the inputs' device:
    fwd int64 [Nq]: nearest gallery row of every query, lowest index on ties;
    col_min float64 [Ng], col_arg int64 [Ng]: nearest query row of every gallery row, lowest row on ties (a later chunk
    replaces the running minimum only where it is strictly smaller);
    mutual bool [Nq]: col_arg[fwd[i]] == i."""
    g = des2.double()
    ng = g.size(0)
    col_min = torch.full((ng,), float("inf"), dtype=torch.float64, device=g.device)
    col_arg = torch.full((ng,), -1, dtype=torch.int64, device=g.device)
    fwd = []
    for s in range(0, des1.size(0), chunk):
        d = distance_matrix_vector_fdl(des1[s:s + chunk].double(), g)
        fwd.append(_first_argmin(d, 1)[1])
        v, a = _first_argmin(d, 0)
        better = v < col_min
        col_min = torch.where(better, v, col_min)
        col_arg = torch.where(better, a + s, col_arg)
    fwd = torch.cat(fwd)
    mutual = col_arg[fwd] == torch.arange(fwd.numel(), device=fwd.device)
    return fwd, col_min, col_arg, mutual

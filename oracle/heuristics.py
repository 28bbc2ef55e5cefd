"""CPU restatement of the common-neighbour link heuristics (plnlp_b200/heuristics.py, csrc/heuristic.cu).

Rules restated here:
  * N(u) = the set of distinct column ids of stored row u of the adjacency, without u itself (values ignored);
    d(w) = |N(w)|;
  * CN(u, v) = |N(u) & N(v)|;
  * AA(u, v) = sum over w in N(u) & N(v) of 1 / ln d(w), a term with d(w) < 2 contributing 0;
  * RA(u, v) = sum over w in N(u) & N(v) of 1 / d(w), a term with d(w) = 0 (possible only when the adjacency is
    not symmetric) contributing 0;
  * the terms are fp64, summed exactly (math.fsum) and rounded to fp32 once.
"""
import math

import numpy as np
import torch


def neighbour_sets(rowptr, col, n_rows):
    """[set of int] per row: the distinct column ids of each stored row of a CSR, the diagonal dropped"""
    rowptr = torch.as_tensor(rowptr).tolist()
    col = torch.as_tensor(col).tolist()
    return [set(col[rowptr[u]:rowptr[u + 1]]) - {u} for u in range(n_rows)]


def term(method, d):
    """the fp64 term a common neighbour of degree d adds"""
    if method == "CN":
        return 1.0
    if method == "AA":
        return 1.0 / math.log(d) if d >= 2 else 0.0
    if method == "RA":
        return 1.0 / d if d >= 1 else 0.0
    raise ValueError(method)


def score_sets(sets, edges, method, keep=None):
    """fp64 exact sums (before the fp32 rounding) of the pairs edges [P, 2]; ``keep(w)``: count only the common
    neighbours w it accepts (a shard's block of intermediate nodes)"""
    out = []
    for u, v in torch.as_tensor(edges).reshape(-1, 2).tolist():
        common = sets[u] & sets[v]
        out.append(math.fsum(term(method, len(sets[w])) for w in sorted(common) if keep is None or keep(w)))
    return np.array(out, dtype=np.float64)


def score(rowptr, col, n_rows, edges, method):
    """fp32 [P] tensor: the heuristic of every pair, each exact sum rounded to fp32 once"""
    return torch.from_numpy(score_sets(neighbour_sets(rowptr, col, n_rows), edges, method).astype(np.float32))

"""CPU restatement of the NCN predictor (plnlp_b200/layer.py NCNPredictor, heuristics.common_neighbour_lists).

Rules restated here:
  * N(u) as in oracle/heuristics.py (distinct columns of stored row u without u; values ignored); a negative id has
    an empty N;
  * C(u, v) = N(u) & N(v) in ascending id order;
  * c_uv = sum over w in C(u, v) of h_w;
  * the score is the MLP of MLPPredictor on [h_u * h_v | c_uv]: Linear(2H, hidden), relu, ..., Linear(-> 1), with
    relu after every Linear but the last (no dropout here).

``lists`` builds C from Python sets; ``dense_lists`` gives the same from a dense 0/1 restatement (row p of the
matrix A[u] * A[v]), so the two rules check each other.  ``score`` is fp64 torch with autograd.
"""
import math

import torch

from oracle import plnlp_ref
from oracle.heuristics import neighbour_sets


def lists(sets, edges):
    """(rowptr int64 [P + 1], col int64): C(u, v) of every pair, from Python sets"""
    rowptr, col = [0], []
    for u, v in torch.as_tensor(edges).reshape(-1, 2).tolist():
        common = sorted(sets[u] & sets[v]) if u >= 0 and v >= 0 else []
        col += common
        rowptr.append(len(col))
    return torch.tensor(rowptr, dtype=torch.int64), torch.tensor(col, dtype=torch.int64)


def dense_lists(sets, edges):
    """the same lists from the dense 0/1 matrix A (A[u, w] = 1 for w in N(u)): the nonzeros of A[u] * A[v]"""
    n = len(sets)
    A = torch.zeros(n + 1, n, dtype=torch.int64)         # row n: the empty row of a negative id
    for u, s in enumerate(sets):
        A[u, list(s)] = 1
    e = torch.as_tensor(edges).reshape(-1, 2)
    e = torch.where(e < 0, torch.full_like(e, n), e)
    M = A[e[:, 0]] * A[e[:, 1]]
    rowptr = torch.zeros(e.size(0) + 1, dtype=torch.int64)
    rowptr[1:] = torch.cumsum(M.sum(1), 0)
    return rowptr, M.nonzero()[:, 1]


def sets_of(adj):
    rowptr, col, _ = adj.csr()
    return neighbour_sets(rowptr.cpu(), col.cpu(), adj.size(0))


def cn_sum(h, cn):
    """c [P, H]: the sum of h[w] over each list (fp64 when h is)"""
    rowptr, col = (t.cpu() for t in cn)
    P = rowptr.numel() - 1
    row = torch.repeat_interleave(torch.arange(P), rowptr[1:] - rowptr[:-1])
    return torch.zeros(P, h.size(1), dtype=h.dtype).index_add_(0, row, h[col])


def score(h, edges, cn, lins):
    """fp64 [P]: the NCN head, ``lins`` = [(W, b), ...] with W_0 [hidden, 2H]; -1 reads the last row of h"""
    e = torch.as_tensor(edges).reshape(-1, 2).cpu()
    x = torch.cat([h[e[:, 0]] * h[e[:, 1]], cn_sum(h, cn)], 1)
    for W, b in lins[:-1]:
        x = torch.relu(x @ W.t() + b)
    W, b = lins[-1]
    return (x @ W.t() + b).reshape(-1)


class OracleNCNModel(plnlp_ref.OracleModel):
    """``plnlp_ref.OracleModel`` with the NCN head: pred.{i}.weight / .bias, pred.0.weight [hidden, 2H], and the
    common-neighbour lists of every scored batch taken from ``sets``"""

    def __init__(self, sets, **kw):
        mlp_layers, hidden = kw["mlp_layers"], kw["mlp_hidden"]
        dtype = kw.get("dtype", torch.float32)
        super().__init__(**dict(kw, predictor="DOT"))
        self.pred_kind, self.mlp_layers, self.sets = "NCN", mlp_layers, sets
        g = torch.Generator().manual_seed(99)
        for i in range(mlp_layers):
            fi = 2 * hidden if i == 0 else hidden
            fo = 1 if i == mlp_layers - 1 else hidden
            b = 1.0 / math.sqrt(fi)
            self.params[f"pred.{i}.weight"] = ((torch.rand(fo, fi, generator=g) * 2 - 1) * b).to(dtype).requires_grad_()
            self.params[f"pred.{i}.bias"] = ((torch.rand(fo, generator=g) * 2 - 1) * b).to(dtype).requires_grad_()
        self._make_optimizer()

    def score(self, h, edges, keep_masks=None):
        lins = [(self.params[f"pred.{i}.weight"], self.params[f"pred.{i}.bias"]) for i in range(self.mlp_layers)]
        return score(h, edges, lists(self.sets, edges), lins)

"""CPU restatement of candidate sets (the ``candidates`` argument of plnlp_b200/recommend.py and the candidate-set
entry points of csrc/topk.cu), in the rules of oracle/ranking.py.

Rule: with a candidate set C, every pair (nodes[q], j) with j not in C is one more known link of the query.
  * recommend: the k best of the row masked with the known links, the query itself and every node outside C;
  * rank: the filtered rank with that same exclusion; the target is never excluded, so it is ranked among
    C + {target}, whether it is in C or not;
  * an empty C leaves no candidate: rows of (-1, -inf), rank 1.
``complement_exclusion`` builds that exclusion as a CSR for oracle.ranking; ``mask_candidates`` applies the same
rule directly to a score row."""
import torch

from oracle import ranking


def complement_exclusion(nodes, candidates, n, rowptr=None, col=None):
    """(rowptr int64 [n + 1], col int32): the known links of the CSR (rowptr, col) plus, for every query node, every
    node j in [0, n) outside ``candidates``"""
    inside = torch.zeros(n, dtype=torch.bool)
    inside[torch.as_tensor(candidates, dtype=torch.int64)] = True
    outside = torch.nonzero(~inside).reshape(-1).tolist()
    queries = set(torch.as_tensor(nodes).tolist())
    out_ptr, out_col = [0], []
    for r in range(n):
        row = [] if rowptr is None else torch.as_tensor(col[int(rowptr[r]):int(rowptr[r + 1])]).tolist()
        if r in queries:
            row = row + outside
        out_col += row
        out_ptr.append(len(out_col))
    return torch.tensor(out_ptr, dtype=torch.int64), torch.tensor(out_col, dtype=torch.int32)


def mask_candidates(s, nodes, candidates, rowptr=None, col=None, exclude_self=True):
    """copy of s [Q, N] masked as oracle.ranking.mask_scores, and every column outside ``candidates`` set to -inf"""
    s = ranking.mask_scores(s, nodes, rowptr, col, exclude_self)
    inside = torch.zeros(s.size(1), dtype=torch.bool)
    inside[torch.as_tensor(candidates, dtype=torch.int64)] = True
    s[:, ~inside] = float("-inf")
    return s


def filtered_ranks(S, targets, nodes, candidates, rowptr=None, col=None, exclude_self=True):
    """1 + (gt + ge) / 2 of each target among ``candidates`` and the target, on full score rows S [P, N]: the target
    score is read before masking, so the target is never excluded"""
    t = torch.as_tensor(targets)
    ts = S[torch.arange(S.size(0)), t]
    gt, ge = ranking.rank_counts(mask_candidates(S, nodes, candidates, rowptr, col, exclude_self), t, ts)
    return 1.0 + 0.5 * (gt.double() + ge.double())

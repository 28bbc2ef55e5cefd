"""CPU checks of candidate sets (-m "not gpu"): the rule of tests/ranking_candidates.py against the complement
exclusion through oracle/ranking.py and against brute force, the candidate-set argument checks of
plnlp_b200/recommend.py, and the per-shard slices of a candidate set."""
import math

import pytest
import torch

from oracle import ranking
from tests import ranking_candidates as rc

NAN, INF = float("nan"), float("inf")


def _brute(s, nodes, cand, links, exclude_self, k, targets):
    """per row: the top-k (ids, scores) and the filtered rank of the target, by plain loops over the candidates"""
    ids, scores, ranks = [], [], []
    for q, n in enumerate(nodes):
        row = s[q].tolist()
        allowed = [j for j in sorted(set(cand)) if j not in links.get(n, ()) and not (exclude_self and j == n)]
        live = [(0.0 if row[j] == 0 else row[j], j) for j in allowed if math.isfinite(row[j])]
        live.sort(key=lambda x: (-x[0], x[1]))
        top = live[:k]
        ids.append([j for _, j in top] + [-1] * (k - len(top)))
        scores.append([v for v, _ in top] + [-INF] * (k - len(top)))
        t = targets[q]
        ts = row[t]
        others = [row[j] for j in allowed if j != t and math.isfinite(row[j])]
        gt, ge = sum(v > ts for v in others), sum(v >= ts for v in others)
        ranks.append(1.0 + 0.5 * (gt + ge))
    return torch.tensor(ids), torch.tensor(scores), torch.tensor(ranks, dtype=torch.float64)


def _case(kind, Q, N, g):
    if kind == "ties":                                      # few distinct values: ties across non-adjacent ids
        s = torch.randint(-2, 3, (Q, N), generator=g).float()
    else:
        s = torch.randn(Q, N, generator=g)
    if kind == "special":
        r = torch.rand(Q, N, generator=g)
        s[r < 0.2] = -INF
        s[(r >= 0.2) & (r < 0.35)] = NAN
        s[(r >= 0.35) & (r < 0.4)] = INF
        s[(r >= 0.4) & (r < 0.45)] = -0.0
    return s


@pytest.mark.parametrize("kind", ["normal", "ties", "special"])
@pytest.mark.parametrize("n_cand", [0, 1, 7, 30, 60])
@pytest.mark.parametrize("exclude_self", [True, False])
def test_candidate_rule_equals_complement_exclusion_and_brute_force(kind, n_cand, exclude_self):
    g = torch.Generator().manual_seed(n_cand * 10 + len(kind))
    Q, N, k = 9, 60, 12
    s = _case(kind, Q, N, g)
    nodes = torch.randint(0, N, (Q,), generator=g)
    nodes[1] = nodes[0]                                     # a repeated query
    cand = torch.randperm(N, generator=g)[:n_cand]
    cand = torch.cat([cand, cand[:3]])                      # duplicates and any order: a set
    targets = torch.randint(0, N, (Q,), generator=g)
    if n_cand:
        targets[2] = cand[0]                                 # a target in C
        nodes[3] = cand[0]                                   # a query in C
    cset = set(cand.tolist())
    outside = [j for j in range(N) if j not in cset]
    if outside:
        targets[4] = outside[0]                              # a target outside C
        nodes[5] = outside[-1]                               # a query outside C
    targets[6] = nodes[6]                                    # the query itself as target
    links = {int(n): torch.randint(0, N, (6,), generator=g).tolist() for n in nodes[::2]}
    if n_cand:
        links[int(nodes[2])] = links.get(int(nodes[2]), []) + [int(targets[2])]     # a known link as target
    rowptr, col = [0], []
    for r in range(N):
        col += links.get(r, [])
        rowptr.append(len(col))
    rowptr, col = torch.tensor(rowptr), torch.tensor(col, dtype=torch.int32)

    b_ids, b_sc, b_rank = _brute(s, nodes.tolist(), cand.tolist(), links, exclude_self, k, targets.tolist())
    c_ptr, c_col = rc.complement_exclusion(nodes, cand, N, rowptr, col)
    via_exclusion = ranking.mask_scores(s, nodes, c_ptr, c_col, exclude_self)
    via_rule = rc.mask_candidates(s, nodes, cand, rowptr, col, exclude_self)
    assert torch.equal(via_exclusion.isnan(), via_rule.isnan())
    assert torch.equal(via_exclusion.nan_to_num(), via_rule.nan_to_num())
    for masked in (via_exclusion, via_rule):
        ids, sc = ranking.topk_rows(masked, k)
        assert torch.equal(ids, b_ids) and torch.equal(sc, b_sc)
    assert torch.equal(ranking.filtered_ranks(s, targets, nodes, c_ptr, c_col, exclude_self), b_rank)
    assert torch.equal(rc.filtered_ranks(s, targets, nodes, cand, rowptr, col, exclude_self), b_rank)
    if n_cand == 0:
        assert (b_ids == -1).all() and (b_rank == 1).all()
    if n_cand == N:                                          # C = every node: the rule changes nothing
        full_ids, full_sc = ranking.topk_rows(ranking.mask_scores(s, nodes, rowptr, col, exclude_self), k)
        assert torch.equal(full_ids, b_ids) and torch.equal(full_sc, b_sc)


def test_candidate_set_argument_checks():
    from plnlp_b200 import recommend
    c = recommend.candidate_set(torch.tensor([5, 1, 5, 3, 0]), 6, "cpu")
    assert c.tolist() == [0, 1, 3, 5]
    assert recommend.candidate_set(None, 6, "cpu") is None
    assert recommend.candidate_set(torch.zeros(0, dtype=torch.int64), 6, "cpu").numel() == 0
    for bad in (torch.tensor([1, 2], dtype=torch.int32), torch.tensor([1.0]), torch.tensor([[1, 2]]),
                torch.tensor(3), torch.tensor([0, 6]), torch.tensor([-1, 2])):
        with pytest.raises(ValueError):
            recommend.candidate_set(bad, 6, "cpu")


def _splits(N):
    from plnlp_b200 import parallel
    out = [[parallel.row_block(N, r, R) for r in range(R)] for R in (1, 2, 3, 4, 8)]
    a, b = N // 3, N // 3 + 1
    out.append([(0, a), (a, a), (a, b), (b, N)])
    return out


@pytest.mark.parametrize("N", [9, 200, 1001])
def test_candidate_slices_cover_the_set_once(N):
    from plnlp_b200 import recommend
    g = torch.Generator().manual_seed(N)
    for m in (0, 1, 5, N // 2, N):
        cand = torch.unique(torch.randperm(N, generator=g)[:m])
        if m == 5:
            cand = torch.arange(N // 3, N // 3 + 5).clamp_max(N - 1).unique()     # all in one or two blocks
        for bounds in _splits(N):
            sl = recommend.candidate_slices(cand, bounds)
            assert len(sl) == len(bounds)
            got = []
            for (lo, hi), (a, b) in zip(bounds, sl):
                part = cand[a:b]
                assert ((part >= lo) & (part < hi)).all()
                assert part.numel() == int(((cand >= lo) & (cand < hi)).sum())
                got += part.tolist()
            assert got == cand.tolist(), (N, m, bounds)

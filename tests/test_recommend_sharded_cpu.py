"""CPU checks of candidate-sharded link recommendation (-m "not gpu"): the cross-shard merge of the oracle
(tests/ranking_merge.py) against the top-k of the whole row and brute force, and the per-shard known-link CSR
(plnlp_b200/recommend.shard_exclude_csr) against the whole graph's."""
import math

import pytest
import torch

from oracle import ranking
from tests.ranking_merge import merge_topk

NAN, INF = float("nan"), float("inf")


def _brute_topk(row, k):
    cand = [(0.0 if v == 0 else v, j) for j, v in enumerate(row) if math.isfinite(v)]
    cand.sort(key=lambda t: (-t[0], t[1]))
    cand = cand[:k]
    return [j for _, j in cand] + [-1] * (k - len(cand)), [v for v, _ in cand] + [-INF] * (k - len(cand))


def _rows(kind, Q, N, g):
    if kind == "normal":
        return torch.randn(Q, N, generator=g)
    if kind == "ties":                                      # few distinct values: ties across every block
        return torch.randint(-2, 3, (Q, N), generator=g).float()
    if kind == "signed_zero":
        s = torch.zeros(Q, N)
        s[:, 1::3] = -0.0
        s[:, ::7] = 1.0
        return s
    s = torch.randn(Q, N, generator=g)                      # "special": -inf / NaN / +inf, one row all dead
    r = torch.rand(Q, N, generator=g)
    s[r < 0.25] = -INF
    s[(r >= 0.25) & (r < 0.4)] = NAN
    s[(r >= 0.4) & (r < 0.45)] = INF
    s[(r >= 0.45) & (r < 0.5)] = -0.0
    s[0] = NAN
    return s


def _block_lists(s, bounds, k):
    """per block [lo, hi): the oracle's top-k of the column slice, with global ids -> [R, Q, k]"""
    Q = s.size(0)
    ids, sc = [], []
    for lo, hi in bounds:
        if hi == lo:
            i, v = torch.full((Q, k), -1, dtype=torch.int64), torch.full((Q, k), -INF)
        else:
            i, v = ranking.topk_rows(s[:, lo:hi], k)
            i = torch.where(i >= 0, i + lo, i)
        ids.append(i)
        sc.append(v)
    return torch.stack(ids), torch.stack(sc)


def _splits(N):
    """row_block partitions for R = 1 ... 4 and an uneven split with an empty block"""
    from plnlp_b200 import parallel
    out = [[parallel.row_block(N, r, R) for r in range(R)] for R in (1, 2, 3, 4)]
    a, b = N // 3, N // 3 + 1
    out.append([(0, a), (a, a), (a, b), (b, N)])
    return out


@pytest.mark.parametrize("kind", ["normal", "ties", "signed_zero", "special"])
@pytest.mark.parametrize("N,k", [(5, 3), (9, 20), (40, 7), (257, 100), (300, 1)])
def test_merge_of_block_topk_equals_topk_of_the_row(kind, N, k):
    g = torch.Generator().manual_seed(N * 7 + k)
    s = _rows(kind, 5, N, g)
    want_i, want_s = ranking.topk_rows(s, k)
    for q in range(s.size(0)):
        bi, bs = _brute_topk(s[q].tolist(), k)
        assert want_i[q].tolist() == bi and torch.equal(want_s[q], torch.tensor(bs))
    for bounds in _splits(N):
        ids, sc = merge_topk(*_block_lists(s, bounds, k), k)
        assert torch.equal(ids, want_i), (kind, N, k, bounds)
        assert torch.equal(sc, want_s), (kind, N, k, bounds)
        assert all(not (v == 0 and math.copysign(1.0, v) < 0) for v in sc.reshape(-1).tolist())


def test_merge_drops_dead_entries():
    ids = torch.tensor([[[3, -1, 7]], [[-1, -1, -1]], [[2, 5, -1]]])
    sc = torch.tensor([[[1.0, 9.0, NAN]], [[5.0, 5.0, 5.0]], [[1.0, -0.0, -INF]]])
    i, v = merge_topk(ids, sc, 4)
    assert i.tolist() == [[2, 3, 5, -1]]
    assert v.tolist() == [[1.0, 1.0, 0.0, -INF]]


def _graph(n, symmetric, seed):
    from plnlp_b200.graph import CSRGraph
    g = torch.Generator().manual_seed(seed)
    E = 6 * n
    src, dst = torch.randint(0, n, (E,), generator=g), torch.randint(0, n // 2 + 1, (E,), generator=g)
    if symmetric:
        src, dst = torch.cat([src, dst]), torch.cat([dst, src])
    key = torch.unique(src * n + dst)                        # distinct entries, sorted by row
    row, col = key // n, key % n
    rowptr = torch.zeros(n + 1, dtype=torch.int64)
    rowptr[1:] = torch.cumsum(torch.bincount(row, minlength=n), 0)
    return CSRGraph(rowptr, col, None, (n, n)), set(zip(row.tolist(), col.tolist()))


def _pairs_of(rowptr, col, lo, hi):
    out = set()
    for q in range(rowptr.numel() - 1):
        for c in col[int(rowptr[q]):int(rowptr[q + 1])].tolist():
            assert lo <= c < hi
            out.add((q, c))
    return out


@pytest.mark.parametrize("symmetric", [True, False])
@pytest.mark.parametrize("n", [9, 200])
def test_shard_exclude_csr_union_is_the_whole_graph(symmetric, n):
    from plnlp_b200 import parallel, recommend
    from plnlp_b200.graph import CSRGraph
    adj, entries = _graph(n, symmetric, seed=n)
    g = torch.Generator().manual_seed(1)
    edges = torch.stack([torch.randint(0, n, (5 * n,), generator=g), torch.randint(0, n, (5 * n,), generator=g)], 1)
    edge_set = set(map(tuple, edges.tolist()))
    for R in (1, 2, 3, 4):
        got_adj, got_edges = set(), set()
        for r in range(R):
            lo, hi = parallel.row_block(n, r, R)
            sadj = parallel.shard_graph(adj, r, R, CSRGraph)
            assert sadj.symmetric == symmetric
            rowptr, col = recommend.shard_exclude_csr("adj", lo, hi, n, sadj.local_t)
            assert rowptr.dtype == torch.int64 and col.dtype == torch.int32 and rowptr.numel() == n + 1
            part = _pairs_of(rowptr, col, lo, hi)
            assert not part & got_adj
            got_adj |= part
            rowptr, col = recommend.shard_exclude_csr(edges, lo, hi, n)
            got_edges |= _pairs_of(rowptr, col, lo, hi)
        assert got_adj == entries, (R, symmetric)
        assert got_edges == edge_set, R
        if n == 9 and R == 4:
            assert parallel.row_block(n, 3, 4) == (9, 9)     # the empty shard took part
    assert recommend.shard_exclude_csr(None, 0, n, n) == (None, None)

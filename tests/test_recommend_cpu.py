"""CPU checks of link recommendation over all nodes (-m "not gpu"): the oracle restatement (oracle/ranking.py) against
brute-force python loops, and the chunk-size arithmetic of plnlp_b200/recommend.py."""
import math

import pytest
import torch

from oracle import ranking

NAN, INF = float("nan"), float("inf")


def _brute_topk(row, k):
    cand = [(0.0 if v == 0 else v, j) for j, v in enumerate(row) if math.isfinite(v)]
    cand.sort(key=lambda t: (-t[0], t[1]))
    cand = cand[:k]
    ids = [j for _, j in cand] + [-1] * (k - len(cand))
    sc = [v for v, _ in cand] + [-INF] * (k - len(cand))
    return ids, sc


def _brute_counts(row, target, ts):
    gt = sum(1 for j, v in enumerate(row) if j != target and math.isfinite(v) and v > ts)
    ge = sum(1 for j, v in enumerate(row) if j != target and math.isfinite(v) and v >= ts)
    return gt, ge


def _rows(kind, Q, N, g):
    if kind == "normal":
        return torch.randn(Q, N, generator=g)
    if kind == "ties":
        return torch.randint(-3, 4, (Q, N), generator=g).float()
    if kind == "constant":
        return torch.full((Q, N), 0.5)
    if kind == "signed_zero":
        s = torch.zeros(Q, N)
        s[:, ::2] = -0.0
        return s
    s = torch.randn(Q, N, generator=g)                    # "special": -inf / NaN / +inf sprinkled, one row all excluded
    r = torch.rand(Q, N, generator=g)
    s[r < 0.2] = -INF
    s[(r >= 0.2) & (r < 0.35)] = NAN
    s[(r >= 0.35) & (r < 0.4)] = INF
    s[0] = -INF
    return s


@pytest.mark.parametrize("kind", ["normal", "ties", "constant", "signed_zero", "special"])
@pytest.mark.parametrize("N,k", [(1, 1), (5, 3), (5, 20), (33, 33), (40, 7), (257, 100)])
def test_oracle_topk_matches_brute_force(kind, N, k):
    g = torch.Generator().manual_seed(N * 31 + k)
    s = _rows(kind, 4, N, g)
    ids, sc = ranking.topk_rows(s, k)
    for q in range(s.size(0)):
        bi, bs = _brute_topk(s[q].tolist(), k)
        assert ids[q].tolist() == bi
        assert torch.equal(sc[q], torch.tensor(bs, dtype=torch.float32))
        assert all(not (v == 0 and math.copysign(1.0, v) < 0) for v in sc[q].tolist())     # -0 reported as +0


@pytest.mark.parametrize("kind", ["normal", "ties", "constant", "special"])
def test_oracle_rank_counts_match_brute_force(kind):
    g = torch.Generator().manual_seed(7)
    Q, N = 6, 50
    s = _rows(kind, Q, N, g)
    target = torch.randint(0, N, (Q,), generator=g)
    ts = s[torch.arange(Q), target]
    ts[1] = 0.25                                         # a target score that is not in the row
    gt, ge = ranking.rank_counts(s, target, ts)
    for q in range(Q):
        assert (int(gt[q]), int(ge[q])) == _brute_counts(s[q].tolist(), int(target[q]), float(ts[q]))


def test_oracle_mask_and_filtered_ranks():
    g = torch.Generator().manual_seed(3)
    Q, N = 5, 12
    s = torch.randn(Q, N, generator=g)
    nodes = torch.tensor([0, 3, 3, 7, 11])
    # CSR over 12 rows: an empty row, duplicates, a self loop, out-of-range columns
    lists = {0: [1, 1, 0], 3: [], 7: [7, 2, 12, -1], 11: [10]}
    rowptr, col = [0], []
    for r in range(N):
        col += lists.get(r, [])
        rowptr.append(len(col))
    rowptr, col = torch.tensor(rowptr), torch.tensor(col, dtype=torch.int32)
    m = ranking.mask_scores(s, nodes, rowptr, col, exclude_self=True)
    for q, n in enumerate(nodes.tolist()):
        banned = {c for c in lists.get(n, []) if 0 <= c < N} | {n}
        for j in range(N):
            assert (m[q, j] == -INF) == (j in banned) or s[q, j] == -INF
    targets = torch.tensor([1, 4, 5, 2, 10])             # targets 1, 2, 10 are known links: never excluded
    r = ranking.filtered_ranks(s, targets, nodes, rowptr, col)
    for q, n in enumerate(nodes.tolist()):
        t = int(targets[q])
        banned = ({c for c in lists.get(n, []) if 0 <= c < N} | {n}) - {t}
        row = [(-INF if j in banned else v) for j, v in enumerate(s[q].tolist())]
        gt, ge = _brute_counts(row, t, float(s[q, t]))
        assert float(r[q]) == 1.0 + 0.5 * (gt + ge)


def test_oracle_topk_k_equals_n_is_a_full_sort():
    g = torch.Generator().manual_seed(11)
    s = torch.randint(0, 5, (3, 64), generator=g).float()
    ids, sc = ranking.topk_rows(s, 64)
    for q in range(3):
        assert sorted(ids[q].tolist()) == list(range(64))
        assert ids[q].tolist() == sorted(range(64), key=lambda j: (-float(s[q, j]), j))


def test_chunk_arithmetic():
    from plnlp_b200 import recommend as R
    N = 2927963
    # GEMM paths: one fp32 score row per query
    assert R.query_bytes(N, "gemm") == 4 * N
    bs = R.default_batch_size(N, "gemm")
    assert bs == (1 << 30) // (4 * N) == 91
    assert bs * R.query_bytes(N, "gemm") <= R.CHUNK_BYTES < (bs + 1) * R.query_bytes(N, "gemm")
    # fused MLP path: score row + int64 pair list + two partial rows + their sum
    assert R.query_bytes(N, "fused_mlp", 2) == N * (4 + 16 + 8 + 4)
    bs = R.default_batch_size(N, "fused_mlp", 2)
    assert bs * R.query_bytes(N, "fused_mlp", 2) <= R.CHUNK_BYTES < (bs + 1) * R.query_bytes(N, "fused_mlp", 2)
    # never below one query, whatever the graph
    assert R.default_batch_size(10 ** 10, "fused_mlp", 8) == 1
    assert R.default_batch_size(100, "gemm", budget=1) == 1
    # the GEMM configuration depends on the candidate side only
    assert R.gemm_backend(100, 256) == "ffma"              # small graph
    assert R.gemm_backend(N, 1) == "ffma"                  # MLPDOT's width-1 node embedding
    assert R.gemm_backend(8192, 200) == R.gemm_backend(N, 200) != "ffma"

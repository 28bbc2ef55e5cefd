"""CPU tests (-m "not gpu") of heuristic recommendation and full ranking (plnlp_b200/heuristics.py recommend /
rank_against_all): dense score rows built from the oracle's pair sums (oracle/heuristics.py) against its pair
scores, a restatement of the two-hop reach set the mark kernel enumerates, the per-rank partial rows of the
row-partitioned graph added in rank order, a 2-rank gloo run of both collective calls with the raw ops swapped for
the references below, and the argument checks."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import heuristics as oh
from oracle import ranking
from tests.ranking_merge import merge_topk
from tests.test_heuristics_cpu import _csr, _graph, _ulp_close, ref_clean, ref_op

METHODS = ("CN", "AA", "RA")


def transpose_sets(sets):
    """R(w) = {j : w in N(j)}"""
    R = [set() for _ in sets]
    for j, s in enumerate(sets):
        for w in s:
            R[w].add(j)
    return R


def dense_rows(sets, nodes, method, cols=None):
    """fp64 [Q, W] numpy: row q holds the exact sums (oracle/heuristics.py score_sets) of the pairs (nodes[q], j) for
    every column node j -- all nodes in ascending order, or the given ``cols``: the rows recommend / rank_against_all
    select from, before the fp32 rounding; nodes outside the two-hop set of the query score 0"""
    nodes = torch.as_tensor(nodes).reshape(-1).tolist()
    cols = list(range(len(sets))) if cols is None else torch.as_tensor(cols).reshape(-1).tolist()
    out = np.zeros((len(nodes), len(cols)), dtype=np.float64)
    for q, u in enumerate(nodes):
        out[q] = oh.score_sets(sets, [[u, j] for j in cols], method)
    return out


def reach_set(sets, R, u):
    """the nodes the mark kernel reaches from u: R(w) for every w in N(u)"""
    out = set()
    for w in sets[u]:
        out |= R[w]
    return out


def _column_nodes(W, col0, cand):
    return list(range(col0, col0 + W)) if cand is None else cand.tolist()


def ref_mark(rowptr, col, rrowptr, rcol, nodes, W, col0=0, cand=None):
    """CPU restatement of _ops.two_hop_mark_raw"""
    rowptr, col, rrowptr, rcol = rowptr.tolist(), col.tolist(), rrowptr.tolist(), rcol.tolist()
    cols = {j: c for c, j in enumerate(_column_nodes(W, col0, cand))}
    bits = np.zeros((len(nodes), (W + 31) // 32), dtype=np.uint32)
    for q, u in enumerate(torch.as_tensor(nodes).tolist()):
        for w in col[rowptr[u]:rowptr[u + 1]]:
            for j in rcol[rrowptr[w]:rrowptr[w + 1]]:
                if j in cols:
                    c = cols[j]
                    bits[q, c >> 5] |= np.uint32(1 << (c & 31))
    return torch.from_numpy(bits.view(np.int32))


def bitmap_columns(bitmap, W):
    """[set of columns] per row of a bitmap"""
    b = bitmap.cpu().numpy().view(np.uint32)
    return [{c for c in range(W) if (int(b[q, c >> 5]) >> (c & 31)) & 1} for q in range(b.shape[0])]


def ref_score(rowptr, col, weight, nodes, bitmap, W, col0=0, cand=None, dtype=torch.float32):
    """CPU restatement of _ops.two_hop_score_raw (exact fp64 sums)"""
    js = _column_nodes(W, col0, cand)
    s = torch.zeros(len(nodes), W, dtype=dtype)
    for q, (u, cs) in enumerate(zip(torch.as_tensor(nodes).tolist(), bitmap_columns(bitmap, W))):
        cs = sorted(cs)
        if cs:
            v = ref_op(rowptr, col, weight, torch.tensor([[u, js[c]] for c in cs]))
            s[q, cs] = v.to(dtype)
    return s


def ref_mask(s, nodes, rowptr=None, col=None, exclude_self=True, col0=0, cand=None):
    """CPU restatement of _ops.score_mask_raw (in place)"""
    js = _column_nodes(s.size(1), col0, cand)
    cols = {j: c for c, j in enumerate(js)}
    for q, u in enumerate(nodes.tolist()):
        drop = [] if rowptr is None else col[int(rowptr[u]):int(rowptr[u + 1])].tolist()
        if exclude_self:
            drop.append(u)
        for j in drop:
            if j in cols:
                s[q, cols[j]] = float("-inf")
    return s


def ref_topk(s, k, target=None, target_score=None, col0=0, cand=None):
    """CPU restatement of _ops.topk_rows_raw"""
    js = torch.tensor(_column_nodes(s.size(1), col0, cand), dtype=torch.int64)
    ids = sc = gt = ge = None
    if k > 0:
        c, sc = ranking.topk_rows(s, k)
        ids = torch.where(c >= 0, js[c.clamp_min(0)], c)
    if target is not None:
        cols = {j: i for i, j in enumerate(js.tolist())}
        tcol = torch.tensor([cols.get(t, -1) for t in target.tolist()], dtype=torch.int64)
        gt, ge = ranking.rank_counts(s, tcol, target_score)
    return ids, sc, gt, ge


def _patch_ops(ops):
    ops.two_hop_mark_raw = ref_mark
    ops.two_hop_score_raw = ref_score
    ops.link_heuristic_raw = ref_op
    ops.score_mask_raw = ref_mask
    ops.topk_rows_raw = ref_topk
    ops.topk_merge_raw = merge_topk


@pytest.fixture
def ref_ops(monkeypatch):
    from plnlp_b200 import _ops, heuristics
    for name, fn in (("two_hop_mark_raw", ref_mark), ("two_hop_score_raw", ref_score),
                     ("link_heuristic_raw", ref_op), ("score_mask_raw", ref_mask), ("topk_rows_raw", ref_topk),
                     ("topk_merge_raw", merge_topk)):
        monkeypatch.setattr(_ops, name, fn)
    monkeypatch.setattr(heuristics, "clean_csr", ref_clean)


def _sets(src, dst, n):
    rowptr, col, _ = _csr(src, dst, n).csr()
    return oh.neighbour_sets(rowptr, col, n)


@pytest.mark.parametrize("method", METHODS)
def test_oracle_rows_match_pair_scores(method):
    n = 30
    sets = _sets(*_graph(n, 90, 2, symmetric=False), n)
    nodes = torch.tensor([0, 3, 3, 29, 7])
    rows = dense_rows(sets, nodes, method)
    pairs = torch.stack([nodes.repeat_interleave(n), torch.arange(n).repeat(nodes.numel())], 1)
    assert rows.shape == (5, n)
    assert np.array_equal(rows.reshape(-1).astype(np.float32), oh.score_sets(sets, pairs, method).astype(np.float32))
    cols = torch.tensor([2, 5, 11, 28])
    assert np.array_equal(dense_rows(sets, nodes, method, cols), rows[:, cols.numpy()])


@pytest.mark.parametrize("symmetric", [True, False])
def test_reach_set_covers_every_nonzero_score(symmetric):
    from plnlp_b200 import heuristics
    n = 60
    src, dst = _graph(n, 200, 5, symmetric)
    adj = _csr(src, dst, n)
    rowptr, col, _ = adj.csr()
    sets = oh.neighbour_sets(rowptr, col, n)
    R = transpose_sets(sets)
    rows = torch.repeat_interleave(torch.arange(n), rowptr[1:] - rowptr[:-1])
    table = heuristics.NeighbourTable(*ref_clean(rows, col.to(torch.int64), n), clean=ref_clean)
    rr, rc = table.reach()
    assert oh.neighbour_sets(rr, rc, n) == R                  # the transpose the kernel walks
    if symmetric:
        assert R == sets
    nodes = torch.arange(n)
    bitmap = ref_mark(table.rowptr, table.col, rr, rc, nodes, n)
    for u, got in zip(range(n), bitmap_columns(bitmap, n)):
        reach = reach_set(sets, R, u)
        assert got == reach
        assert all(sets[u] & sets[j] for j in reach)
        for m in METHODS:
            nz = set(np.flatnonzero(dense_rows(sets, [u], m)[0]).tolist())
            assert nz <= reach, (u, m)
    # a column range and a candidate set see the same reach
    cand = torch.tensor([1, 4, 9, 33, 59])
    for c0, W, cd in ((10, 25, None), (0, 5, cand)):
        js = _column_nodes(W, c0, cd)
        bm = bitmap_columns(ref_mark(table.rowptr, table.col, rr, rc, nodes, W, c0, cd), W)
        for u in range(n):
            assert bm[u] == {c for c, j in enumerate(js) if j in reach_set(sets, R, u)}


def _splits(n):
    from plnlp_b200 import parallel
    return [(R, [parallel.row_block(n, r, R) for r in range(R)]) for R in (1, 2, 3)]


@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("n,symmetric,cand", [(50, True, None), (41, False, None), (41, False, "set"),
                                               (4, True, None), (4, True, "set")])   # n = 4: an empty last block
def test_shard_partial_rows_add_up_to_the_whole(ref_ops, method, n, symmetric, cand):
    from plnlp_b200 import heuristics, parallel
    from plnlp_b200.graph import CSRGraph
    src, dst = _graph(n, 5 * n, 7, symmetric)
    adj = _csr(src, dst, n)
    sets = _sets(src, dst, n)
    nodes = torch.tensor([0, 1, n - 1, 2, 0])
    cols = None if cand is None else torch.tensor(sorted({0, 1, n // 2, n - 1}), dtype=torch.int64)
    whole = dense_rows(sets, nodes, method, cols)
    for R, bounds in _splits(n):
        shards = []
        for r, (lo, hi) in enumerate(bounds):
            sadj = parallel.shard_graph(adj, r, R, CSRGraph)
            table = heuristics.shard_table(sadj.local, sadj.local_t, lo, hi, n, clean=ref_clean)
            shards.append(heuristics.RankShard(table, method, n, r, R, cand=cols))
        sends = []
        for r, sh in enumerate(shards):
            P, send = sh.partial(nodes)
            lo, hi = bounds[r]
            W = whole.shape[1]
            want = np.stack([oh.score_sets(sets, [[u, j] for j in _column_nodes(W, 0, cols)], method,
                                           keep=lambda w: lo <= w < hi) for u in nodes.tolist()])
            assert np.allclose(P[:, :W].numpy(), want, rtol=1e-14, atol=0), (R, r)
            assert not P[:, W:].any()                         # the padding columns past the last node
            sends.append(send)
        got = []
        for s, sh in enumerate(shards):
            got.append(sh.combine(torch.stack([sends[r][s] for r in range(R)])))
        got = torch.cat(got, 1)
        assert got.shape == whole.shape
        ref = torch.from_numpy(whole.astype(np.float32))
        assert torch.equal(got, ref) if method == "CN" else _ulp_close(got, ref), R


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


N_GLOO = 37


def _gloo_args():
    src, dst = _graph(N_GLOO, 150, 11, symmetric=False)
    g = torch.Generator().manual_seed(13)
    nodes = torch.randint(0, N_GLOO, (9,), generator=g)
    edges = torch.stack([nodes, torch.randint(0, N_GLOO, (9,), generator=g)], 1)
    exclude = torch.randint(0, N_GLOO, (40, 2), generator=g)
    cand = torch.tensor([3, 30, 1, 17, 17, 22, 36, 8])
    return src, dst, nodes, edges, exclude, cand


def _worker(rank, ws, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=ws)
    try:
        from plnlp_b200 import _ops, heuristics, parallel
        from plnlp_b200.graph import CSRGraph
        heuristics.clean_csr = ref_clean                  # this process only
        _patch_ops(_ops)
        real_gather = dist.all_gather_into_tensor

        def flat_gather(out, inp, group=None, async_op=False):   # gloo wants the outputs flat
            return real_gather(out.view(-1), inp.reshape(-1), group=group, async_op=async_op)
        dist.all_gather_into_tensor = flat_gather
        src, dst, nodes, edges, exclude, cand = _gloo_args()
        sadj = parallel.shard_graph(_csr(src, dst, N_GLOO), rank, ws, CSRGraph)
        out = {}
        for m in METHODS:
            for ex in (None, exclude):
                for c in (None, cand):
                    key = (m, ex is not None, c is not None)
                    out[key] = (heuristics.recommend(sadj, nodes, 6, m, ex, True, 4, c),
                                heuristics.rank_against_all(sadj, edges, m, ex, True, 4, c))
        errors = []
        for bad in ({"method": "CN" if rank == 0 else "AA"}, {"k": 5 + rank}, {"batch_size": 3 + rank}):
            kw = {"method": "RA", "k": 5, "batch_size": None, **bad}
            try:
                heuristics.recommend(sadj, nodes, kw["k"], kw["method"], batch_size=kw["batch_size"])
                errors.append(None)
            except ValueError as e:
                errors.append(str(e))
        try:
            heuristics.rank_against_all(sadj, edges[:5 + rank], "CN")
            errors.append(None)
        except ValueError as e:
            errors.append(str(e))
        out["errors"] = errors
        ret[rank] = out
    finally:
        dist.destroy_process_group()


def _oracle_calls(m, ex, c):
    src, dst, nodes, edges, exclude, cand = _gloo_args()
    rowptr, col, _ = _csr(src, dst, N_GLOO).csr()
    sets = oh.neighbour_sets(rowptr, col, N_GLOO)
    S = torch.from_numpy(dense_rows(sets, nodes, m).astype(np.float32))
    er, ec = (None, None)
    if ex:
        er = torch.zeros(N_GLOO + 1, dtype=torch.int64)
        er[1:] = torch.cumsum(torch.bincount(exclude[:, 0], minlength=N_GLOO), 0)
        ec = exclude[torch.argsort(exclude[:, 0], stable=True), 1]
    keep = torch.ones(N_GLOO, dtype=torch.bool)
    if c:
        keep[:] = False
        keep[cand] = True
    Sm = ranking.mask_scores(S, nodes, er, ec, True)
    Sm[:, ~keep] = float("-inf")
    ids, sc = ranking.topk_rows(Sm, 6)
    St = torch.from_numpy(dense_rows(sets, edges[:, 0], m).astype(np.float32))
    t = edges[:, 1]
    ts = St[torch.arange(t.numel()), t]
    Sr = ranking.mask_scores(St, edges[:, 0], er, ec, True)
    drop = ~keep[None, :].expand_as(Sr).clone()
    drop[torch.arange(t.numel()), t] = False                  # the target is never excluded
    Sr[drop] = float("-inf")
    gt, ge = ranking.rank_counts(Sr, t, ts)
    return ids, sc, (1.0 + 0.5 * (gt.double() + ge.double())).float()


def test_collective_recommend_and_rank_gloo():
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(2, _free_port(), ret), nprocs=2, join=True)
    for m in METHODS:
        for ex in (False, True):
            for c in (False, True):
                ids, sc, ranks = _oracle_calls(m, ex, c)
                for r in range(2):
                    (gi, gs), gr = ret[r][(m, ex, c)]
                    assert gi.shape == (9, 6) and gs.dtype == torch.float32 and gr.dtype == torch.float32
                    if m == "CN":
                        assert torch.equal(gi, ids) and torch.equal(gs, sc), (m, ex, c)
                        assert torch.equal(gr, ranks), (m, ex, c)
                    else:
                        fin = torch.isfinite(sc)
                        assert torch.equal(fin, torch.isfinite(gs))
                        assert _ulp_close(gs[fin], sc[fin]), (m, ex, c)
    for r in range(2):
        assert all(e is not None and "collective" in e for e in ret[r]["errors"]), ret[r]["errors"]


def test_argument_checks():
    from plnlp_b200 import heuristics
    n = 20
    adj = _csr(*_graph(n, 50, 1), n)
    nodes = torch.tensor([0, 1])
    edges = torch.zeros(3, 2, dtype=torch.int64)
    bad_rec = [dict(method="Jaccard"), dict(k=0), dict(k=1025), dict(nodes=nodes.to(torch.int32)),
               dict(nodes=torch.tensor([n])), dict(nodes=torch.tensor([-1])), dict(exclude="known"),
               dict(exclude=torch.zeros(3, 3, dtype=torch.int64)), dict(exclude=torch.tensor([[0, n]])),
               dict(exclude=torch.zeros(3, 2, dtype=torch.int32)), dict(candidates=torch.tensor([0, n])),
               dict(candidates=torch.zeros(2, 2, dtype=torch.int64)), dict(candidates=torch.tensor([1.0])),
               dict(batch_size=-1)]
    for bad in bad_rec:
        kw = {"nodes": nodes, "k": 3, "method": "CN"}
        kw.update({k: v for k, v in bad.items() if k in kw})
        extra = {k: v for k, v in bad.items() if k not in kw}
        with pytest.raises(ValueError):
            heuristics.recommend(adj, kw["nodes"], kw["k"], kw["method"], **extra)
    bad_rank = [dict(method="jaccard"), dict(edges=edges.to(torch.int32)), dict(edges=torch.zeros(3, 3, dtype=torch.int64)),
                dict(edges=torch.tensor([[0, n]])), dict(exclude="all"), dict(candidates=torch.tensor([[0]])),
                dict(batch_size=-2)]
    for bad in bad_rank:
        e = bad.pop("edges", edges)
        m = bad.pop("method", "AA")
        with pytest.raises(ValueError):
            heuristics.rank_against_all(adj, e, m, **bad)
    from plnlp_b200.graph import CSRGraph
    rect = CSRGraph.from_coo(torch.tensor([0, 1]), torch.tensor([1, 2]), None, (2, 3))
    with pytest.raises(ValueError):
        heuristics.recommend(rect, torch.tensor([0]), 1, "CN")
    with pytest.raises(ValueError):
        heuristics.rank_against_all(rect, torch.tensor([[0, 1]]), "CN")

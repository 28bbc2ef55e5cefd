"""CPU tests (-m "not gpu") of the common-neighbour link heuristics: the oracle (oracle/heuristics.py) against brute
force on dense matrices, the neighbour-set cleaning rules, the decomposition of a score into per-shard partials over
blocks of intermediate nodes (plnlp_b200/heuristics.Shard with reference ops), the collective bookkeeping over
torch.distributed gloo, and the argument checks of score_edges."""
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import heuristics as oh

METHODS = ("CN", "AA", "RA")


def ref_clean(row, col, n):
    """CPU restatement of heuristics.clean_csr"""
    keep = row != col
    key = torch.unique(row[keep] * n + col[keep])
    rowptr = torch.zeros(n + 1, dtype=torch.int64)
    rowptr[1:] = torch.cumsum(torch.bincount(key // n, minlength=n), 0)
    return rowptr, (key % n).to(torch.int32)


def ref_op(rowptr, col, weight, edges):
    """CPU restatement of _ops.link_heuristic_raw: exact fp64 sums over the common neighbours"""
    rowptr, col = rowptr.tolist(), col.tolist()
    w = None if weight is None else weight.tolist()
    out = []
    for u, v in edges.tolist():
        common = set(col[rowptr[u]:rowptr[u + 1]]) & set(col[rowptr[v]:rowptr[v + 1]])
        out.append(math.fsum(1.0 if w is None else w[x] for x in sorted(common)))
    return torch.tensor(out, dtype=torch.float64)


def _graph(n, m, seed, symmetric=True, loops=True, dups=True):
    g = torch.Generator().manual_seed(seed)
    # a few hubs: power-law-ish rows
    src = torch.cat([torch.randint(0, n, (m,), generator=g), torch.zeros(n // 2, dtype=torch.int64)])
    dst = torch.cat([torch.randint(0, n, (m,), generator=g), torch.arange(n // 2)])
    if not loops:
        keep = src != dst
        src, dst = src[keep], dst[keep]
    if dups:
        src, dst = torch.cat([src, src[:m // 4]]), torch.cat([dst, dst[:m // 4]])
    if symmetric:
        src, dst = torch.cat([src, dst]), torch.cat([dst, src])
    return src, dst


def _csr(src, dst, n, value=True):
    from plnlp_b200.graph import CSRGraph
    v = torch.rand(src.numel(), dtype=torch.float32, generator=torch.Generator().manual_seed(1)) if value else None
    return CSRGraph.from_coo(src, dst, v, (n, n))


def _pairs(n, P, seed):
    g = torch.Generator().manual_seed(seed)
    e = torch.randint(0, n, (P, 2), generator=g)
    e[:5, 1] = e[:5, 0]                                    # (u, u) pairs
    e[5:10, 0] = 0                                         # the hub
    return e


def _brute(src, dst, n, edges, method):
    A = np.zeros((n, n), dtype=bool)
    A[src.numpy(), dst.numpy()] = True
    np.fill_diagonal(A, False)
    d = A.sum(1)
    with np.errstate(divide="ignore"):
        w = {"CN": np.ones(n), "AA": np.where(d >= 2, 1.0 / np.log(np.maximum(d, 2)), 0.0),
             "RA": np.where(d >= 1, 1.0 / np.maximum(d, 1), 0.0)}[method]
    e = edges.numpy()
    return (A[e[:, 0]] & A[e[:, 1]]).astype(np.float64) @ w


def _ulp_close(a, b, ulps=1):
    a, b = torch.as_tensor(a, dtype=torch.float32), torch.as_tensor(b, dtype=torch.float32)
    ia = a.view(torch.int32).to(torch.int64)
    ib = b.view(torch.int32).to(torch.int64)
    return bool(((ia - ib).abs() <= ulps).all())


@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("symmetric", [True, False])
def test_oracle_matches_brute_force(method, symmetric):
    n = 60
    src, dst = _graph(n, 300, 3, symmetric)
    adj = _csr(src, dst, n)
    rowptr, col, _ = adj.csr()
    edges = _pairs(n, 400, 4)
    got = oh.score(rowptr, col, n, edges, method)
    want = torch.from_numpy(_brute(src, dst, n, edges, method).astype(np.float32))
    if method == "CN":
        assert torch.equal(got, want)
    else:
        assert _ulp_close(got, want)


def test_cleaning_rules():
    from plnlp_b200.graph import CSRGraph
    n = 6
    # row 0: duplicates and a self loop; row 1: only a self loop; row 2: empty; rows 3 -> 4 but not 4 -> 3
    src = torch.tensor([0, 0, 0, 0, 1, 3, 5, 5])
    dst = torch.tensor([1, 1, 0, 5, 1, 4, 0, 1])
    adj = CSRGraph.from_coo(src, dst, torch.tensor([9.0, -2.0, 1.0, 0.5, 3.0, 1.0, 1.0, 1.0]), (n, n))
    rowptr, col, _ = adj.csr()
    sets = oh.neighbour_sets(rowptr, col, n)
    assert sets == [{1, 5}, set(), set(), {4}, set(), {0, 1}]
    # the same sets through the reference of clean_csr, and after set_diag (values and diagonal do not matter)
    r2, c2 = ref_clean(src, dst, n)
    assert oh.neighbour_sets(r2, c2, n) == sets
    assert torch.equal(c2, torch.tensor([1, 5, 4, 0, 1], dtype=torch.int32))
    rd, cd, _ = adj.set_diag().csr()
    assert oh.neighbour_sets(rd, cd, n) == sets
    # non-symmetric: row u as stored.  CN(0, 5): N(0) & N(5) = {1}; d(1) = 0, so AA and RA add nothing
    e = torch.tensor([[0, 5], [3, 4], [4, 3], [2, 2], [0, 0]])
    assert oh.score(rowptr, col, n, e, "CN").tolist() == [1.0, 0.0, 0.0, 0.0, 2.0]
    assert oh.score(rowptr, col, n, e, "RA").tolist() == [0.0, 0.0, 0.0, 0.0, 0.5]
    # (0, 0): common neighbours 1 (d = 0) and 5 (d = 2): AA = 1 / ln 2
    assert oh.score(rowptr, col, n, e, "AA")[4].item() == np.float32(1.0 / math.log(2.0))


def _splits(n):
    from plnlp_b200 import parallel
    return [(R, [parallel.row_block(n, r, R) for r in range(R)]) for R in (1, 2, 3)]


@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("n,symmetric", [(50, True), (41, False), (4, True)])   # (4, 3 blocks): 2, 2 and 0 rows
def test_shard_partials_add_up_to_the_whole(method, n, symmetric):
    from plnlp_b200 import heuristics, parallel
    from plnlp_b200.graph import CSRGraph
    src, dst = _graph(n, 5 * n, 7, symmetric)
    adj = _csr(src, dst, n)
    rowptr, col, _ = adj.csr()
    edges = _pairs(n, 200, 8)
    sets = oh.neighbour_sets(rowptr, col, n)
    whole = oh.score_sets(sets, edges, method)
    for R, bounds in _splits(n):
        total = torch.zeros(edges.size(0), dtype=torch.float64)
        for r, (lo, hi) in enumerate(bounds):
            sadj = parallel.shard_graph(adj, r, R, CSRGraph)
            table = heuristics.shard_table(sadj.local, sadj.local_t, lo, hi, n, clean=ref_clean)
            part = heuristics.Shard(table, op=ref_op).partial(edges, method)
            want = oh.score_sets(sets, edges, method, keep=lambda w: lo <= w < hi)
            assert np.allclose(part.numpy(), want, rtol=1e-14, atol=0), (R, r)
            total += part
        if method == "CN":
            assert np.array_equal(total.numpy(), whole)
        else:
            assert np.allclose(total.numpy(), whole, rtol=1e-14, atol=0), R
            assert _ulp_close(total.to(torch.float32), torch.from_numpy(whole.astype(np.float32)))


def test_score_edges_argument_checks():
    from plnlp_b200 import heuristics
    adj = _csr(*_graph(20, 50, 1), 20)
    good = torch.zeros(3, 2, dtype=torch.int64)
    with pytest.raises(ValueError):
        heuristics.score_edges(adj, good, "Jaccard")
    with pytest.raises(ValueError):
        heuristics.score_edges(adj, good.to(torch.int32), "CN")
    with pytest.raises(ValueError):
        heuristics.score_edges(adj, torch.zeros(3, 3, dtype=torch.int64), "CN")
    with pytest.raises(ValueError):
        heuristics.score_edges(adj, torch.zeros(6, dtype=torch.int64), "CN")
    with pytest.raises(ValueError):
        heuristics.score_edges(adj, torch.tensor([[0, 20]]), "AA")
    with pytest.raises(ValueError):
        heuristics.score_edges(adj, torch.tensor([[-1, 0]]), "RA")


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


N_GLOO = 37


def _worker(rank, ws, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=ws)
    try:
        from plnlp_b200 import _ops, heuristics, parallel
        from plnlp_b200.graph import CSRGraph
        heuristics.clean_csr = ref_clean                  # this process only
        _ops.link_heuristic_raw = ref_op
        real_gather = dist.all_gather_into_tensor

        def flat_gather(out, inp, group=None, async_op=False):   # gloo wants the [R, n] output of _agree flat
            return real_gather(out.view(-1), inp, group=group, async_op=async_op)
        dist.all_gather_into_tensor = flat_gather
        src, dst = _graph(N_GLOO, 150, 11, symmetric=False)
        sadj = parallel.shard_graph(_csr(src, dst, N_GLOO), rank, ws, CSRGraph)
        edges = _pairs(N_GLOO, 120, 12)
        out = {m: heuristics.score_edges(sadj, edges, m, batch_size=50) for m in METHODS}
        out["cached"] = heuristics.neighbour_table(sadj) is heuristics.neighbour_table(sadj)
        errors = []
        for bad in ({"method": "CN" if rank == 0 else "AA"}, {"edges": edges[: 100 + rank]},
                    {"batch_size": 10 + rank}):
            kw = {"edges": edges, "method": "RA", "batch_size": None, **bad}
            try:
                heuristics.score_edges(sadj, kw["edges"], kw["method"], kw["batch_size"])
                errors.append(None)
            except ValueError as e:
                errors.append(str(e))
        out["errors"] = errors
        ret[rank] = out
    finally:
        dist.destroy_process_group()


def test_collective_score_edges_gloo():
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(2, _free_port(), ret), nprocs=2, join=True)
    src, dst = _graph(N_GLOO, 150, 11, symmetric=False)
    rowptr, col, _ = _csr(src, dst, N_GLOO).csr()
    edges = _pairs(N_GLOO, 120, 12)
    for m in METHODS:
        want = oh.score(rowptr, col, N_GLOO, edges, m)
        for r in range(2):
            got = ret[r][m]
            assert got.dtype == torch.float32 and got.shape == (120,)
            assert torch.equal(got, want) if m == "CN" else _ulp_close(got, want), (m, r)
    for r in range(2):
        assert ret[r]["cached"]
        assert all(e is not None and "collective" in e for e in ret[r]["errors"]), ret[r]["errors"]

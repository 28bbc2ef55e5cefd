"""GPU tests of the common-neighbour link heuristics (plnlp_b200/heuristics.py, csrc/heuristic.cu) against the CPU
oracle (oracle/heuristics.py): CN bit for bit, AA and RA within one fp32 ulp, on a graph with hub rows of several
thousand entries, hub-hub pairs, isolated nodes, (u, u) pairs and more pairs than one pass of the grid covers; the
neighbour table against its CPU restatement; the ABI error codes; virtual shards of the row-partitioned graph; a
one-rank NCCL run of the collective path; and ``heuristics.test`` against the metric code on the oracle's scores."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import heuristics as oh
from tests.test_heuristics_cpu import _ulp_close, ref_clean

pytestmark = pytest.mark.gpu

METHODS = ("CN", "AA", "RA")
N, HUBS, HUB_DEG, N_ISOLATED = 12000, 4, 5000, 200
P = 40000                       # > 8 warps x 1184 blocks: several grid-stride passes


def _edges_coo(symmetric=True, seed=0):
    """random graph on N nodes, the last N_ISOLATED isolated, rows 0..HUBS-1 hubs of ~HUB_DEG entries sharing
    neighbours, with duplicates and self loops"""
    g = torch.Generator().manual_seed(seed)
    m = N - N_ISOLATED
    src = [torch.randint(0, m, (60000,), generator=g)]
    dst = [torch.randint(0, m, (60000,), generator=g)]
    for h in range(HUBS):
        nb = torch.randint(0, m, (HUB_DEG,), generator=g)
        src.append(torch.full((HUB_DEG,), h, dtype=torch.int64))
        dst.append(nb)
    src.append(torch.arange(0, m, 97))                    # self loops
    dst.append(torch.arange(0, m, 97))
    src, dst = torch.cat(src), torch.cat(dst)
    src, dst = torch.cat([src, src[:3000]]), torch.cat([dst, dst[:3000]])     # duplicates
    if symmetric:
        src, dst = torch.cat([src, dst]), torch.cat([dst, src])
    return src, dst


def _adj(symmetric=True, dev="cuda"):
    from plnlp_b200.graph import CSRGraph
    src, dst = _edges_coo(symmetric)
    v = torch.rand(src.numel(), generator=torch.Generator().manual_seed(2))
    return CSRGraph.from_coo(src.to(dev), dst.to(dev), v.to(dev), (N, N))


def _pairs(seed=1):
    g = torch.Generator().manual_seed(seed)
    e = torch.randint(0, N, (P, 2), generator=g)
    hubs = torch.arange(HUBS)
    e[:HUBS * HUBS] = torch.stack([hubs.repeat_interleave(HUBS), hubs.repeat(HUBS)], 1)   # hub-hub, (h, h)
    e[20:1000, 0] = torch.randint(0, HUBS, (980,), generator=g)                            # hub-small
    e[1000:1100, 1] = e[1000:1100, 0]                                                    # (u, u)
    e[1100:1200, 0] = torch.randint(N - N_ISOLATED, N, (100,), generator=g)               # isolated
    return e


_ORACLE = {}


def _oracle(symmetric, method):
    key = (symmetric, method)
    if key not in _ORACLE:
        rowptr, col, _ = _adj(symmetric, "cpu").csr()
        _ORACLE[key] = oh.score(rowptr, col, N, _pairs(), method)
    return _ORACLE[key]


def test_neighbour_table_matches_cpu_restatement():
    from plnlp_b200 import heuristics
    for symmetric in (True, False):
        src, dst = _edges_coo(symmetric)
        rowptr, col = heuristics.clean_csr(src.cuda(), dst.cuda(), N)
        r0, c0 = ref_clean(src, dst, N)
        assert torch.equal(rowptr.cpu(), r0) and torch.equal(col.cpu(), c0)
    # all entries diagonal, and no entries
    d = torch.arange(5, device="cuda")
    rowptr, col = heuristics.clean_csr(d, d, 5)
    assert rowptr.tolist() == [0] * 6 and col.numel() == 0
    e = torch.empty(0, dtype=torch.int64, device="cuda")
    rowptr, col = heuristics.clean_csr(e, e, 5)
    assert rowptr.tolist() == [0] * 6 and col.numel() == 0


@pytest.mark.parametrize("symmetric", [True, False])
@pytest.mark.parametrize("method", METHODS)
def test_scores_match_oracle(method, symmetric):
    from plnlp_b200 import heuristics
    adj = _adj(symmetric)
    e = _pairs().cuda()
    got = heuristics.score_edges(adj, e, method)
    assert got.dtype == torch.float32 and got.device.type == "cuda" and got.shape == (P,)
    want = _oracle(symmetric, method)
    if method == "CN":
        assert torch.equal(got.cpu(), want)
    else:
        assert _ulp_close(got.cpu(), want)
    assert float(want[:HUBS * HUBS].max()) > 0                # the hub-hub pairs do share neighbours
    # run to run and batch to batch: the same bits
    assert torch.equal(heuristics.score_edges(adj, e, method), got)
    assert torch.equal(heuristics.score_edges(adj, e, method, batch_size=7777), got)


def test_table_is_cached_and_values_ignored():
    from plnlp_b200 import heuristics
    from plnlp_b200.utils import gcn_normalization
    adj = _adj()
    assert heuristics.neighbour_table(adj) is heuristics.neighbour_table(adj)
    e = _pairs().cuda()
    for m in METHODS:
        assert torch.equal(heuristics.score_edges(gcn_normalization(adj), e, m), heuristics.score_edges(adj, e, m))


def test_empty_and_checks():
    from plnlp_b200 import heuristics
    adj = _adj()
    out = heuristics.score_edges(adj, torch.empty(0, 2, dtype=torch.int64, device="cuda"), "AA")
    assert out.shape == (0,) and out.dtype == torch.float32
    with pytest.raises(ValueError):
        heuristics.score_edges(adj, torch.tensor([[0, N]], device="cuda"), "CN")
    with pytest.raises(ValueError):
        heuristics.score_edges(adj, torch.zeros(2, 2, dtype=torch.float32, device="cuda"), "CN")


def test_abi_error_codes():
    from plnlp_b200 import _lib
    lib = _lib.load()
    t = _lib.stream()
    rowptr = torch.zeros(11, dtype=torch.int64, device="cuda")
    col = torch.zeros(4, dtype=torch.int32, device="cuda")
    e = torch.zeros(3, 2, dtype=torch.int64, device="cuda")
    out = torch.empty(3, dtype=torch.float64, device="cuda")
    p = _lib.ptr
    f = lib.plnlp_link_heuristic_f64
    assert f(p(rowptr), p(col), 10, 4, None, p(e), 3, p(out), t) == 0
    assert torch.equal(out.cpu(), torch.zeros(3, dtype=torch.float64))
    assert f(None, p(col), 10, 4, None, p(e), 3, p(out), t) == -1
    assert f(p(rowptr), None, 10, 4, None, p(e), 3, p(out), t) == -1
    assert f(p(rowptr), p(col), 10, 4, None, None, 3, p(out), t) == -1
    assert f(p(rowptr), p(col), 10, 4, None, p(e), 3, None, t) == -1
    assert f(p(rowptr), None, 10, 0, None, p(e), 3, p(out), t) == 0          # no entries: col may be NULL
    assert f(p(rowptr), p(col), -1, 4, None, p(e), 3, p(out), t) == -2
    assert f(p(rowptr), p(col), 10, -1, None, p(e), 3, p(out), t) == -2
    assert f(p(rowptr), p(col), 10, 4, None, p(e), -1, p(out), t) == -2
    assert f(None, None, 10, 4, None, None, 0, None, t) == 0                 # P = 0: nothing to do
    torch.cuda.synchronize()


@pytest.mark.parametrize("symmetric", [True, False])
def test_virtual_shards(symmetric):
    from plnlp_b200 import heuristics, parallel
    from plnlp_b200.graph import CSRGraph
    adj = _adj(symmetric)
    e = _pairs().cuda()
    single = {m: heuristics.score_edges(adj, e, m) for m in METHODS}
    for R, bounds in [(R, [parallel.row_block(N, r, R) for r in range(R)]) for R in (1, 2, 3)] + [
            (3, "uneven")]:
        n = N
        if bounds == "uneven":                  # 4 nodes in 3 blocks: 2, 2 and an empty last block
            n = 4
            bounds = [parallel.row_block(n, r, R) for r in range(R)]
            assert bounds[-1][0] == bounds[-1][1]
        a = adj if n == N else _small_adj()
        pe = e if n == N else torch.randint(0, n, (50, 2), device="cuda")
        ref = single if n == N else {m: heuristics.score_edges(a, pe, m) for m in METHODS}
        for m in METHODS:
            total = torch.zeros(pe.size(0), dtype=torch.float64, device="cuda")
            for r, (lo, hi) in enumerate(bounds):
                sadj = parallel.shard_graph(a, r, R, CSRGraph)
                total += heuristics.Shard(heuristics.shard_table(sadj.local, sadj.local_t, lo, hi, n)).partial(pe, m)
            got = total.to(torch.float32)
            if m == "CN" or R == 1:
                assert torch.equal(got, ref[m]), (R, m)
            else:
                assert _ulp_close(got.cpu(), ref[m].cpu()), (R, m)


def _small_adj():
    from plnlp_b200.graph import CSRGraph
    src = torch.tensor([0, 1, 1, 2, 3, 3, 0, 2], device="cuda")
    dst = torch.tensor([1, 0, 2, 1, 0, 2, 3, 3], device="cuda")
    return CSRGraph.from_coo(src, dst, None, (4, 4))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _split_hits(dev):
    g = torch.Generator().manual_seed(9)
    return {"train": {"edge": torch.zeros(1, 2, dtype=torch.int64)},
            **{s: {"edge": torch.randint(0, N, (3000, 2), generator=g).to(dev),
                   "edge_neg": torch.randint(0, N, (5000, 2), generator=g).to(dev)} for s in ("valid", "test")}}


def _split_mrr(dev):
    g = torch.Generator().manual_seed(10)
    return {"train": {"source_node": torch.zeros(1, dtype=torch.int64)},
            **{s: {"source_node": torch.randint(0, HUBS * 50, (500,), generator=g).to(dev),
                   "target_node": torch.randint(0, N, (500,), generator=g).to(dev),
                   "target_node_neg": torch.randint(0, N, (500, 100), generator=g).to(dev)} for s in ("valid", "test")}}


def _oracle_test(split, metric, method):
    from plnlp_b200.utils import evaluate_hits, evaluate_mrr, get_pos_neg_edges
    rowptr, col, _ = _adj(True, "cpu").csr()
    sets = oh.neighbour_sets(rowptr, col, N)
    preds = []
    for s in ("valid", "test"):
        for e in get_pos_neg_edges(s, split, device="cpu"):
            preds.append(torch.from_numpy(oh.score_sets(sets, e, method).astype(np.float32)).cuda())
    return (evaluate_hits if metric == "hits" else evaluate_mrr)(None, *preds)


class _Data:
    pass


@pytest.mark.parametrize("metric", ["hits", "mrr"])
@pytest.mark.parametrize("method", METHODS)
def test_heuristics_test_matches_metric_code(metric, method):
    from plnlp_b200 import heuristics
    data = _Data()
    data.adj_t = _adj()
    split = _split_hits("cuda") if metric == "hits" else _split_mrr("cuda")
    got = heuristics.test(data, split, method, 4096, None, metric)
    want = _oracle_test(split, metric, method)
    assert set(got) == set(want)
    for k in want:
        for a, b in zip(got[k], want[k]):
            # CN is exact; AA and RA may differ in one ulp, which can move a tie at the threshold
            assert a == b if method == "CN" else abs(a - b) <= 2e-3, (k, a, b)


def _worker(rank, ws, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=ws, device_id=dev)
    try:
        from plnlp_b200 import heuristics, parallel
        from plnlp_b200.graph import CSRGraph
        out = {}
        for symmetric in (True, False):
            adj = _adj(symmetric, dev)
            sadj = parallel.shard_graph(adj, rank, ws, CSRGraph)
            e = _pairs().to(dev)
            for m in METHODS:
                out[(symmetric, m)] = (heuristics.score_edges(sadj, e, m, batch_size=15000).cpu(),
                                       heuristics.score_edges(adj, e, m).cpu())
        data, d1 = _Data(), _Data()
        d1.adj_t = _adj(True, dev)
        data.adj_t = parallel.shard_graph(d1.adj_t, rank, ws, CSRGraph)
        split = _split_mrr(dev)
        out["test"] = (heuristics.test(data, split, "RA", None, None, "mrr"),
                       heuristics.test(d1, split, "RA", None, None, "mrr"))
        try:
            heuristics.score_edges(sadj, _pairs().to(dev)[: 10 + rank], "CN")
            out["mismatch"] = None if ws > 1 else "ok"
        except ValueError as err:
            out["mismatch"] = str(err)
        ret[rank] = out
    finally:
        dist.destroy_process_group()


def _check(ret, ws):
    for r in range(ws):
        out = ret[r]
        for (symmetric, m), (got, single) in ((k, v) for k, v in out.items() if isinstance(k, tuple)):
            if m == "CN" or ws == 1:
                assert torch.equal(got, single), (r, symmetric, m)
            else:
                assert _ulp_close(got, single), (r, symmetric, m)
            if ws == 1:
                assert torch.equal(got, _oracle(symmetric, m)) if m == "CN" else _ulp_close(got, _oracle(symmetric, m))
        got, single = out["test"]
        assert got == single if ws == 1 else all(abs(a - b) <= 2e-3 for k in got for a, b in zip(got[k], single[k]))
        assert out["mismatch"] == "ok" if ws == 1 else "collective" in out["mismatch"]


def test_collective_one_rank_nccl():
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(1, _free_port(), ret), nprocs=1, join=True)
    _check(ret, 1)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_collective_two_ranks_nccl():
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(2, _free_port(), ret), nprocs=2, join=True)
    _check(ret, 2)

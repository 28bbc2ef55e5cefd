"""GPU tests of heuristic recommendation and full ranking (plnlp_b200/heuristics.py recommend / rank_against_all,
csrc/heuristic.cu plnlp_two_hop_mark / plnlp_two_hop_score_*) on the graph of test_gpu_heuristics.py (hub rows of
5 000 entries, isolated nodes, duplicates, self loops; symmetric and not), for CN, AA and RA: bit for bit against
oracle.ranking on dense rows built by score_edges over every (u, j); the returned scores against the fp64 oracle;
chunking and run-to-run identity; candidate sets; the mark bitmap against its CPU restatement and the ABI error
codes; virtual shards of the row-partitioned graph; a one-rank NCCL run of the collective calls."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import heuristics as oh
from oracle import ranking
from tests import ranking_candidates as rc
from tests.test_gpu_heuristics import HUBS, N, N_ISOLATED, _adj, _free_port, _small_adj
from tests.test_heuristics_cpu import _ulp_close
from tests.test_heuristics_recommend_cpu import bitmap_columns, ref_mark

pytestmark = pytest.mark.gpu

METHODS = ("CN", "AA", "RA")
NODES = [0, 1, 5, 5, 777, N - 1, N - N_ISOLATED, 4000, 3, 11111]      # hubs, a repeat, isolated nodes


def _nodes(dev="cuda"):
    return torch.tensor(NODES, dtype=torch.int64, device=dev)


_DENSE = {}


def _dense(adj, symmetric, method, nodes):
    """fp32 [Q, N] on the CPU: score_edges of every (nodes[q], j)"""
    from plnlp_b200 import heuristics
    key = (symmetric, method, tuple(nodes.tolist()))
    if key not in _DENSE:
        q = nodes.to("cuda")
        pairs = torch.stack([q.repeat_interleave(N), torch.arange(N, device="cuda").repeat(q.numel())], 1)
        _DENSE[key] = heuristics.score_edges(adj, pairs, method).reshape(q.numel(), N).cpu()
    return _DENSE[key]


def _exclude_edges(seed=4):
    g = torch.Generator().manual_seed(seed)
    e = torch.stack([torch.tensor(NODES).repeat(30), torch.randint(0, N, (30 * len(NODES),), generator=g)], 1)
    return e.cuda()


def _known(adj, exclude):
    """the known-link CSR of an exclude argument, on the CPU"""
    from plnlp_b200 import recommend
    rowptr, col = recommend.exclude_csr(adj, exclude, N, torch.device("cuda"))
    return (None, None) if rowptr is None else (rowptr.cpu(), col.cpu())


@pytest.mark.parametrize("symmetric", [True, False])
@pytest.mark.parametrize("method", METHODS)
def test_recommend_matches_dense_rows(method, symmetric):
    from plnlp_b200 import heuristics
    adj = _adj(symmetric)
    nodes = _nodes()
    S = _dense(adj, symmetric, method, nodes.cpu())
    assert float(S[0].max()) > 0 and float(S[NODES.index(N - 1)].abs().max()) == 0
    for exclude in (None, "adj", _exclude_edges()):
        rowptr, col = _known(adj, exclude)
        for exclude_self in (True, False):
            Sm = ranking.mask_scores(S, nodes.cpu(), rowptr, col, exclude_self)
            for k in (1, 20, 1024):
                ids, sc = heuristics.recommend(adj, nodes, k, method, exclude, exclude_self)
                assert ids.dtype == torch.int64 and sc.dtype == torch.float32 and ids.shape == (len(NODES), k)
                wi, ws = ranking.topk_rows(Sm, k)
                assert torch.equal(ids.cpu(), wi), (exclude, exclude_self, k)
                assert torch.equal(sc.cpu(), ws), (exclude, exclude_self, k)


@pytest.mark.parametrize("symmetric", [True, False])
@pytest.mark.parametrize("method", METHODS)
def test_scores_against_oracle_and_chunking(method, symmetric):
    from plnlp_b200 import heuristics
    adj = _adj(symmetric)
    nodes = _nodes()
    ids, sc = heuristics.recommend(adj, nodes, 1024, method, "adj")
    rowptr, col, _ = _adj(symmetric, "cpu").csr()
    sets = oh.neighbour_sets(rowptr, col, N)
    pairs = torch.stack([nodes.cpu().repeat_interleave(1024), ids.cpu().reshape(-1)], 1)
    want = torch.from_numpy(oh.score_sets(sets, pairs, method).astype(np.float32)).reshape(len(NODES), 1024)
    got = sc.cpu()
    assert torch.equal(got, want) if method == "CN" else _ulp_close(got, want)
    for bs in (1, 7):
        i2, s2 = heuristics.recommend(adj, nodes, 1024, method, "adj", batch_size=bs)
        assert torch.equal(i2, ids) and torch.equal(s2, sc), bs
    i3, s3 = heuristics.recommend(adj, nodes, 1024, method, "adj")
    assert torch.equal(i3, ids) and torch.equal(s3, sc)


def _rank_edges(adj):
    """sources NODES; targets: a neighbour (a known link), a score-0 node, the source itself, random nodes"""
    rowptr, col, _ = adj.csr()
    rowptr, col = rowptr.cpu(), col.cpu()
    g = torch.Generator().manual_seed(8)
    src, tgt = [], []
    for u in NODES:
        nb = col[int(rowptr[u]):int(rowptr[u + 1])].tolist()
        ts = ([nb[0]] if nb else []) + [N - 2, u] + torch.randint(0, N, (4,), generator=g).tolist()
        src += [u] * len(ts)
        tgt += ts
    return torch.tensor([src, tgt], dtype=torch.int64).t().contiguous().cuda()


@pytest.mark.parametrize("symmetric", [True, False])
@pytest.mark.parametrize("method", METHODS)
def test_rank_against_all_matches_filtered_ranks(method, symmetric):
    from plnlp_b200 import heuristics
    adj = _adj(symmetric)
    edges = _rank_edges(adj)
    src = edges[:, 0].cpu()
    S = _dense(adj, symmetric, method, torch.tensor(NODES))
    rows = S[torch.tensor([NODES.index(u) for u in src.tolist()])]
    assert (rows[torch.arange(src.numel()), edges[:, 1].cpu()] == 0).any()      # score-0 targets are covered
    for exclude in (None, "adj", _exclude_edges()):
        rowptr, col = _known(adj, exclude)
        for exclude_self in (True, False):
            got = heuristics.rank_against_all(adj, edges, method, exclude, exclude_self)
            want = ranking.filtered_ranks(rows, edges[:, 1].cpu(), src, rowptr, col, exclude_self)
            assert got.dtype == torch.float32 and torch.equal(got.cpu().double(), want), (exclude, exclude_self)
            assert torch.equal(heuristics.rank_against_all(adj, edges, method, exclude, exclude_self, batch_size=7),
                               got)


@pytest.mark.parametrize("symmetric", [True, False])
@pytest.mark.parametrize("method", METHODS)
def test_candidates(method, symmetric):
    from plnlp_b200 import heuristics
    adj = _adj(symmetric)
    nodes = _nodes()
    g = torch.Generator().manual_seed(12)
    cand = torch.cat([torch.randint(0, N, (3000,), generator=g), torch.tensor([0, 5, N - 1, 5])])
    S = _dense(adj, symmetric, method, nodes.cpu())
    rowptr, col = _known(adj, "adj")
    for k in (1, 20, 1024):
        ids, sc = heuristics.recommend(adj, nodes, k, method, "adj", candidates=cand.cuda())
        wi, ws = ranking.topk_rows(rc.mask_candidates(S, nodes.cpu(), cand, rowptr, col), k)
        assert torch.equal(ids.cpu(), wi) and torch.equal(sc.cpu(), ws), k
        a = heuristics.recommend(adj, nodes, k, method, "adj", candidates=torch.arange(N))
        b = heuristics.recommend(adj, nodes, k, method, "adj")
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]), k
    edges = _rank_edges(adj)                            # most targets lie outside the candidate set
    src = edges[:, 0].cpu()
    rows = S[torch.tensor([NODES.index(u) for u in src.tolist()])]
    got = heuristics.rank_against_all(adj, edges, method, "adj", candidates=cand, batch_size=5)
    want = rc.filtered_ranks(rows, edges[:, 1].cpu(), src, cand, rowptr, col)
    assert torch.equal(got.cpu().double(), want)
    assert torch.equal(heuristics.rank_against_all(adj, edges, method, "adj", candidates=torch.arange(N)),
                       heuristics.rank_against_all(adj, edges, method, "adj"))
    empty = torch.empty(0, dtype=torch.int64)
    ids, sc = heuristics.recommend(adj, nodes, 3, method, candidates=empty)
    assert (ids == -1).all() and torch.isinf(sc).all()
    assert (heuristics.rank_against_all(adj, edges, method, candidates=empty) == 1).all()


@pytest.mark.parametrize("symmetric", [True, False])
def test_mark_bitmap_against_reach_set(symmetric):
    from plnlp_b200 import _ops, heuristics
    adj = _adj(symmetric)
    t = heuristics.neighbour_table(adj)
    rr, rcol = t.reach()
    nodes = _nodes()
    cpu = [x.cpu() for x in (t.rowptr, t.col, rr, rcol)]
    cand = torch.unique(torch.randint(0, N, (2000,), generator=torch.Generator().manual_seed(3))).cuda()
    for W, col0, cd in ((N, 0, None), (5000, 4001, None), (cand.numel(), 0, cand)):
        got = _ops.two_hop_mark_raw(t.rowptr, t.col, rr, rcol, nodes, W, col0, cd)
        want = ref_mark(*cpu, nodes.cpu(), W, col0, None if cd is None else cd.cpu())
        assert bitmap_columns(got, W) == bitmap_columns(want, W), (W, col0)
        S = _ops.two_hop_score_raw(t.rowptr, t.col, t.weight("RA"), nodes, got, W, col0, cd)
        js = torch.arange(col0, col0 + W, device="cuda") if cd is None else cd
        pairs = torch.stack([nodes.repeat_interleave(W), js.repeat(nodes.numel())], 1)
        assert torch.equal(S.reshape(-1), heuristics.score_edges(adj, pairs, "RA"))
        S64 = _ops.two_hop_score_raw(t.rowptr, t.col, t.weight("AA"), nodes, got, W, col0, cd, torch.float64)
        assert torch.equal(S64.reshape(-1), _ops.link_heuristic_raw(t.rowptr, t.col, t.weight("AA"), pairs))


def test_abi_error_codes():
    from plnlp_b200 import _lib
    lib = _lib.load()
    st = _lib.stream()
    p = _lib.ptr
    rowptr = torch.zeros(11, dtype=torch.int64, device="cuda")
    col = torch.zeros(4, dtype=torch.int32, device="cuda")
    nodes = torch.zeros(3, dtype=torch.int64, device="cuda")
    item = torch.zeros(4, dtype=torch.int64, device="cuda")
    cand = torch.arange(5, dtype=torch.int64, device="cuda")
    bm = torch.zeros(3, 1, dtype=torch.int32, device="cuda")
    s32 = torch.zeros(3, 5, dtype=torch.float32, device="cuda")
    s64 = torch.zeros(3, 5, dtype=torch.float64, device="cuda")
    m = lib.plnlp_two_hop_mark
    assert m(p(rowptr), p(col), p(rowptr), p(col), 10, p(nodes), p(item), 3, 0, 5, None, p(bm), st) == 0
    assert m(p(rowptr), p(col), p(rowptr), p(col), 10, p(nodes), p(item), 3, 0, 5, p(cand), p(bm), st) == 0
    assert m(None, p(col), p(rowptr), p(col), 10, p(nodes), p(item), 3, 0, 5, None, p(bm), st) == -1
    assert m(p(rowptr), p(col), None, p(col), 10, p(nodes), p(item), 3, 0, 5, None, p(bm), st) == -1
    assert m(p(rowptr), p(col), p(rowptr), p(col), 10, p(nodes), None, 3, 0, 5, None, p(bm), st) == -1
    assert m(p(rowptr), p(col), p(rowptr), p(col), 10, p(nodes), p(item), 3, 0, 5, None, None, st) == -1
    assert m(p(rowptr), p(col), p(rowptr), p(col), -1, p(nodes), p(item), 3, 0, 5, None, p(bm), st) == -2
    assert m(p(rowptr), p(col), p(rowptr), p(col), 10, p(nodes), p(item), -1, 0, 5, None, p(bm), st) == -2
    assert m(p(rowptr), p(col), p(rowptr), p(col), 10, p(nodes), p(item), 3, -1, 5, None, p(bm), st) == -2
    assert m(p(rowptr), p(col), p(rowptr), p(col), 10, p(nodes), p(item), 3, 2, 5, p(cand), p(bm), st) == -4
    assert m(None, None, None, None, 10, None, None, 0, 0, 5, None, None, st) == 0          # nothing to mark
    assert int(bm.abs().sum()) == 0
    for f, s in ((lib.plnlp_two_hop_score_f32, s32), (lib.plnlp_two_hop_score_f64, s64)):
        assert f(p(rowptr), p(col), 10, 4, None, p(nodes), 3, 0, 5, None, p(bm), p(s), 5, st) == 0
        assert f(p(rowptr), p(col), 10, 4, None, p(nodes), 3, 0, 5, p(cand), p(bm), p(s), 5, st) == 0
        assert f(None, p(col), 10, 4, None, p(nodes), 3, 0, 5, None, p(bm), p(s), 5, st) == -1
        assert f(p(rowptr), p(col), 10, 4, None, None, 3, 0, 5, None, p(bm), p(s), 5, st) == -1
        assert f(p(rowptr), p(col), 10, 4, None, p(nodes), 3, 0, 5, None, None, p(s), 5, st) == -1
        assert f(p(rowptr), p(col), 10, 4, None, p(nodes), 3, 0, 5, None, p(bm), None, 5, st) == -1
        assert f(p(rowptr), None, 10, 0, None, p(nodes), 3, 0, 5, None, p(bm), p(s), 5, st) == 0   # no entries
        assert f(p(rowptr), p(col), 10, 4, None, p(nodes), 3, 0, 5, None, p(bm), p(s), 4, st) == -2  # lds < W
        assert f(p(rowptr), p(col), -1, 4, None, p(nodes), 3, 0, 5, None, p(bm), p(s), 5, st) == -2
        assert f(p(rowptr), p(col), 10, 4, None, p(nodes), -3, 0, 5, None, p(bm), p(s), 5, st) == -2
        assert f(p(rowptr), p(col), 10, 4, None, p(nodes), 3, 1, 5, p(cand), p(bm), p(s), 5, st) == -4
        assert f(None, None, 10, 4, None, None, 0, 0, 5, None, None, None, 5, st) == 0          # Qc = 0
    torch.cuda.synchronize()
    assert int(s32.abs().sum()) == 0 and int(s64.abs().sum()) == 0


def _virtual(adj, n, R, method, nodes, edges, k, exclude, cand):
    """recommend / rank_against_all through R RankShards in one process, the collectives done by hand"""
    from plnlp_b200 import _ops, heuristics, parallel, recommend
    from plnlp_b200.graph import CSRGraph
    cs = None if cand is None else recommend.candidate_set(cand, n, "cuda")
    shards = []
    for r in range(R):
        sadj = parallel.shard_graph(adj, r, R, CSRGraph)
        lo, hi = parallel.row_block(n, r, R)
        table = heuristics.shard_table(sadj.local, sadj.local_t, lo, hi, n)
        rowptr, col = recommend.shard_exclude_csr(exclude, lo, hi, n, sadj.local_t)
        shards.append(heuristics.RankShard(table, method, n, r, R, rowptr, col, True, cs))

    def exchange(q):
        parts = [sh.partial(q) for sh in shards]
        return [p for p, _ in parts], [sh.combine(torch.stack([parts[r][1][s] for r in range(R)]))
                                       for s, sh in enumerate(shards)]
    P, S = exchange(nodes)
    tops = [sh.topk(S[s], nodes, k) for s, sh in enumerate(shards)]
    ids, sc = _ops.topk_merge_raw(torch.stack([t[0] for t in tops]), torch.stack([t[1] for t in tops]), k)
    q, t = edges[:, 0].contiguous(), edges[:, 1].contiguous()
    P, S = exchange(q)
    ts = heuristics.RankShard.target_scores(torch.stack([sh.ranker.target_values(P[s], q, t)
                                                         for s, sh in enumerate(shards)]))
    c = sum(sh.counts(S[s], q, t, ts) for s, sh in enumerate(shards))
    return ids, sc, 0.5 * (c[0].float() + c[1].float()) + 1.0


@pytest.mark.parametrize("symmetric", [True, False])
def test_virtual_shards(symmetric):
    from plnlp_b200 import heuristics, parallel
    adj = _adj(symmetric)
    nodes, edges = _nodes(), _rank_edges(adj)
    small = _small_adj()
    cases = [(adj, N, R, nodes, edges, 20) for R in (1, 2, 3)] + [
        (small, 4, 3, torch.tensor([0, 1, 3, 2], device="cuda"), torch.tensor([[0, 2], [3, 1], [1, 1]], device="cuda"), 3)]
    assert parallel.row_block(4, 2, 3)[0] == parallel.row_block(4, 2, 3)[1]          # an empty last block
    for a, n, R, nd, ed, k in cases:
        for m in METHODS:
            for exclude, cand in ((None, None), ("adj", None), ("adj", torch.arange(0, n, 3))):
                want_i, want_s = heuristics.recommend(a, nd, k, m, exclude, candidates=cand)
                want_r = heuristics.rank_against_all(a, ed, m, exclude, candidates=cand)
                ids, sc, ranks = _virtual(a, n, R, m, nd, ed, k, exclude, cand)
                if m == "CN" or R == 1:
                    assert torch.equal(ids, want_i) and torch.equal(sc, want_s), (R, m, exclude)
                    assert torch.equal(ranks, want_r), (R, m, exclude)
                else:
                    fin = torch.isfinite(want_s)
                    assert torch.equal(fin, torch.isfinite(sc))
                    assert _ulp_close(sc[fin].cpu(), want_s[fin].cpu()), (R, m, exclude)
                    # an id may differ only where the single-GPU scores of two candidates lie within an ulp
                    S = _dense(a, symmetric, m, nd.cpu()) if n == N else None
                    if S is not None:
                        got_single = S.gather(1, ids.cpu().clamp_min(0))
                        assert _ulp_close(got_single[fin.cpu()], want_s[fin].cpu())


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
            nodes, edges = _nodes(dev), _rank_edges(adj).to(dev)
            cand = torch.arange(0, N, 5, device=dev)
            for m in METHODS:
                for c in (None, cand):
                    key = (symmetric, m, c is not None)
                    out[key] = ([x.cpu() for x in heuristics.recommend(sadj, nodes, 50, m, "adj", True, 4, c)]
                                + [heuristics.rank_against_all(sadj, edges, m, "adj", True, 9, c).cpu()],
                                [x.cpu() for x in heuristics.recommend(adj, nodes, 50, m, "adj", True, None, c)]
                                + [heuristics.rank_against_all(adj, edges, m, "adj", True, None, c).cpu()])
        try:
            heuristics.recommend(sadj, nodes, 50, "CN" if rank == 0 else "RA")
            out["mismatch"] = None if ws > 1 else "ok"
        except ValueError as err:
            out["mismatch"] = str(err)
        ret[rank] = out
    finally:
        dist.destroy_process_group()


def _check(ret, ws):
    for r in range(ws):
        out = ret[r]
        for key, (got, single) in ((k, v) for k, v in out.items() if isinstance(k, tuple)):
            if key[1] == "CN" or ws == 1:
                assert all(torch.equal(a, b) for a, b in zip(got, single)), (r, key)
            else:
                fin = torch.isfinite(single[1])
                assert _ulp_close(got[1][fin], single[1][fin]), (r, key)
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

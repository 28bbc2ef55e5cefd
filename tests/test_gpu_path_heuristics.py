"""GPU tests of the path-based link scores Katz and PPR (plnlp_b200/paths.py, csrc/propagate.cu): the kernel bit for
bit against the exact restatement of the hop rule (tests/path_oracle.py) for B = 32 .. 256 on graphs with empty rows,
isolated nodes, self loops, duplicate entries, hub rows longer than PROP_CHUNK, a non-symmetric adjacency and padding
columns; the live map against reading every row; the fp64 series; batch and run invariance; a gcn-normalized
adjacency; recommend / rank_against_all against a selection on the restatement's scores; candidates, exclude and
exclude_self; one process playing every shard of R = 1, 2, 3; a one-rank NCCL run of the collective calls; and
``heuristics.test``."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests import path_oracle as po
from tests.test_path_heuristics_cpu import PARAMS, _oracle_calls, method_obj

pytestmark = pytest.mark.gpu

N, N_ISOLATED = 900, 40


def _coo(symmetric, seed=0):
    """random graph on N nodes: the last N_ISOLATED isolated; every other node links to node 3 (R(3) spans several
    work items) and node 5 links to every second node (a long row of N); self loops and duplicates; on the
    non-symmetric graph the nodes just below the isolated ones have no row of their own (an empty row)"""
    g = torch.Generator().manual_seed(seed)
    m = N - N_ISOLATED
    src = torch.cat([torch.randint(0, m, (2500,), generator=g), torch.arange(m), torch.full((m // 2,), 5),
                     torch.arange(50)])
    dst = torch.cat([torch.randint(0, m, (2500,), generator=g), torch.full((m,), 3), torch.arange(0, m, 2),
                     torch.arange(50)])
    src, dst = torch.cat([src, src[:300]]), torch.cat([dst, dst[:300]])
    if symmetric:
        return torch.cat([src, dst]), torch.cat([dst, src])
    keep = (src < m - 20) | (src == dst)
    return src[keep], dst[keep]


def _adj(symmetric, dev="cuda"):
    from plnlp_b200.graph import CSRGraph
    src, dst = _coo(symmetric)
    v = torch.rand(src.numel(), generator=torch.Generator().manual_seed(1))
    return CSRGraph.from_coo(src.to(dev), dst.to(dev), v.to(dev), (N, N))


_SETS = {}


def _sets(symmetric):
    if symmetric not in _SETS:
        _SETS[symmetric] = po.sets_of(_adj(symmetric, "cpu"))
    return _SETS[symmetric]


def _bits(t):
    return np.ascontiguousarray(t.cpu().numpy() if isinstance(t, torch.Tensor) else t).view(np.uint32)


def _sources(B):
    """B columns: the hub, an isolated node, a node with an empty row, a repeat, random nodes, 5 padding columns"""
    g = torch.Generator().manual_seed(B)
    fixed = torch.tensor([3, 5, N - 1, N - N_ISOLATED - 6, 3, 0])
    rest = torch.randint(0, N, (B - fixed.numel() - 5,), generator=g)
    return torch.cat([fixed, rest, torch.full((5,), -1)])


def test_graph_has_the_shapes_the_kernel_must_handle():
    from plnlp_b200 import paths
    for symmetric in (True, False):
        sets = _sets(symmetric)
        R = po.reach_lists(sets)
        assert max(len(r) for r in R) > 2 * paths.PROP_CHUNK
        assert all(not s for s in sets[N - N_ISOLATED:]) and all(not r for r in R[N - N_ISOLATED:])
    sets = _sets(False)
    assert not sets[N - N_ISOLATED - 6] and po.reach_lists(sets)[N - N_ISOLATED - 6]   # no row of its own, reached


@pytest.mark.parametrize("symmetric", [True, False])
@pytest.mark.parametrize("B", [32, 64, 128, 256])
def test_kernel_bit_identical_to_exact_restatement(B, symmetric):
    from plnlp_b200 import paths
    adj = _adj(symmetric)
    shard = paths.path_shard(adj)
    all_live = paths.PathShard(shard.rowptr, shard.col, 0, N, N, inv_deg=shard.inv_deg, live=False)
    src = _sources(B)
    for name in ("Katz", "PPR"):
        p = dict(PARAMS[name], **({"T": 8} if name == "PPR" else {}))
        m = method_obj(name) if name == "Katz" else type(method_obj(name))(p["alpha"], p["T"])
        want = po.propagate_exact(_sets(symmetric), src.numpy(), name, **p)
        x, live = paths.propagate(shard, src.cuda(), m)
        assert np.array_equal(_bits(x), _bits(want)), name
        assert np.array_equal(live.cpu().numpy().astype(bool), (want != 0).any(1)), name
        assert not x[:, -5:].any()                                       # padding columns stay zero
        x2, live2 = paths.propagate(all_live, src.cuda(), m)
        assert torch.equal(x2, x) and torch.equal(live2, live), name


@pytest.mark.parametrize("B", [32, 256])
def test_one_hop_of_a_row_range_with_random_state(B):
    """one hop from an arbitrary non-negative state and weights, for the rows [lo, hi), from a strided state"""
    from plnlp_b200 import _ops, graph, paths
    shard = paths.path_shard(_adj(False))
    rowptr, col = shard.rowptr.cpu(), shard.col.cpu()
    lo, hi = 2, 700                                                       # holds the hub row R(3)
    g = torch.Generator().manual_seed(5)
    wide = torch.rand(N, B + 8, generator=g) * (torch.rand(N, 1, generator=g) < 0.6)   # 40 % zero rows
    x = wide[:, :B]
    weight = torch.rand(N, dtype=torch.float64, generator=g) * 3
    src = torch.randint(0, hi + 50, (B,), generator=g)
    c, b = 0.37, 0.91
    sub_ptr = rowptr[lo:hi + 1] - rowptr[lo]
    sub_col = col[int(rowptr[lo]):int(rowptr[hi])]
    plan = graph.build_plan(sub_ptr.cuda(), sub_col.cuda(), None, hi - lo, N, chunk=paths.PROP_CHUNK)
    live_in = (x != 0).any(1).to(torch.uint8)
    R = [None] * lo + [sub_col[sub_ptr[i]:sub_ptr[i + 1]].tolist() for i in range(hi - lo)]
    for w in (None, weight):
        want = po.hop_exact(R, None if w is None else w.numpy(), x.numpy(), src.numpy(), c, b, lo, hi)
        for live in (live_in, None):
            y, lv = _ops.propagate_raw(plan, None if w is None else w.cuda(), wide.cuda()[:, :B], src.cuda(), c, b,
                                       None if live is None else live.cuda(), lo)
            assert np.array_equal(_bits(y), _bits(want))
            assert np.array_equal(lv.cpu().numpy().astype(bool), (want != 0).any(1))
    assert plan.n_fix > 0                                                 # the hub row went through the second pass


def test_abi_error_codes():
    from plnlp_b200 import _ops, paths
    shard = paths.path_shard(_adj(True))
    plan = shard.plan()
    x = torch.zeros(N, 129, device="cuda")
    src = torch.zeros(48, dtype=torch.int64, device="cuda")
    with pytest.raises(RuntimeError, match="invalid argument"):          # B must be 32, 64, 128 or 256
        _ops.propagate_raw(plan, None, x[:, :48], src, 1.0, 0.0)
    with pytest.raises(RuntimeError, match="invalid argument"):          # misaligned for 4-wide accesses
        _ops.propagate_raw(plan, None, x[:, 1:129], torch.zeros(128, dtype=torch.int64, device="cuda"), 1.0, 0.0)
    with pytest.raises(RuntimeError):
        _ops.propagate_raw(plan, torch.zeros(N, device="cuda"), x[:, :32], src[:32], 1.0, 0.0)


def _edges(seed=2, P=3000):
    g = torch.Generator().manual_seed(seed)
    e = torch.randint(0, N, (P, 2), generator=g)
    e[:50, 1] = e[:50, 0]                                                 # (u, u) pairs
    return e


@pytest.mark.parametrize("symmetric", [True, False])
def test_scores_against_fp64_series_and_invariance(symmetric):
    from plnlp_b200 import heuristics
    from plnlp_b200.utils import gcn_normalization
    adj = _adj(symmetric)
    e = _edges()
    us = torch.unique(e[:, 0])
    pos = torch.searchsorted(us, e[:, 0])
    for name in ("Katz", "PPR"):
        ref = (po.katz_fp64 if name == "Katz" else po.ppr_fp64)(_sets(symmetric), us.numpy())
        want = ref[pos.numpy(), e[:, 1].numpy()]
        got = heuristics.score_edges(adj, e.cuda(), name)
        g = got.cpu().numpy().astype(np.float64)
        assert np.all(np.abs(g - want) <= 1e-5 * np.abs(want)), name
        for bs in (1, 64, 200, 256, 10 ** 6):
            assert torch.equal(heuristics.score_edges(adj, e.cuda(), name, bs), got), (name, bs)
        assert torch.equal(heuristics.score_edges(adj, e.cuda(), name), got)              # run to run
        assert torch.equal(heuristics.score_edges(gcn_normalization(adj), e.cuda(), name), got)
        assert torch.equal(heuristics.score_edges(adj, e.cuda(), heuristics.path_method(name)), got)


def _calls_args(symmetric):
    g = torch.Generator().manual_seed(7)
    nodes = torch.cat([torch.tensor([3, 5, N - 1, N - N_ISOLATED - 6]), torch.randint(0, N, (36,), generator=g)])
    edges = torch.stack([nodes, torch.randint(0, N, (40,), generator=g)], 1)
    edges[0, 1] = 3
    exclude = torch.randint(0, N, (4000, 2), generator=g)
    cand = torch.randint(0, N, (300,), generator=g)
    return nodes, edges, exclude, cand


@pytest.mark.parametrize("symmetric", [True, False])
@pytest.mark.parametrize("name", ["Katz", "PPR"])
def test_recommend_and_rank_against_exact_selection(name, symmetric):
    from plnlp_b200 import heuristics
    adj, adj_cpu = _adj(symmetric), _adj(symmetric, "cpu")
    m = method_obj(name)
    nodes, edges, exclude, cand = _calls_args(symmetric)
    for ex in (None, exclude):
        for c in (None, cand):
            ids, sc, ranks = _oracle_calls(adj_cpu, N, name, nodes, edges, 20, ex, c)
            gi, gs = heuristics.recommend(adj, nodes.cuda(), 20, m, None if ex is None else ex.cuda(), True, 32,
                                          None if c is None else c.cuda())
            assert torch.equal(gi.cpu(), ids) and torch.equal(gs.cpu(), sc), (ex is None, c is None)
            gr = heuristics.rank_against_all(adj, edges.cuda(), m, None if ex is None else ex.cuda(), True, 64,
                                             None if c is None else c.cuda())
            assert torch.equal(gr.cpu(), ranks), (ex is None, c is None)
    # every returned score is score_edges of its pair, bit for bit
    gi, gs = heuristics.recommend(adj, nodes.cuda(), 50, m, "adj")
    ok = gi >= 0
    pairs = torch.stack([nodes.cuda()[:, None].expand_as(gi)[ok], gi[ok]], 1)
    assert torch.equal(heuristics.score_edges(adj, pairs, m), gs[ok])
    # the adjacency's own rows are excluded, and the query itself unless exclude_self=False
    sets = _sets(symmetric)
    for q, row in zip(nodes.tolist(), gi.cpu().tolist()):
        assert q not in row and not (set(row) & sets[q])
    gi2, gs2 = heuristics.recommend(adj, nodes.cuda(), 50, m, None, False)
    assert any(q in row for q, row in zip(nodes.tolist(), gi2.cpu().tolist()))
    # candidates = every node is the call without candidates, bit for bit
    every = torch.arange(N, device="cuda")
    for bs in (None, 32, 100):
        a = heuristics.recommend(adj, nodes.cuda(), 20, m, "adj", True, bs)
        b = heuristics.recommend(adj, nodes.cuda(), 20, m, "adj", True, bs, every)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
        assert torch.equal(heuristics.rank_against_all(adj, edges.cuda(), m, "adj", True, bs),
                           heuristics.rank_against_all(adj, edges.cuda(), m, "adj", True, bs, every))


def _virtual(adj, R, m, nodes, edges, k, exclude, cand):
    """the four calls' results with one process playing every rank of R: per-rank hop steps on the all-gathered
    state, the owner's score readout, the common-neighbour calls' per-rank tail and the merge"""
    from plnlp_b200 import _ops, heuristics, parallel, paths
    from plnlp_b200 import recommend as rec
    from plnlp_b200.graph import CSRGraph
    n = N
    sadjs = [parallel.shard_graph(adj, r, R, CSRGraph) for r in range(R)]
    shards, degs = [], []
    for r, sadj in enumerate(sadjs):
        lo, hi = parallel.row_block(n, r, R)
        rowptr, col, deg = paths.reach_rows(sadj.local, sadj.local_t, lo, hi, n)
        shards.append(paths.PathShard(rowptr, col, lo, hi, n, sadj.blk))
        degs.append(torch.cat([deg, deg.new_zeros(sadj.blk - deg.numel())]))
    inv = heuristics.weight_table(torch.cat(degs), "RA")[:n].contiguous()
    for sh in shards:
        sh.inv_deg = inv

    def run(src):
        blocks = [sh.start(src) for sh in shards]
        for c, b, weighted in paths.hops(m):
            xf, lf = torch.cat([x for x, _ in blocks]), torch.cat([lv for _, lv in blocks])
            blocks = [sh.hop(xf, lf, src, c, b, weighted) for sh in shards]
        return [x for x, _ in blocks]

    B = 64
    dev = nodes.device
    scores = torch.zeros(edges.size(0), device=dev)
    for srcs, sel, col in paths.source_blocks(edges[:, 0], B):
        xs = run(paths.padded(srcs, B))
        for sh, x in zip(shards, xs):
            v = edges[sel, 1]
            own = (v >= sh.lo) & (v < sh.hi)
            scores[sel[own]] += x[v[own] - sh.lo, col[own]]
    tails = []
    for r, sh in enumerate(shards):
        rp, cl = rec.shard_exclude_csr(exclude, sh.lo, sh.hi, n, sadjs[r].local_t)
        tails.append(heuristics.RankShard(None, "CN", n, r, R, rp, cl, True, cand))
    Q = nodes.numel()
    ids = torch.empty(Q, k, dtype=torch.int64, device=dev)
    sc = torch.empty(Q, k, device=dev)
    for i in range(0, Q, B):
        q = nodes[i:i + B]
        xs = run(paths.padded(q, B))
        parts = [t.topk(paths._rank_chunk(x, q.numel(), t), q, k) for t, x in zip(tails, xs)]
        ids[i:i + B], sc[i:i + B] = _ops.topk_merge_raw(torch.stack([a for a, _ in parts]),
                                                        torch.stack([b for _, b in parts]), k)
    ranks = torch.empty(edges.size(0), device=dev)
    for i in range(0, edges.size(0), B):
        q, t = edges[i:i + B, 0], edges[i:i + B, 1]
        xs = run(paths.padded(q, B))
        ts = torch.zeros(q.numel(), device=dev)
        for sh, x in zip(shards, xs):
            own = (t >= sh.lo) & (t < sh.hi)
            ts[own] = x[t[own] - sh.lo, torch.arange(q.numel(), device=dev)[own]]
        cnt = sum(tl.counts(paths._rank_chunk(x, q.numel(), tl), q, t, ts) for tl, x in zip(tails, xs))
        ranks[i:i + B] = 0.5 * (cnt[0].float() + cnt[1].float()) + 1.0
    return scores, (ids, sc), ranks


@pytest.mark.parametrize("symmetric", [True, False])
def test_virtual_shards_bit_identical_to_one_gpu(symmetric):
    from plnlp_b200 import heuristics
    adj = _adj(symmetric)
    nodes, edges, exclude, cand = _calls_args(symmetric)
    nodes, edges, exclude = nodes.cuda(), edges.cuda(), exclude.cuda()
    for name in ("Katz", "PPR"):
        m = heuristics.path_method(name)
        for c in (None, torch.unique(cand).cuda()):
            want = (heuristics.score_edges(adj, edges, m), heuristics.recommend(adj, nodes, 10, m, exclude, True, 64, c),
                    heuristics.rank_against_all(adj, edges, m, exclude, True, 64, c))
            for R in (1, 2, 3):
                s, (i, sc), r = _virtual(adj, R, m, nodes, edges, 10, exclude, c)
                assert torch.equal(s, want[0]), (name, R)
                assert torch.equal(i, want[1][0]) and torch.equal(sc, want[1][1]), (name, R)
                assert torch.equal(r, want[2]), (name, R)


class _Data:
    pass


@pytest.mark.parametrize("metric", ["hits", "mrr"])
def test_heuristics_test_matches_metric_code(metric):
    from plnlp_b200 import heuristics
    from plnlp_b200.utils import evaluate_hits, evaluate_mrr, get_pos_neg_edges
    g = torch.Generator().manual_seed(9)
    if metric == "hits":
        split = {s: {"edge": torch.randint(0, N, (300, 2), generator=g),
                     "edge_neg": torch.randint(0, N, (500, 2), generator=g)} for s in ("valid", "test")}
        split["train"] = {"edge": torch.zeros(1, 2, dtype=torch.int64)}
    else:
        split = {s: {"source_node": torch.randint(0, 40, (200,), generator=g),
                     "target_node": torch.randint(0, N, (200,), generator=g),
                     "target_node_neg": torch.randint(0, N, (200, 50), generator=g)} for s in ("valid", "test")}
        split["train"] = {"source_node": torch.zeros(1, dtype=torch.int64)}
    data = _Data()
    data.adj_t = _adj(True)
    name = "PPR"
    p = dict(alpha=0.15, T=30)
    preds = []
    for s in ("valid", "test"):
        for e in get_pos_neg_edges(s, split, device="cpu"):
            e = e.reshape(-1, 2)
            us = torch.unique(e[:, 0])
            x = po.propagate_exact(_sets(True), us.numpy(), name, **p)
            preds.append(torch.from_numpy(x[e[:, 1].numpy(), torch.searchsorted(us, e[:, 0]).numpy()]).cuda())
    want = (evaluate_hits if metric == "hits" else evaluate_mrr)(None, *preds)
    cuda_split = {s: {k: v.cuda() for k, v in d.items()} for s, d in split.items()}
    got = heuristics.test(data, cuda_split, name, None, None, metric)
    assert got == want


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def worker(rank, ws, port, ret):
    """the collective calls on a ``ShardedAdj`` of ws ranks beside the one-GPU calls on the full graph"""
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
            nodes, edges, exclude, cand = (t.to(dev) for t in _calls_args(symmetric))
            for name in ("Katz", "PPR"):
                m = method_obj(name)
                for c in (None, cand):
                    key = (symmetric, name, c is None)
                    out[key] = [(heuristics.score_edges(sadj, edges, m, 64).cpu(),
                                 heuristics.score_edges(adj, edges, m).cpu())]
                    got = heuristics.recommend(sadj, nodes, 15, m, exclude, True, 32, c)
                    want = heuristics.recommend(adj, nodes, 15, m, exclude, True, None, c)
                    out[key] += [(got[0].cpu(), want[0].cpu()), (got[1].cpu(), want[1].cpu())]
                    out[key].append((heuristics.rank_against_all(sadj, edges, m, "adj", True, 32, c).cpu(),
                                     heuristics.rank_against_all(adj, edges, m, "adj", True, 256, c).cpu()))
        try:
            heuristics.score_edges(sadj, edges, heuristics.Katz(0.005, 3 + rank))
            out["mismatch"] = None if ws > 1 else "ok"
        except ValueError as err:
            out["mismatch"] = str(err)
        ret[rank] = out
    finally:
        dist.destroy_process_group()


def check(ret, ws):
    for r in range(ws):
        out = ret[r]
        for key, pairs in ((k, v) for k, v in out.items() if isinstance(k, tuple)):
            for got, want in pairs:
                assert torch.equal(got, want), (r, key)
        assert out["mismatch"] == "ok" if ws == 1 else "collective" in out["mismatch"]


def test_collective_one_rank_nccl():
    ret = mp.Manager().dict()
    mp.spawn(worker, args=(1, _free_port(), ret), nprocs=1, join=True)
    check(ret, 1)

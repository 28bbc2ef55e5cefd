"""GPU checks of candidate sets (-m gpu): the candidate-set mask / select (csrc/topk.cu) against the CPU rule of
tests/ranking_candidates.py bit for bit; ``recommend`` / ``rank_against_all`` with ``candidates=C`` against the same
calls with C's complement as excluded links, for every head; the per-shard step with candidate slices against the
single-GPU calls; and the collective calls on a row-partitioned model.

Bit-exact everywhere on one GPU: a candidate chunk runs the kernels of the all-node call.  Across virtual shards
DOT, the fused MLP head and MLPCAT are bit-exact; BIL, MLPDOT and MLPBIL are held to 1e-5 of the row maximum, as in
tests/test_gpu_recommend_sharded.py."""
import pytest
import torch
import torch.multiprocessing as mp

from oracle import ranking
from tests import ranking_candidates as rc
from tests.test_gpu_recommend_sharded import (Data, _check_against, _csr, _edges_for, _free_port, _local_t, _scores,
                                              _setup)

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
INF = float("inf")
HEADS = ["DOT", "BIL", "MLP", "MLPDOT", "MLPBIL", "MLPCAT"]


# ----------------------------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("ties", [False, True])
@pytest.mark.parametrize("exclude_self", [True, False])
def test_mask_and_select_on_candidate_sets(ties, exclude_self):
    from plnlp_b200 import _ops
    g = torch.Generator().manual_seed(11 + ties)
    Q, N = 23, 140001
    s = _scores(Q, N, g, ties)
    nodes = torch.randint(0, N, (Q,), generator=g)
    lists = {int(n): torch.randint(0, N, (60,), generator=g).tolist() + [int(n), N, -3] for n in nodes[::2]}
    rowptr, col = _csr(lists, N)
    target = torch.randint(0, N, (Q,), generator=g)
    ts = s[torch.arange(Q), target].clone()
    ts[::4] = 0.5
    perm = torch.randperm(N, generator=g)
    for m in (1, 7, 1023, 70000):                           # 70 000 columns: two segments of the select
        cand = torch.sort(perm[:m]).values
        if m > 1:
            cand = torch.unique(torch.cat([cand, nodes[:3], target[:5]]))       # queries and targets inside C
        masked = rc.mask_candidates(s, nodes, cand, rowptr, col, exclude_self)
        d = s[:, cand].contiguous().to(DEV)
        c = cand.to(DEV)
        _ops.score_mask_raw(d, nodes.to(DEV), rowptr.to(DEV), col.to(DEV), exclude_self, cand=c)
        want = ranking.mask_scores(s, nodes, rowptr, col, exclude_self)[:, cand]
        torch.testing.assert_close(d.cpu(), want, rtol=0, atol=0, equal_nan=True)
        r_gt, r_ge = ranking.rank_counts(masked, target, ts)
        for k in (1, 20, 1024):
            ids, sc, gt, ge = _ops.topk_rows_raw(d, k, target=target.to(DEV), target_score=ts.to(DEV), cand=c)
            r_ids, r_sc = ranking.topk_rows(masked, k)
            assert torch.equal(ids.cpu(), r_ids) and torch.equal(sc.cpu(), r_sc), (m, k)
            assert torch.equal(gt.cpu(), r_gt) and torch.equal(ge.cpu(), r_ge), (m, k)


def test_candidate_entry_points_reject_invalid_arguments():
    from plnlp_b200 import _lib, _ops
    lib = _lib.load()
    s = torch.randn(4, 100, device=DEV)
    nodes = torch.zeros(4, dtype=torch.int64, device=DEV)
    cand = torch.arange(100, device=DEV)
    for bad in (cand[:99], cand.int(), cand.reshape(10, 10)):
        with pytest.raises(RuntimeError):
            _ops.topk_rows_raw(s, 5, cand=bad)
        with pytest.raises(RuntimeError):
            _ops.score_mask_raw(s, nodes, cand=bad)
    with pytest.raises(RuntimeError):                       # a column offset with a candidate set
        _ops.topk_rows_raw(s, 5, col0=3, cand=cand)
    with pytest.raises(RuntimeError):
        _lib.check(lib.plnlp_score_mask_cand_f32(s.data_ptr(), 100, 4, 100, None, nodes.data_ptr(), None, None, 1,
                                                 _lib.stream()), "plnlp_score_mask_cand_f32")


# ----------------------------------------------------------------------------------------------- model level
def _adj_edges(adj):
    rowptr, col, _ = adj.csr()
    src = torch.repeat_interleave(torch.arange(rowptr.numel() - 1, device=col.device), rowptr[1:] - rowptr[:-1])
    return torch.stack([src, col.to(torch.int64)], 1)


def _complement(nodes, cand, n, exclude, adj):
    """the ``exclude`` links as an edge tensor plus (q, j) for every query q and every j outside cand"""
    out = torch.ones(n, dtype=torch.bool, device=DEV)
    out[cand] = False
    outside = torch.nonzero(out).reshape(-1)
    uq = torch.unique(nodes)
    parts = [torch.stack([uq.repeat_interleave(outside.numel()), outside.repeat(uq.numel())], 1)]
    if isinstance(exclude, str):
        parts.append(_adj_edges(adj))
    elif exclude is not None:
        parts.append(exclude)
    return torch.cat(parts)


def _both(model, data, nodes, edges, k, **kw):
    return (*model.recommend(data, nodes, k, **kw), model.rank_against_all(data, edges, **kw))


def _assert_same(a, b, what):
    for x, y in zip(a, b):
        assert torch.equal(x, y), what


def _pick(n, g, m, nodes, edges):
    """m candidates, among them some queries and targets, not all of either"""
    c = torch.randperm(n, generator=g)[:m].to(DEV)
    return torch.cat([c, nodes[:2], edges[5:7, 1]])


@pytest.mark.parametrize("encoder", ["SAGE", "GCN"])
@pytest.mark.parametrize("predictor", HEADS)
def test_candidates_equal_the_complement_exclusion(encoder, predictor):
    n, k = 1000, 40
    model, data = _setup(encoder, predictor, n, hid=32)
    g = torch.Generator().manual_seed(7)
    nodes = torch.randint(0, n, (19,), generator=g).to(DEV)
    edges = _edges_for(nodes, n, g)
    known = torch.stack([nodes.repeat_interleave(15), torch.randint(0, n, (19 * 15,), generator=g).to(DEV)], 1)
    edges[4, 1] = known[4 * 15, 1]                           # a known link as target: never filtered
    cand = _pick(n, g, 300, nodes, edges)
    for exclude, exclude_self in ((None, True), ("adj", True), (known, False)):
        got = _both(model, data, nodes, edges, k, exclude=exclude, exclude_self=exclude_self, candidates=cand)
        want = _both(model, data, nodes, edges, k, exclude=_complement(nodes, cand, n, exclude, data.adj_t),
                     exclude_self=exclude_self)
        _assert_same(got, want, (predictor, encoder, exclude_self))
        for bs in (1, 7):
            _assert_same(_both(model, data, nodes, edges, k, exclude=exclude, exclude_self=exclude_self,
                               candidates=cand, batch_size=bs), got, (predictor, bs))
    every = torch.arange(n - 1, -1, -1, device=DEV)         # C = every node, in any order
    _assert_same(_both(model, data, nodes, edges, k, exclude="adj", candidates=every),
                 _both(model, data, nodes, edges, k, exclude="adj"), (predictor, "all nodes"))


@pytest.mark.parametrize("predictor", ["DOT", "MLP"])
def test_candidates_on_the_tensor_core_shape(predictor):
    """N = 20 000, H = 64: gemm_backend picks the tensor-core kernel (MLP: the fused edge-MLP kernel), pinned for the
    narrow chunks of small candidate sets and the [p, p] products that score targets outside C"""
    from plnlp_b200 import _ops, recommend
    n, k = 20000, 100
    model, data = _setup("SAGE", predictor, n, hid=64, seed=2)
    g = torch.Generator().manual_seed(6)
    nodes = torch.randint(0, n, (33,), generator=g).to(DEV)
    edges = _edges_for(nodes, n, g)
    h = recommend._encode(model, data)
    for m in (1, 7, 129, 5000):
        cand = torch.randperm(n, generator=g)[:m].to(DEV)
        sc = recommend._Scorer(model, h, cand=torch.unique(cand))
        assert sc.path == ("gemm" if predictor == "DOT" else "fused_mlp")
        if predictor == "DOT":
            assert sc.backend == _ops.GEMM_BACKEND != "ffma"
        got = _both(model, data, nodes, edges, k, exclude="adj", candidates=cand)
        want = _both(model, data, nodes, edges, k, exclude=_complement(nodes, cand, n, "adj", data.adj_t))
        _assert_same(got, want, (predictor, m))
        _assert_same(_both(model, data, nodes, edges, k, exclude="adj", candidates=cand, batch_size=5), got,
                     (predictor, m, 5))


def test_empty_candidate_set_and_argument_errors():
    from plnlp_b200 import _lib
    n = 300
    model, data = _setup("GCN", "DOT", n, hid=32)
    nodes = torch.arange(5, device=DEV)
    edges = torch.stack([nodes, nodes + 1], 1)
    launches = _lib.launch_count()
    ids, sc = model.recommend(data, nodes, 7, candidates=torch.zeros(0, dtype=torch.int64))
    ranks = model.rank_against_all(data, edges, candidates=torch.zeros(0, dtype=torch.int64, device=DEV))
    assert _lib.launch_count() == launches                   # nothing scored
    assert (ids == -1).all() and (sc == -INF).all() and ids.shape == (5, 7) and ids.device.type == "cuda"
    assert (ranks == 1).all() and ranks.shape == (5,)
    short, _ = model.recommend(data, nodes, 7, candidates=torch.tensor([3, 9, 3]))   # fewer candidates than k
    assert [sorted(r) for r in short[:, :2].tolist()] == [[3, 9]] * 3 + [[-1, 9]] + [[3, 9]]   # node 3: not itself
    assert (short[:, 2:] == -1).all()
    for bad in (torch.tensor([1, 2], dtype=torch.int32), torch.tensor([[1, 2]]), torch.tensor([0, n]),
                torch.tensor([-1]), torch.tensor(4)):
        with pytest.raises(ValueError):
            model.recommend(data, nodes, 7, candidates=bad)
        with pytest.raises(ValueError):
            model.rank_against_all(data, edges, candidates=bad)


# ----------------------------------------------------------------------------------------------- virtual shards
def _virtual(model, data, h, bounds, nodes, k, edges, exclude, cand, batch_size):
    """every shard's step on its slice of the candidate set, combined as the collectives would"""
    from plnlp_b200 import _ops, recommend
    n = h.size(0) - 1
    cand = recommend.candidate_set(cand, n, DEV)
    shards = []
    for (lo, hi), (a, b) in zip(bounds, recommend.candidate_slices(cand, bounds)):
        local_t = _local_t(data.adj_t, lo, hi) if isinstance(exclude, str) else None
        rowptr, col = recommend.shard_exclude_csr(exclude, lo, hi, n, local_t)
        shards.append(recommend.Shard(model, h[lo:hi], lo, hi, n, rowptr, col, True, cand[a:b]))
    table = torch.cat([sh.table[:sh.hi - sh.lo] for sh in shards])
    ids, scores, ranks = [], [], []
    for i in range(0, nodes.numel(), batch_size):
        q = nodes[i:i + batch_size]
        lists = [sh.topk(q, table[q], k) for sh in shards]
        a, b = _ops.topk_merge_raw(torch.stack([x[0] for x in lists]), torch.stack([x[1] for x in lists]), k)
        ids.append(a)
        scores.append(b)
    src, tgt = edges[:, 0].contiguous(), edges[:, 1].contiguous()
    for i in range(0, src.numel(), batch_size):
        q, t = src[i:i + batch_size], tgt[i:i + batch_size]
        parts = [sh.target_scores(q, table[q], t) for sh in shards]
        ts = sum(x for _, x in parts)
        c = sum(sh.counts(S, q, t, ts) for sh, (S, _) in zip(shards, parts))
        ranks.append(0.5 * (c[0].float() + c[1].float()) + 1.0)
    return torch.cat(ids), torch.cat(scores), torch.cat(ranks)


@pytest.mark.parametrize("encoder", ["SAGE", "GCN"])
@pytest.mark.parametrize("predictor", HEADS)
def test_virtual_shards_with_candidates_match_single_gpu(encoder, predictor):
    from plnlp_b200 import parallel, recommend
    n, k = 1000, 40
    model, data = _setup(encoder, predictor, n, hid=32)
    g = torch.Generator().manual_seed(5)
    nodes = torch.randint(0, n, (19,), generator=g).to(DEV)
    edges = _edges_for(nodes, n, g)
    edges[7, 1] = 450                                        # a target in the block without candidates
    cand = _pick(n, g, 250, nodes, edges)
    cand = cand[(cand < 400) | (cand >= 600)]                # nothing in [400, 600)
    h = recommend._encode(model, data)
    S = recommend._Scorer(model, h).chunk(nodes)
    splits = [[parallel.row_block(n, r, R) for r in range(R)] for R in (1, 2, 3)] + [[(0, 400), (400, 600), (600, n)]]
    for exclude in (None, "adj"):
        want = _both(model, data, nodes, edges, k, exclude=exclude, candidates=cand)
        for bounds in splits:
            got = _virtual(model, data, h, bounds, nodes, k, edges, exclude, cand, 7 if len(bounds) == 3 else 19)
            eps = _check_against(predictor, got, want, S)
            if eps is not None:
                ts = S.gather(1, edges[:, 1:2])
                near = ((S - ts).abs() <= 2 * eps).sum(1)
                assert ((got[2] - want[2]).abs() <= near).all(), (predictor, bounds)


# ----------------------------------------------------------------------------------------------- collective calls
def _worker(rank, ws, port, ret):
    import os

    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=ws, device_id=dev)
    try:
        from plnlp_b200 import parallel, recommend
        from plnlp_b200.graph import CSRGraph
        from plnlp_b200.model import BaseModel
        from tests.test_gpu_recommend_sharded import _single_process
        n, k = 1001, 30
        out = {}
        for predictor in ("DOT", "MLP"):
            single, data = _setup("GCN", predictor, n, hid=32, seed=8)
            lo, hi = parallel.row_block(n, rank, ws)
            blk = parallel.block_size(n, ws)
            torch.manual_seed(0)
            part = BaseModel(lr=0.01, dropout=0.3, grad_clip_norm=2.0, gnn_num_layers=2, mlp_num_layers=2,
                             emb_hidden_channels=16, gnn_hidden_channels=32, mlp_hidden_channels=32, num_nodes=blk,
                             num_node_feats=16, gnn_encoder_name="GCN", predictor_name=predictor, loss_func="AUC",
                             optimizer_name="Adam", device=dev, use_node_feats=True, train_node_emb=True)
            with torch.no_grad():
                for a, b in zip(part.para_list, single.para_list):
                    if a.shape == b.shape:
                        a.copy_(b)
                part.emb.weight.zero_()
                part.emb.weight[: hi - lo].copy_(single.emb.weight[lo:hi])
            part.world_size, part.rank, part.partitioned = ws, rank, True
            part.num_nodes = n
            d2 = Data()
            d2.adj_t = parallel.shard_graph(data.adj_t, rank, ws, CSRGraph)
            d2.edge_index = None
            d2.x = parallel.pad_rows(data.x[lo:hi].contiguous(), blk)
            g = torch.Generator().manual_seed(9)
            nodes = torch.randint(0, n, (41,), generator=g).to(dev)
            edges = _edges_for(nodes, n, g)
            cand = torch.randperm(n, generator=g)[:200].to(dev)
            cand = cand[cand < 480]                          # rank 1 of 2 holds no candidate
            part.encoder.eval()
            part.predictor.eval()
            h = part.encode_for_test(d2)
            S = recommend._Scorer(part, h).chunk(nodes)
            res = {}
            for exclude in (None, "adj"):
                for bs in (None, 6):
                    got = (*part.recommend(d2, nodes, k, exclude=exclude, batch_size=bs, candidates=cand),
                           part.rank_against_all(d2, edges, exclude=exclude, batch_size=bs, candidates=cand))
                    want = (*_single_process(part, h, data, recommend.recommend, nodes, k, exclude,
                                             candidates=cand),
                            _single_process(part, h, data, recommend.rank_against_all, edges, exclude,
                                            candidates=cand))
                    res[f"{exclude}/{bs}"] = {"got": [t.detach().cpu() for t in got],
                                              "want": [t.detach().cpu() for t in want]}
            empty = (*part.recommend(d2, nodes, k, candidates=cand[:0]),
                     part.rank_against_all(d2, edges, candidates=cand[:0]))
            res["empty"] = {"got": [t.cpu() for t in empty],
                            "want": [t.cpu() for t in (*recommend._no_candidates(nodes.numel(), k, dev),
                                                       torch.ones(edges.size(0), device=dev))]}
            res["S"] = S.detach().cpu()
            try:                                             # a different candidate count fails on every rank
                part.recommend(d2, nodes, k, candidates=cand[:100 + rank])
                res["mismatch"] = None
            except ValueError as ex:
                res["mismatch"] = str(ex)[:40]
            out[predictor] = res
        ret[rank] = out
    finally:
        dist.destroy_process_group()


def _check_ranks(ret, ws):
    for r in range(ws):
        for predictor, res in ret[r].items():
            S = res.pop("S")
            mismatch = res.pop("mismatch")
            if ws > 1:
                assert mismatch is not None, (r, predictor)
            for key, v in res.items():
                _check_against(predictor, tuple(v["got"]), tuple(v["want"]), S)
                if r > 0:
                    for a, b in zip(v["got"], ret[0][predictor][key]["got"]):
                        assert torch.equal(a, b), (r, predictor, key)


def test_partitioned_one_rank_with_candidates():
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(1, _free_port(), ret), nprocs=1, join=True)
    _check_ranks(ret, 1)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_partitioned_two_ranks_with_candidates():
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(2, _free_port(), ret), nprocs=2, join=True)
    _check_ranks(ret, 2)

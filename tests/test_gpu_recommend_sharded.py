"""GPU checks of candidate-sharded link recommendation (-m gpu): the column-offset mask / select and the cross-shard
merge (csrc/topk.cu) against the CPU restatement (oracle/ranking.py) bit for bit; the per-shard step
(recommend.Shard) played for every block of a partition in one process, merged, against the single-GPU
``recommend`` / ``rank_against_all``; and the collective calls on a row-partitioned model (one rank here, two
ranks where the machine has two GPUs) against the single-GPU code on the all-gathered encoding.

Bit-exact: DOT, the fused MLP head and the generic ``score_edges`` path (MLPCAT) -- the shards score the same
encoded rows with the same kernels.  BIL, MLPDOT and MLPBIL apply their node-level transform to a row block, whose
GEMM may take another kernel than the one over the whole matrix: those heads are held to scores within 1e-5 of the
row maximum and ids equal up to near-ties."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import ranking
from tests.ranking_merge import merge_topk

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
NAN, INF = float("nan"), float("inf")
TOL = 1e-5
EXACT = ("DOT", "MLP", "MLPCAT")


# ----------------------------------------------------------------------------------------------- kernels
def _scores(Q, N, g, ties):
    s = torch.randint(-3, 4, (Q, N), generator=g).float() if ties else torch.randn(Q, N, generator=g)
    r = torch.rand(Q, N, generator=g)
    s[r < 0.1] = -INF
    s[(r >= 0.1) & (r < 0.15)] = NAN
    s[(r >= 0.15) & (r < 0.17)] = INF
    s[(r >= 0.17) & (r < 0.2)] = -0.0
    return s


def _csr(lists, n_rows):
    rowptr, col = [0], []
    for r in range(n_rows):
        col += lists.get(r, [])
        rowptr.append(len(col))
    return torch.tensor(rowptr), torch.tensor(col, dtype=torch.int32)


@pytest.mark.parametrize("ties", [False, True])
def test_mask_and_select_on_column_slices(ties):
    from plnlp_b200 import _ops
    g = torch.Generator().manual_seed(3)
    Q, N = 37, 140001
    s = _scores(Q, N, g, ties)
    nodes = torch.randint(0, N, (Q,), generator=g)
    lists = {int(n): torch.randint(0, N, (50,), generator=g).tolist() + [int(n), N, -3] for n in nodes[::2]}
    rowptr, col = _csr(lists, N)
    masked = ranking.mask_scores(s, nodes, rowptr, col, True)
    target = torch.randint(0, N, (Q,), generator=g)
    ts = s[torch.arange(Q), target].clone()
    ts[::4] = 0.5
    for lo, hi in [(0, N), (0, 1), (17, 4000), (65535, 65537), (12345, N), (N - 1, N)]:
        d = s[:, lo:hi].contiguous().to(DEV)
        _ops.score_mask_raw(d, nodes.to(DEV), rowptr.to(DEV), col.to(DEV), True, col0=lo)
        torch.testing.assert_close(d.cpu(), masked[:, lo:hi], rtol=0, atol=0, equal_nan=True)
        for k in (1, 20, 1024):
            ids, sc, gt, ge = _ops.topk_rows_raw(d, k, target=target.to(DEV), target_score=ts.to(DEV), col0=lo)
            r_ids, r_sc = ranking.topk_rows(masked[:, lo:hi], k)
            assert torch.equal(ids.cpu(), torch.where(r_ids >= 0, r_ids + lo, r_ids)), (lo, hi, k)
            assert torch.equal(sc.cpu(), r_sc), (lo, hi, k)
            local_t = torch.where((target >= lo) & (target < hi), target - lo, torch.full_like(target, -1))
            r_gt, r_ge = ranking.rank_counts(masked[:, lo:hi], local_t, ts)
            assert torch.equal(gt.cpu(), r_gt) and torch.equal(ge.cpu(), r_ge), (lo, hi, k)


def test_column_offset_zero_is_the_plain_entry_point():
    from plnlp_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(4)
    s = _scores(9, 5000, g, True).to(DEV)
    nodes = torch.randint(0, 5000, (9,), generator=g).to(DEV)
    a, b = s.clone(), s.clone()
    _lib.check(lib.plnlp_score_mask_f32(a.data_ptr(), 5000, 9, 5000, nodes.data_ptr(), None, None, 1, _lib.stream()),
               "plnlp_score_mask_f32")
    _lib.check(lib.plnlp_score_mask_cols_f32(b.data_ptr(), 5000, 9, 5000, 0, nodes.data_ptr(), None, None, 1,
                                             _lib.stream()), "plnlp_score_mask_cols_f32")
    assert torch.equal(a.isnan(), b.isnan()) and torch.equal(a.nan_to_num(), b.nan_to_num())
    out = []
    for fn, extra in ((lib.plnlp_topk_rows_f32, ()), (lib.plnlp_topk_rows_cols_f32, (0,))):
        ids = torch.empty(9, 50, dtype=torch.int64, device=DEV)
        sc = torch.empty(9, 50, device=DEV)
        ws = torch.empty(1 << 20, dtype=torch.uint8, device=DEV)
        _lib.check(fn(a.data_ptr(), 5000, 9, 5000, *extra, 50, None, None, ids.data_ptr(), sc.data_ptr(), None, None,
                      ws.data_ptr(), ws.numel(), _lib.stream()), "topk")
        out.append((ids, sc))
    assert torch.equal(out[0][0], out[1][0]) and torch.equal(out[0][1], out[1][1])


@pytest.mark.parametrize("k", [1, 20, 1024])
@pytest.mark.parametrize("R", [1, 2, 3, 4, 5, 6, 7, 8])
def test_merge_equals_topk_of_the_whole_row(R, k):
    """per-shard lists from the column-offset select on the row blocks, merged: the top-k of the concatenated rows,
    whatever the split (the last blocks are short or empty when R does not divide N)"""
    from plnlp_b200 import _ops, parallel
    g = torch.Generator().manual_seed(R * 100 + k)
    Q, N = 13, 9 * R + 3 if k == 1024 else 2500
    s = _scores(Q, N, g, ties=k != 20)
    s[1] = NAN                                              # a row without a candidate: every list dead
    d = s.to(DEV)
    ids_l, sc_l = [], []
    for r in range(R):
        lo, hi = parallel.row_block(N, r, R)
        if hi == lo:
            ids_l.append(torch.full((Q, k), -1, dtype=torch.int64, device=DEV))
            sc_l.append(torch.full((Q, k), -INF, device=DEV))
            continue
        i, v, _, _ = _ops.topk_rows_raw(d[:, lo:hi], k, col0=lo)
        ids_l.append(i)
        sc_l.append(v)
    ids_l.insert(R // 2, torch.full((Q, k), -1, dtype=torch.int64, device=DEV))     # one more, empty, shard
    sc_l.insert(R // 2, torch.full((Q, k), -INF, device=DEV))
    ids_in, sc_in = torch.stack(ids_l), torch.stack(sc_l)
    ids, sc = _ops.topk_merge_raw(ids_in, sc_in, k)
    r_ids, r_sc = ranking.topk_rows(s, k)
    assert torch.equal(ids.cpu(), r_ids) and torch.equal(sc.cpu(), r_sc)
    o_ids, o_sc = merge_topk(ids_in.cpu(), sc_in.cpu(), k)
    assert torch.equal(o_ids, r_ids) and torch.equal(o_sc, r_sc)
    for k_out in {1, max(1, k // 2)}:                       # fewer out than in
        i2, s2 = _ops.topk_merge_raw(ids_in, sc_in, k_out)
        assert torch.equal(i2.cpu(), r_ids[:, :k_out]) and torch.equal(s2.cpu(), r_sc[:, :k_out])


def test_sharded_entry_points_reject_invalid_arguments():
    from plnlp_b200 import _lib, _ops
    lib = _lib.load()
    s = torch.randn(4, 100, device=DEV)
    nodes = torch.zeros(4, dtype=torch.int64, device=DEV)
    for col0 in (-1, (1 << 31) - 100):                      # negative, or col0 + N reaches 2^31
        with pytest.raises(RuntimeError):
            _ops.topk_rows_raw(s, 5, col0=col0)
        with pytest.raises(RuntimeError):
            _ops.score_mask_raw(s, nodes, col0=col0)
    ids = torch.zeros(2, 4, 5, dtype=torch.int64, device=DEV)
    sc = torch.zeros(2, 4, 5, device=DEV)
    for k in (0, 1025):
        with pytest.raises(RuntimeError):
            _ops.topk_merge_raw(ids, sc, k)
    with pytest.raises(RuntimeError):
        _ops.topk_merge_raw(ids[0], sc[0], 5)               # not [R, Q, k_in]
    out_i = torch.empty(4, 5, dtype=torch.int64, device=DEV)
    out_s = torch.empty(4, 5, device=DEV)
    for R, k_in in ((0, 5), (2, 0)):
        with pytest.raises(RuntimeError):
            _lib.check(lib.plnlp_topk_merge_f32(ids.data_ptr(), sc.data_ptr(), R, 4, k_in, 5, out_i.data_ptr(),
                                                out_s.data_ptr(), _lib.stream()), "plnlp_topk_merge_f32")


# ----------------------------------------------------------------------------------------------- virtual shards
class Data:
    pass


def _setup(encoder, predictor, n, hid, seed=0, directed=None):
    """a random graph (directed for SAGE: A != A^T; symmetric and GCN-normalised for GCN) and a model on it"""
    from plnlp_b200.graph import CSRGraph
    from plnlp_b200.model import BaseModel
    from plnlp_b200.utils import gcn_normalization
    g = torch.Generator().manual_seed(seed)
    E = 5 * n
    src, dst = torch.randint(0, n, (E,), generator=g), torch.randint(0, n, (E,), generator=g)
    keep = src != dst
    ei = torch.stack([src[keep], dst[keep]]).to(DEV)
    adj = CSRGraph.from_edge_index(ei, None, n)
    if encoder == "GCN":
        adj = gcn_normalization(adj.to_symmetric())
    data = Data()
    data.adj_t, data.edge_index = adj, ei
    data.x = torch.randn(n, 16, generator=g).to(DEV)
    torch.manual_seed(seed + 1)
    model = BaseModel(lr=0.01, dropout=0.3, grad_clip_norm=2.0, gnn_num_layers=2, mlp_num_layers=2,
                      emb_hidden_channels=16, gnn_hidden_channels=hid, mlp_hidden_channels=hid, num_nodes=n,
                      num_node_feats=16, gnn_encoder_name=encoder, predictor_name=predictor, loss_func="AUC",
                      optimizer_name="Adam", device=DEV, use_node_feats=True, train_node_emb=True)
    model.param_init()
    return model, data


def _local_t(adj, lo, hi):
    """rows [lo, hi) of A^T as a CSRGraph (what ShardedAdj.local_t holds for that block)"""
    from plnlp_b200 import parallel
    from plnlp_b200.graph import CSRGraph
    rowptr, col, _ = adj.csr()
    n = adj.size(0)
    t_rowptr, t_col, _, _ = parallel.transpose_csr(rowptr, col, None, n)
    return CSRGraph(t_rowptr[lo:hi + 1] - t_rowptr[lo], t_col[int(t_rowptr[lo]):int(t_rowptr[hi])], None,
                    (hi - lo, n))


def _virtual(model, data, h, bounds, nodes, k, edges, exclude, exclude_self, batch_size=None):
    """every shard's step in one process, combined as the collectives would: -> (ids, scores, ranks)"""
    from plnlp_b200 import _ops, recommend
    n = h.size(0) - 1
    shards = []
    for lo, hi in bounds:
        local_t = _local_t(data.adj_t, lo, hi) if isinstance(exclude, str) else None
        rowptr, col = recommend.shard_exclude_csr(exclude, lo, hi, n, local_t)
        shards.append(recommend.Shard(model, h[lo:hi], lo, hi, n, rowptr, col, exclude_self))
    table = torch.cat([sh.table[:sh.hi - sh.lo] for sh in shards])      # what fetch_rows serves
    bs = batch_size or nodes.numel()
    ids, scores, ranks = [], [], []
    for i in range(0, nodes.numel(), bs):
        q = nodes[i:i + bs]
        rows = table[q]
        lists = [sh.topk(q, rows, k) for sh in shards]
        a, b = _ops.topk_merge_raw(torch.stack([x[0] for x in lists]), torch.stack([x[1] for x in lists]), k)
        ids.append(a)
        scores.append(b)
    src, tgt = edges[:, 0].contiguous(), edges[:, 1].contiguous()
    for i in range(0, src.numel(), bs):
        q, t = src[i:i + bs], tgt[i:i + bs]
        rows = table[q]
        parts = [sh.target_scores(q, rows, t) for sh in shards]
        ts = parts[0][1].clone()
        for _, x in parts[1:]:
            ts += x
        c = sum(sh.counts(S, q, t, ts) for sh, (S, _) in zip(shards, parts))
        ranks.append(0.5 * (c[0].float() + c[1].float()) + 1.0)
    return torch.cat(ids), torch.cat(scores), torch.cat(ranks)


def _check_against(predictor, got, want, S):
    """bit for bit (EXACT heads) or within TOL of the row maximum of the single-GPU score rows S, ids up to
    near-ties"""
    (i1, s1, r1), (i0, s0, r0) = got, want
    if predictor in EXACT:
        assert torch.equal(i1, i0) and torch.equal(s1, s0), predictor
        assert torch.equal(r1, r0), predictor
        return
    eps = TOL * S.nan_to_num(0, 0, 0).abs().amax(1, keepdim=True)
    fin = s0.isfinite()
    assert torch.equal(fin, s1.isfinite())
    assert ((s1 - s0).abs()[fin] <= eps.expand_as(s0)[fin]).all(), predictor
    same = (i1 == i0) | (i0 < 0)
    sa = S.gather(1, i1.clamp_min(0))
    sb = S.gather(1, i0.clamp_min(0))
    assert (same | ((sa - sb).abs() <= 2 * eps)).all(), predictor
    return eps


def _edges_for(nodes, n, g):
    t = torch.randint(0, n, (nodes.numel(),), generator=g).to(DEV)
    t[1] = nodes[1]                                          # the source itself as target
    return torch.stack([nodes, t], 1)


@pytest.mark.parametrize("encoder", ["SAGE", "GCN"])
@pytest.mark.parametrize("predictor", ["DOT", "BIL", "MLP", "MLPDOT", "MLPBIL", "MLPCAT"])
def test_virtual_shards_match_single_gpu(encoder, predictor):
    from plnlp_b200 import parallel, recommend
    n, k = 1000, 40
    model, data = _setup(encoder, predictor, n, hid=32)
    g = torch.Generator().manual_seed(5)
    nodes = torch.randint(0, n, (19,), generator=g).to(DEV)
    nodes[3] = nodes[2]
    edges = _edges_for(nodes, n, g)
    known = torch.stack([nodes.repeat_interleave(15), torch.randint(0, n, (19 * 15,), generator=g).to(DEV)], 1)
    edges[4, 1] = known[4 * 15, 1]                           # a known link as target: never filtered
    h = recommend._encode(model, data)
    S = recommend._Scorer(model, h).chunk(nodes)
    splits = [[parallel.row_block(n, r, R) for r in range(R)] for R in (1, 2, 3)] + [[(0, 400), (400, 400), (400, n)]]
    for exclude in (None, "adj", known):
        for exclude_self in (True, False):
            want = (*model.recommend(data, nodes, k, exclude=exclude, exclude_self=exclude_self),
                    model.rank_against_all(data, edges, exclude=exclude, exclude_self=exclude_self))
            for bounds in splits:
                got = _virtual(model, data, h, bounds, nodes, k, edges, exclude, exclude_self,
                               batch_size=7 if len(bounds) == 3 else None)
                eps = _check_against(predictor, got, want, S)
                if eps is not None:                          # ranks: the difference is bounded by the near-ties
                    ts = S.gather(1, edges[:, 1:2])
                    near = ((S - ts).abs() <= 2 * eps).sum(1)
                    assert ((got[2] - want[2]).abs() <= near).all(), (predictor, bounds)


@pytest.mark.parametrize("predictor", ["DOT", "MLP"])
def test_virtual_shards_tensor_core_shape(predictor):
    """N = 20 000, H = 64: gemm_backend picks the tensor-core kernel (and MLP the fused edge-MLP kernel)"""
    from plnlp_b200 import _ops, parallel, recommend
    n, k = 20000, 100
    model, data = _setup("SAGE", predictor, n, hid=64, seed=2)
    h = recommend._encode(model, data)
    sc = recommend._Scorer(model, h)
    assert sc.path == ("gemm" if predictor == "DOT" else "fused_mlp")
    if predictor == "DOT":
        assert sc.backend == _ops.GEMM_BACKEND != "ffma"
    g = torch.Generator().manual_seed(6)
    nodes = torch.randint(0, n, (33,), generator=g).to(DEV)
    edges = _edges_for(nodes, n, g)
    want = (*model.recommend(data, nodes, k, exclude="adj"), model.rank_against_all(data, edges, exclude="adj"))
    for R in (2, 3, 8):
        bounds = [parallel.row_block(n, r, R) for r in range(R)]
        got = _virtual(model, data, h, bounds, nodes, k, edges, "adj", True, batch_size=5)
        _check_against(predictor, got, want, None)


# ----------------------------------------------------------------------------------------------- collective calls
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _single_process(model, h, data_full, fn, *args, **kw):
    """the single-GPU code of recommend.py run on the encoded rows h"""
    model.partitioned, model.encode_for_test = False, (lambda data: h)
    try:
        return fn(model, data_full, *args, **kw)
    finally:
        model.partitioned = True
        del model.encode_for_test


def _worker(rank, ws, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=ws, device_id=dev)
    try:
        from plnlp_b200 import parallel, recommend
        from plnlp_b200.graph import CSRGraph
        from plnlp_b200.model import BaseModel
        n, k = 1001, 30
        out = {}
        for predictor in ("DOT", "MLP", "BIL"):
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
            known = torch.stack([nodes.repeat_interleave(10), torch.randint(0, n, (410,), generator=g).to(dev)], 1)
            part.encoder.eval()
            part.predictor.eval()
            h = part.encode_for_test(d2)                     # the all-gathered eval-mode encoding
            S = recommend._Scorer(part, h).chunk(nodes)
            res = {}
            for exclude in (None, "adj", known):
                for bs in (None, 6):
                    got = (*part.recommend(d2, nodes, k, exclude=exclude, batch_size=bs),
                           part.rank_against_all(d2, edges, exclude=exclude, batch_size=bs))
                    want = (*_single_process(part, h, data, recommend.recommend, nodes, k, exclude),
                            _single_process(part, h, data, recommend.rank_against_all, edges, exclude))
                    key = f"{'edges' if torch.is_tensor(exclude) else exclude}/{bs}"
                    res[key] = {"got": [t.detach().cpu() for t in got], "want": [t.detach().cpu() for t in want]}
            res["S"] = S.detach().cpu()
            # a mismatched call fails on every rank
            errors = []
            for call in (lambda: part.recommend(d2, nodes, k + rank), lambda: part.recommend(d2, nodes[:40 + rank], k),
                         lambda: part.rank_against_all(d2, edges, exclude="adj" if rank else None)):
                try:
                    call()
                    errors.append(None)
                except ValueError as ex:
                    errors.append(str(ex)[:40])
            res["mismatch"] = errors if ws > 1 else []
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
                assert all(m is not None for m in mismatch), (r, predictor, mismatch)
            for key, v in res.items():
                _check_against(predictor, tuple(v["got"]), tuple(v["want"]), S)
                if r > 0:                                     # every rank holds the same result
                    for a, b in zip(v["got"], ret[0][predictor][key]["got"]):
                        assert torch.equal(a, b), (r, predictor, key)


def test_partitioned_one_rank_matches_single_process():
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(1, _free_port(), ret), nprocs=1, join=True)
    _check_ranks(ret, 1)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_partitioned_two_ranks_match_single_process():
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(2, _free_port(), ret), nprocs=2, join=True)
    _check_ranks(ret, 2)


def test_partitioned_model_without_sharded_adjacency_raises():
    from plnlp_b200 import recommend
    model, data = _setup("GCN", "DOT", 200, hid=32)
    model.partitioned = True
    with pytest.raises(NotImplementedError, match="ShardedAdj"):
        recommend.recommend(model, data, torch.arange(3, device=DEV), 5)

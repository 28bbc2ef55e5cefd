"""GPU checks of link recommendation over all nodes (-m gpu): the mask / top-k kernels (csrc/topk.cu) against the CPU
restatement (oracle/ranking.py) bit for bit, and BaseModel.recommend / rank_against_all against fp64 oracle scores for
every predictor."""
import pytest
import torch

from oracle import plnlp_ref, ranking, sparse

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
TOL = 1e-5
NAN, INF = float("nan"), float("inf")


# ----------------------------------------------------------------------------------------------- kernels
def _scores(kind, Q, N, g):
    if kind == "normal":
        return torch.randn(Q, N, generator=g)
    if kind == "ties":
        return torch.randint(-4, 5, (Q, N), generator=g).float()
    if kind == "constant":
        return torch.full((Q, N), -1.5)
    if kind == "ascending":                                 # every score beats all before it
        return torch.arange(N, dtype=torch.float32).repeat(Q, 1)
    s = torch.randn(Q, N, generator=g)                      # "special"
    r = torch.rand(Q, N, generator=g)
    s[r < 0.3] = -INF
    s[(r >= 0.3) & (r < 0.4)] = NAN
    s[(r >= 0.4) & (r < 0.42)] = INF
    s[(r >= 0.42) & (r < 0.45)] = -0.0
    s[0] = NAN                                              # a row excluded entirely
    if Q > 2:
        s[2, : N // 2] = -INF
    return s


def _check_topk(s, ks, target=None):
    from plnlp_b200 import _ops
    Q, N = s.shape
    kmax = max(ks)
    ref_ids, ref_sc = ranking.topk_rows(s, kmax)
    d = s.to(DEV)
    for k in ks:
        ids, sc, _, _ = _ops.topk_rows_raw(d, k)
        assert torch.equal(ids.cpu(), ref_ids[:, :k]), (Q, N, k)
        assert torch.equal(sc.cpu(), ref_sc[:, :k]), (Q, N, k)
    if target is not None:
        ts = s[torch.arange(Q), target].clone()
        ts[::3] = 0.125                                     # target scores that are not in the row
        gt, ge = ranking.rank_counts(s, target, ts)
        ids, sc, g1, g2 = _ops.topk_rows_raw(d, 20, target=target.to(DEV), target_score=ts.to(DEV))
        assert torch.equal(g1.cpu(), gt) and torch.equal(g2.cpu(), ge)
        assert torch.equal(ids.cpu(), ref_ids[:, :20])
        _, _, g1, g2 = _ops.topk_rows_raw(d, 0, target=target.to(DEV), target_score=ts.to(DEV))
        assert torch.equal(g1.cpu(), gt) and torch.equal(g2.cpu(), ge)


@pytest.mark.parametrize("Q,N", [(1, 1), (7, 5), (300, 33), (7, 4267), (300, 4267), (1, 100003), (7, 100003)])
@pytest.mark.parametrize("kind", ["normal", "ties", "constant", "ascending", "special"])
def test_topk_rows_matches_oracle(Q, N, kind):
    g = torch.Generator().manual_seed(Q * 1000 + N)
    s = _scores(kind, Q, N, g)
    _check_topk(s, (1, 20, 100, 1024), target=torch.randint(0, N, (Q,), generator=g))


@pytest.mark.parametrize("kind", ["normal", "ties"])
def test_topk_rows_citation2_width(kind):
    g = torch.Generator().manual_seed(5)
    N = 2927963
    s = _scores(kind, 3, N, g)
    _check_topk(s, (20, 1024), target=torch.randint(0, N, (3,), generator=g))


def test_topk_rows_strided_chunk():
    """a column slice of a wider matrix: the kernel reads rows at the given leading dimension"""
    from plnlp_b200 import _ops
    g = torch.Generator().manual_seed(9)
    full = torch.randn(9, 70001, generator=g)
    s = full[:, 3:70000]
    ids, sc, _, _ = _ops.topk_rows_raw(full.to(DEV)[:, 3:70000], 50)
    r_ids, r_sc = ranking.topk_rows(s, 50)
    assert torch.equal(ids.cpu(), r_ids) and torch.equal(sc.cpu(), r_sc)


def _csr(lists, n_rows):
    rowptr, col = [0], []
    for r in range(n_rows):
        col += lists.get(r, [])
        rowptr.append(len(col))
    return torch.tensor(rowptr), torch.tensor(col, dtype=torch.int32)


@pytest.mark.parametrize("exclude_self", [True, False])
def test_score_mask_matches_oracle(exclude_self):
    from plnlp_b200 import _ops
    g = torch.Generator().manual_seed(2)
    Q, N = 40, 4267
    s = torch.randn(Q, N, generator=g)
    s[3, 7] = NAN
    nodes = torch.randint(0, N, (Q,), generator=g)
    nodes[1] = nodes[0]
    lists = {}
    for i, n in enumerate(nodes.tolist()):
        if i % 4 == 0:
            continue                                        # empty rows
        c = torch.randint(0, N, (int(torch.randint(1, 60, (1,), generator=g)),), generator=g).tolist()
        lists[n] = c + c[:3] + [n, N, -5]                   # duplicates, a self loop, out-of-range columns
    rowptr, col = _csr(lists, N)
    want = ranking.mask_scores(s, nodes, rowptr, col, exclude_self)
    d = s.to(DEV)
    _ops.score_mask_raw(d, nodes.to(DEV), rowptr.to(DEV), col.to(DEV), exclude_self)
    torch.testing.assert_close(d.cpu(), want, rtol=0, atol=0, equal_nan=True)
    d = s.to(DEV)
    _ops.score_mask_raw(d, nodes.to(DEV), None, None, True)
    torch.testing.assert_close(d.cpu(), ranking.mask_scores(s, nodes, None, None, True), rtol=0, atol=0, equal_nan=True)


def test_invalid_arguments_raise():
    from plnlp_b200 import _lib, _ops
    s = torch.randn(4, 100, device=DEV)
    for k in (1025, -1):
        with pytest.raises(RuntimeError):
            _ops.topk_rows_raw(s, k)
    with pytest.raises(RuntimeError):
        _ops.topk_rows_raw(s, 0)                            # no k and no target: nothing to compute
    lib = _lib.load()
    ids = torch.empty(4, 5, dtype=torch.int64, device=DEV)
    sc = torch.empty(4, 5, device=DEV)
    ws = torch.empty(1 << 20, dtype=torch.uint8, device=DEV)
    with pytest.raises(RuntimeError):                       # leading dimension below the row length
        _lib.check(lib.plnlp_topk_rows_f32(s.data_ptr(), 99, 4, 100, 5, None, None, ids.data_ptr(), sc.data_ptr(),
                                           None, None, ws.data_ptr(), ws.numel(), _lib.stream()), "plnlp_topk_rows_f32")
    with pytest.raises(RuntimeError):
        _lib.check(lib.plnlp_score_mask_f32(s.data_ptr(), 50, 4, 100, ids.data_ptr(), None, None, 1, _lib.stream()),
                   "plnlp_score_mask_f32")
    with pytest.raises(RuntimeError):                       # N >= 2^31
        _lib.check(lib.plnlp_topk_rows_f32(s.data_ptr(), 1 << 31, 1, 1 << 31, 5, None, None, ids.data_ptr(),
                                           sc.data_ptr(), None, None, ws.data_ptr(), ws.numel(), _lib.stream()),
                   "plnlp_topk_rows_f32")


# ----------------------------------------------------------------------------------------------- model level
class Data:
    pass


N_NODES, FEATS, EMB, HID = 3000, 16, 16, 64


def _graph():
    g = torch.Generator().manual_seed(0)
    E = 15000
    src, dst = torch.randint(0, N_NODES, (E,), generator=g), torch.randint(0, N_NODES, (E,), generator=g)
    keep = src != dst
    src, dst = src[keep], dst[keep]
    ei = torch.cat([torch.stack([src, dst]), torch.stack([dst, src])], 1)
    x = torch.randn(N_NODES, FEATS, generator=g)
    return ei, x


def _setup(encoder, predictor):
    from plnlp_b200.graph import CSRGraph
    from plnlp_b200.model import BaseModel
    ei, x = _graph()
    adj_cpu = sparse.to_sparse_tensor(ei, None, N_NODES)
    if encoder == "GCN":
        adj_cpu = sparse.gcn_normalization(adj_cpu)
    rowptr, col, val = adj_cpu.csr()
    data = Data()
    data.adj_t = CSRGraph(rowptr.to(DEV), col.to(DEV), None if val is None else val.to(DEV), (N_NODES, N_NODES))
    data.edge_index = ei.to(DEV)
    data.x = x.to(DEV)
    torch.manual_seed(1)
    model = BaseModel(lr=0.01, dropout=0.3, grad_clip_norm=2.0, gnn_num_layers=2, mlp_num_layers=2,
                      emb_hidden_channels=EMB, gnn_hidden_channels=HID, mlp_hidden_channels=HID, num_nodes=N_NODES,
                      num_node_feats=FEATS, gnn_encoder_name=encoder, predictor_name=predictor, loss_func="AUC",
                      optimizer_name="Adam", device=DEV, use_node_feats=True, train_node_emb=True)
    model.param_init()
    # fp64 oracle scores of every (query, candidate) pair
    ref = plnlp_ref.OracleModel(num_nodes=N_NODES, emb_hidden=EMB, gnn_hidden=HID, mlp_hidden=HID, gnn_layers=2,
                                mlp_layers=2, encoder=encoder, predictor="DOT", num_node_feats=FEATS,
                                use_node_feats=True, train_node_emb=True, dtype=torch.float64)
    state = {"emb": model.emb.weight.detach().cpu().double()}
    for name, p in model.encoder.named_parameters():
        state["enc." + name[len("convs."):]] = p.detach().cpu().double()
    ref.load(state)
    if val is not None:
        adj_cpu = adj_cpu.set_value(val.double())
    with torch.no_grad():
        h64 = ref.encode(x.double(), adj_cpu)
    pred = model.predictor
    P = {n: p.detach().cpu().double() for n, p in pred.named_parameters()}
    lins = [(P[f"lins.{i}.weight"], P[f"lins.{i}.bias"]) for i in range(len(getattr(pred, "lins", [])))]

    def score64(q):
        xi = h64[q].repeat_interleave(N_NODES, 0)
        xj = h64.repeat(q.numel(), 1)
        with torch.no_grad():
            if predictor == "DOT":
                s = plnlp_ref.dot_score(xi, xj)
            elif predictor == "BIL":
                s = plnlp_ref.bil_score(P["bilin.weight"], xi, xj)
            elif predictor == "MLP":
                s = plnlp_ref.mlp_score(lins, xi, xj).reshape(-1)
            elif predictor == "MLPDOT":
                s = plnlp_ref.mlpdot_score(lins, xi, xj)
            elif predictor == "MLPBIL":
                s = plnlp_ref.mlpbil_score(lins, P["bilin.weight"], xi, xj)
            else:
                s = plnlp_ref.mlpcat_score(lins, xi, xj).reshape(-1)
        return s.reshape(q.numel(), N_NODES)

    return model, data, score64


def _adj_lists(data, nodes):
    rowptr, col, _ = data.adj_t.csr()
    rowptr, col = rowptr.cpu(), col.cpu()
    return [set(col[rowptr[n]:rowptr[n + 1]].tolist()) for n in nodes.tolist()]


@pytest.mark.parametrize("encoder", ["SAGE", "GCN"])
@pytest.mark.parametrize("predictor", ["DOT", "BIL", "MLP", "MLPDOT", "MLPBIL", "MLPCAT"])
def test_recommend_and_rank_against_oracle(encoder, predictor):
    model, data, score64 = _setup(encoder, predictor)
    g = torch.Generator().manual_seed(4)
    nodes = torch.randint(0, N_NODES, (23,), generator=g)
    nodes[1] = nodes[0]
    S64 = score64(nodes)
    scale = S64.abs().amax(1, keepdim=True).clamp_min(1e-30)
    eps = TOL * scale
    k = 50
    for exclude in (None, "adj"):
        ids, sc = model.recommend(data, nodes.to(DEV), k, exclude=exclude)
        assert ids.shape == (23, k) and sc.dtype == torch.float32
        ids_c, sc_c = ids.cpu(), sc.cpu()
        # returned scores are the predictor's scores of the returned pairs
        h = model.encode_for_test(data)
        pairs = torch.stack([nodes.repeat_interleave(k), ids_c.reshape(-1)], 1)
        bp = model.batch_predict(h, pairs.to(DEV), 4096).cpu().reshape(23, k)
        assert ((sc_c.double() - bp.double()).abs() <= TOL * scale).all(), (predictor, exclude)
        # nothing excluded, no duplicates, against the fp64 oracle's top-k up to near-ties
        banned = _adj_lists(data, nodes) if exclude == "adj" else [set() for _ in range(23)]
        Sm = S64.clone()
        for q, n in enumerate(nodes.tolist()):
            banned[q] = banned[q] | {n}
            Sm[q, list(banned[q])] = -INF
            got = ids_c[q].tolist()
            assert len(set(got)) == k and not (set(got) & banned[q])
        ref_ids, _ = ranking.topk_rows(Sm, k)
        a = torch.gather(S64, 1, ids_c)
        b = torch.gather(S64, 1, ref_ids)
        assert ((a - b).abs() <= eps).all(), (predictor, exclude, float(((a - b).abs() / scale).max()))
        # bit-identical across chunk sizes and calls
        for bs in (1, 7, None):
            i2, s2 = model.recommend(data, nodes.to(DEV), k, exclude=exclude, batch_size=bs)
            assert torch.equal(i2, ids) and torch.equal(s2, sc), (predictor, exclude, bs)
        # filtered ranks: the oracle's counts with near-ties either way
        targets = torch.randint(0, N_NODES, (23,), generator=g)
        targets[2] = nodes[2]                                # the source itself as target
        adj_t = next(iter(banned[3] - {int(nodes[3])}), None)
        if adj_t is not None:
            targets[3] = adj_t                                # a known link as target: never filtered
        edges = torch.stack([nodes, targets], 1)
        ranks = model.rank_against_all(data, edges.to(DEV), exclude=exclude).cpu().double()
        for q in range(23):
            t = int(targets[q])
            row = S64[q].clone()
            row[list(banned[q] - {t})] = -INF
            row[t] = -INF                                     # j != target
            ts = S64[q, t]
            lo = 1 + int((row > ts + eps[q]).sum())
            hi = 1 + int((row >= ts - eps[q]).sum())
            assert lo <= ranks[q] <= hi, (predictor, exclude, q, float(ranks[q]), lo, hi)
        for bs in (1, 7):
            r2 = model.rank_against_all(data, edges.to(DEV), exclude=exclude, batch_size=bs).cpu().double()
            assert torch.equal(r2, ranks)


def test_exclude_edge_tensor_and_partitioned():
    from plnlp_b200.utils import full_rank_metrics
    model, data, _ = _setup("SAGE", "DOT")
    nodes = torch.arange(0, 300, 10)
    g = torch.Generator().manual_seed(8)
    known = torch.stack([nodes.repeat_interleave(20), torch.randint(0, N_NODES, (600,), generator=g)], 1)
    ids, _ = model.recommend(data, nodes.to(DEV), 100, exclude=known.to(DEV))
    for q, n in enumerate(nodes.tolist()):
        banned = set(known[known[:, 0] == n, 1].tolist()) | {n}
        assert not set(ids[q].cpu().tolist()) & banned
    edges = torch.stack([nodes, ids[:, 0].cpu()], 1)
    ranks = model.rank_against_all(data, edges.to(DEV), exclude=known.to(DEV))
    assert torch.equal(ranks.cpu(), torch.ones(nodes.numel()))     # the top recommendation ranks first
    m = full_rank_metrics(ranks)
    assert m["MRR"] == 1.0 and m["Hits@1"] == 1.0
    m = full_rank_metrics(torch.tensor([1.0, 2.0, 4.5, 200.0], device=DEV), ks=(1, 3, 100))
    assert m["Hits@1"] == 0.25 and m["Hits@3"] == 0.5 and m["Hits@100"] == 0.75
    assert abs(m["MRR"] - (1 + 0.5 + 1 / 4.5 + 1 / 200) / 4) < 1e-6
    model.partitioned = True
    with pytest.raises(NotImplementedError):
        model.recommend(data, nodes.to(DEV), 10)
    with pytest.raises(NotImplementedError):
        model.rank_against_all(data, edges.to(DEV))


def test_recommend_citation2_shape_dot():
    """citation2 shape (N = 2 927 963, GCN 200 wide), DOT head: a few queries against torch.topk over batch_predict
    of every pair"""
    import bench
    from plnlp_b200.graph import CSRGraph
    from plnlp_b200.utils import gcn_normalization
    cfg = dict(bench.WORKLOADS["citation2"], predictor="DOT")
    torch.manual_seed(0)
    data, _ = bench.build_workload(cfg, DEV, CSRGraph, gcn_normalization)
    model = bench.make_model(cfg, DEV)
    N, k = cfg["N"], 100
    nodes = torch.tensor([0, 17, 123456, N - 1], device=DEV)
    ids, sc = model.recommend(data, nodes, k, exclude_self=False)
    h = model.encode_for_test(data)
    cand = torch.arange(N, device=DEV)
    for q, n in enumerate(nodes.tolist()):
        bp = model.batch_predict(h, torch.stack([torch.full_like(cand, n), cand], 1), 1 << 22)
        top = torch.topk(bp, k)
        eps = TOL * float(bp.abs().max())
        assert (bp[ids[q]] - top.values).abs().max() <= eps
        assert (sc[q] - bp[ids[q]]).abs().max() <= eps
    i1, s1 = model.recommend(data, nodes, k, exclude_self=False, batch_size=1)
    assert torch.equal(i1, ids) and torch.equal(s1, sc)

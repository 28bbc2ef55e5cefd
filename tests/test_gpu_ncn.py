"""GPU tests of the NCN predictor (heuristics.common_neighbour_lists, csrc/heuristic.cu common_neighbour_list_kernel,
layer.NCNPredictor, the NCN paths of model.BaseModel) against the CPU restatement in tests/ncn_oracle.py: the lists
bit for bit on the graph of test_gpu_heuristics.py (hub rows of 5 000 entries for the search mode, hub-hub pairs for
the merge mode, isolated nodes, (u, u) pairs, -1 ids, a non-symmetric adjacency, more pairs than warps in the
grid); the head's forward and gradients in fp32 against fp64; the restricted last conv against the full one and
prepared against unprepared steps; short training trajectories; ``test``; and the calls that raise."""
import pytest
import torch

from oracle import sparse
from tests import ncn_oracle as no
from tests.helpers import fp32_close, rand_graph, rel_err
from tests.test_gpu_heuristics import HUBS, N, N_ISOLATED, P, _edges_coo, _pairs

pytestmark = pytest.mark.gpu
TOL = 1e-5
DEV = torch.device("cuda")


MID = torch.arange(100, 164)        # rows of 40 .. 200 extra entries taken from a hub's row: paired with that hub they
MID_PAIRS = slice(1500, 1564)       # take the search mode over several 32-entry rounds of the shorter list


def _adj(symmetric=True):
    """the graph of test_gpu_heuristics.py with 6 000 more distinct neighbours on each hub row, and the rows MID with
    40 .. 200 more, drawn from the new neighbours of hub MID % HUBS"""
    from plnlp_b200.graph import CSRGraph
    src, dst = _edges_coo(symmetric)
    g = torch.Generator().manual_seed(12)
    hs = torch.arange(HUBS).repeat_interleave(6000)
    nb = torch.cat([torch.randperm(N - N_ISOLATED, generator=g)[:6000] for _ in range(HUBS)])
    deg = torch.randint(40, 201, (MID.numel(),), generator=g)
    ms = torch.cat([torch.full((int(d),), int(m)) for m, d in zip(MID, deg)])
    mn = torch.cat([nb[int(m) % HUBS * 6000:][:int(d)] for m, d in zip(MID, deg)])
    hs, nb = torch.cat([hs, ms]), torch.cat([nb, mn])
    src, dst = torch.cat([src, hs] + ([nb] if symmetric else [])), torch.cat([dst, nb] + ([hs] if symmetric else []))
    return CSRGraph.from_coo(src.cuda(), dst.cuda(), torch.rand(src.numel(), generator=g).cuda(), (N, N))


def _pairs_ncn():
    e = _pairs()
    e[MID_PAIRS] = torch.stack([MID, MID % HUBS], 1)
    return e


def _pairs_with_negatives():
    e = _pairs_ncn()
    e[1200:1300, 0] = -1
    e[1300:1400, 1] = -1
    e[1400, :] = -1
    return e


@pytest.mark.parametrize("symmetric", [True, False])
def test_lists_match_python_sets(symmetric):
    from plnlp_b200 import _ops, heuristics
    adj = _adj(symmetric)
    e = _pairs_with_negatives()
    assert P > 1184 * 8                                          # several grid-stride passes of the fill kernel
    rowptr, col = heuristics.common_neighbour_lists(adj, e.cuda())
    assert rowptr.dtype == torch.int64 and col.dtype == torch.int64 and rowptr.shape == (P + 1,)
    sets = no.sets_of(adj)
    assert max(len(s) for s in sets[:HUBS]) >= 5000
    want_ptr, want_col = no.lists(sets, e)
    assert torch.equal(rowptr.cpu(), want_ptr) and torch.equal(col.cpu(), want_col)
    cnt = rowptr[1:] - rowptr[:-1]
    assert int(cnt[:HUBS * HUBS].min()) > 0                      # hub-hub pairs (merge mode) share neighbours
    assert int(cnt[20:1000].sum()) > 0                           # hub-small pairs (search mode)
    # (mid, hub): search mode with a shorter list of more than one 32-entry round, and hits in several rounds
    assert min(len(sets[int(m)]) for m in MID) > 32
    assert int(cnt[MID_PAIRS].min()) >= 40 and int(cnt[MID_PAIRS].max()) > 100
    assert int(cnt[1100:1200].sum()) == 0 and int(cnt[1200:1401].sum()) == 0      # isolated, -1
    # the counts are the CN scores; the count kernel gives 0 for a -1 id
    ok = (e >= 0).all(1)
    cn = heuristics.score_edges(adj, e[ok].cuda(), "CN")
    assert torch.equal(cnt[ok.cuda()].to(torch.float32), cn)
    t = heuristics.neighbour_table(adj)
    raw = _ops.link_heuristic_raw(t.rowptr, t.col, None, e.cuda())
    assert torch.equal(raw.to(torch.int64), cnt)
    # run to run and batch to batch
    r2, c2 = heuristics.common_neighbour_lists(adj, e.cuda())
    assert torch.equal(r2, rowptr) and torch.equal(c2, col)
    r3, c3 = heuristics.common_neighbour_lists(adj, e[:777].cuda())
    assert torch.equal(r3, rowptr[:778]) and torch.equal(c3, col[:int(rowptr[777])])
    # no pairs
    r4, c4 = heuristics.common_neighbour_lists(adj, torch.empty(0, 2, dtype=torch.int64, device="cuda"))
    assert r4.tolist() == [0] and c4.numel() == 0


def test_lists_ignore_values_and_diagonal():
    from plnlp_b200 import heuristics
    from plnlp_b200.utils import gcn_normalization
    adj = _adj()
    e = _pairs_ncn()[:5000].cuda()
    a, b = heuristics.common_neighbour_lists(adj, e), heuristics.common_neighbour_lists(gcn_normalization(adj), e)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_abi_error_codes():
    from plnlp_b200 import _lib
    lib = _lib.load()
    t = _lib.stream()
    rowptr = torch.zeros(11, dtype=torch.int64, device="cuda")
    col = torch.zeros(4, dtype=torch.int32, device="cuda")
    e = torch.zeros(3, 2, dtype=torch.int64, device="cuda")
    optr = torch.zeros(4, dtype=torch.int64, device="cuda")
    out = torch.zeros(4, dtype=torch.int32, device="cuda")
    p = _lib.ptr
    f = lib.plnlp_common_neighbour_list
    assert f(p(rowptr), p(col), 10, 4, p(e), 3, p(optr), p(out), t) == 0
    assert f(None, p(col), 10, 4, p(e), 3, p(optr), p(out), t) == -1
    assert f(p(rowptr), None, 10, 4, p(e), 3, p(optr), p(out), t) == -1
    assert f(p(rowptr), p(col), 10, 4, None, 3, p(optr), p(out), t) == -1
    assert f(p(rowptr), p(col), 10, 4, p(e), 3, None, p(out), t) == -1
    assert f(p(rowptr), p(col), 10, 4, p(e), 3, p(optr), None, t) == -1
    assert f(p(rowptr), None, 10, 0, p(e), 3, p(optr), None, t) == 0           # no entries: nothing to write
    assert f(p(rowptr), p(col), -1, 4, p(e), 3, p(optr), p(out), t) == -2
    assert f(p(rowptr), p(col), 10, -1, p(e), 3, p(optr), p(out), t) == -2
    assert f(p(rowptr), p(col), 10, 4, p(e), -1, p(optr), p(out), t) == -2
    assert f(p(rowptr), p(col), 0, 4, p(e), 3, p(optr), p(out), t) == -2
    assert f(None, None, 10, 4, None, 0, None, None, t) == 0                   # P = 0: nothing to do
    torch.cuda.synchronize()


def _small_graph(N_=300, E=2400, seed=3):
    ei, _ = rand_graph(N_, E, seed=seed, hub=True)
    o = sparse.to_sparse_tensor(torch.cat([ei, ei.flip(0)], 1), None, N_)
    return ei, o


def _gpu_graph(o, n):
    from plnlp_b200.graph import CSRGraph
    rowptr, col, val = o.csr()
    return CSRGraph(rowptr.cuda(), col.cuda(), None if val is None else val.cuda(), (n, n))


@pytest.mark.parametrize("L", [1, 2])
def test_score_edges_forward_and_gradients(L):
    from plnlp_b200 import heuristics
    from plnlp_b200.layer import NCNPredictor
    torch.manual_seed(L)
    n, H, hid, Pn = 300, 24, 32, 700
    _, o = _small_graph(n)
    adj = _gpu_graph(o, n)
    pred = NCNPredictor(H, hid, 1, L, 0.0).cuda()
    h = torch.randn(n + 1, H, device="cuda").requires_grad_(True)
    e = torch.randint(0, n, (Pn, 2))
    e[:10, 1] = -1
    e[10:20, 1] = e[10:20, 0]
    cn = heuristics.common_neighbour_lists(adj, e.cuda())
    assert int(cn[0][-1]) > Pn                                  # the pairs do have common neighbours
    s = pred.score_edges(h, e.cuda(), cn)
    assert s.shape == (Pn, 1)
    gout = torch.randn(Pn, 1)
    s.backward(gout.cuda())

    def ref(dtype):
        hh = h.detach().cpu().to(dtype).requires_grad_(True)
        lins = [(lin.weight.detach().cpu().to(dtype).requires_grad_(True),
                 lin.bias.detach().cpu().to(dtype).requires_grad_(True)) for lin in pred.lins]
        r = no.score(hh, e, no.lists(no.sets_of(adj), e), lins)
        (r * gout.reshape(-1).to(dtype)).sum().backward()
        return r, hh.grad, [t.grad for wb in lins for t in wb]
    r32, gh32, gw32 = ref(torch.float32)
    r64, gh64, gw64 = ref(torch.float64)
    ok, msg = fp32_close(s.reshape(-1), r32, r64, TOL)
    assert ok, msg
    ok, msg = fp32_close(h.grad, gh32, gh64, TOL)
    assert ok, msg
    floor = TOL * max(float(g.abs().max()) for g in gw64)
    for prm, g32, g64 in zip(pred.flat_params(), gw32, gw64):
        ok, msg = fp32_close(prm.grad.reshape(-1), g32.reshape(-1), g64.reshape(-1), TOL, floor=floor)
        assert ok, msg


def test_common_neighbour_sum_bit_identical_across_batches_and_runs():
    from plnlp_b200 import _ops, heuristics
    adj = _adj()
    e = _pairs_ncn()[:20000].cuda()
    torch.manual_seed(0)
    h = torch.randn(N, 50, device="cuda")
    with torch.no_grad():
        full = _ops.common_neighbour_sum(h, heuristics.common_neighbour_lists(adj, e))
        again = _ops.common_neighbour_sum(h, heuristics.common_neighbour_lists(adj, e))
        assert torch.equal(full, again)
        for bs in (1, 333, 4096):
            parts = [_ops.common_neighbour_sum(h, heuristics.common_neighbour_lists(adj, e[i:i + bs]))
                     for i in range(0, min(e.size(0), 12 * bs), bs)]
            got = torch.cat(parts)
            assert torch.equal(got, full[:got.size(0)]), bs
    # the transposed backward is deterministic too
    grads = []
    for _ in range(2):
        hh = h.clone().requires_grad_(True)
        _ops.common_neighbour_sum(hh, heuristics.common_neighbour_lists(adj, e)).sum().backward()
        grads.append(hh.grad)
    assert torch.equal(grads[0], grads[1])


class Data:
    pass


def _model(encoder, loss, n, H, L=2, lr=0.01, optimizer="SGD", clip=2.0):
    from plnlp_b200.model import BaseModel
    return BaseModel(lr=lr, dropout=0.0, grad_clip_norm=clip, gnn_num_layers=2, mlp_num_layers=L,
                     emb_hidden_channels=H, gnn_hidden_channels=H, mlp_hidden_channels=H, num_nodes=n,
                     num_node_feats=0, gnn_encoder_name=encoder, predictor_name="NCN", loss_func=loss,
                     optimizer_name=optimizer, device=DEV, use_node_feats=False, train_node_emb=True)


def _data(encoder, n, seed=3):
    ei, o = _small_graph(n, 8 * n, seed)
    if encoder == "GCN":
        o = sparse.gcn_normalization(o)
    d = Data()
    d.adj_t = _gpu_graph(o, n)
    d.x, d.edge_index = None, ei.cuda()
    return d, o, ei


def test_restricted_last_conv_matches_full(monkeypatch):
    """GCN + NCN where the batch restricts: the last conv computes the union of endpoints and common neighbours; the
    same step with the restriction off gives the same loss and parameters"""
    from plnlp_b200 import graph, model as M
    monkeypatch.setattr(graph, "DENSE_SPMM", False)
    n, H, B, k = 2000, 32, 64, 2
    d, _, ei = _data("GCN", n)
    pos = ei.t()[:B].contiguous().cuda()
    neg = torch.randint(0, n, (B * k, 2), generator=torch.Generator().manual_seed(1)).cuda()
    out = []
    for restrict in (True, False):
        monkeypatch.setattr(M, "ROW_SPARSE_GRAD", restrict)
        torch.manual_seed(5)
        m = _model("GCN", "AUC", n, H)
        m.param_init()
        m.encoder.train(); m.predictor.train()
        assert m._sparse_rows(pos, neg) == restrict
        if restrict:
            calls = []
            orig = m.encoder.forward
            m.encoder.forward = lambda *a, **kw: (calls.append(kw.get("out_rows")), orig(*a, **kw))[1]
        loss = m.train_batch(d, pos, neg, k)
        if restrict:
            from plnlp_b200.heuristics import common_neighbour_lists
            cn = common_neighbour_lists(d.adj_t, torch.cat([pos, neg]))
            ends = torch.unique(torch.cat([pos, neg]).reshape(-1))
            assert torch.equal(calls[0], torch.unique(torch.cat([ends, cn[1]])))
            assert calls[0].numel() > ends.numel()                  # the union grew
        out.append((loss, [p.detach().clone() for p in m.para_list]))
    assert rel_err(out[0][0], out[1][0]) < TOL
    _params_close(out[0][1], out[1][1])


def _params_close(got, want, names=None):
    """every tensor within TOL relative, or within TOL x the largest parameter of the model absolute: a bias that
    starts at 0 (GCNConv) holds only its summed updates, column sums of d loss / d y that cancel, and its rounding
    is set by the magnitude of the whole model, as in the floor of test_gpu_model.py"""
    floor = TOL * max(float(w.detach().double().abs().max()) for w in want)
    for i, (a, b) in enumerate(zip(got, want)):
        a, b = a.detach().double().cpu(), b.detach().double().cpu()
        err = float((a - b).abs().max())
        assert err <= TOL * float(b.abs().max()) or err <= floor, (names[i] if names else i, err, floor)


def test_prepared_batches_equal_unprepared(monkeypatch):
    """run_batches prepares batch i + 1 on the side stream (prepare_batch with wait_main=False); the first prepared
    batch finds no neighbour table and must order its side-stream reads after the build on the main stream.  Each run
    starts from a fresh adjacency object, so the prepared run takes that cold path; both runs give the same bits."""
    from plnlp_b200 import graph, heuristics, model as M
    monkeypatch.setattr(graph, "DENSE_SPMM", False)
    n, H, B, k = 20000, 32, 64, 2
    outs = []
    for ahead in (True, False):
        d, _, ei = _data("GCN", n)
        assert heuristics.cached_table(d.adj_t) is None
        batches = [(ei.t()[i * B:(i + 1) * B].contiguous().cuda(),
                    torch.randint(0, n, (B * k, 2), generator=torch.Generator().manual_seed(2 + i)).cuda(), None)
                   for i in range(3)]
        monkeypatch.setattr(M, "PREPARE_AHEAD", ahead)
        torch.manual_seed(5)
        m = _model("GCN", "AUC", n, H)
        m.param_init()
        m.encoder.train(); m.predictor.train()
        preps = []
        orig = m.prepare_batch
        m.prepare_batch = lambda *a, **kw: (lambda r: (preps.append(r), r)[1])(orig(*a, **kw))
        tot, _, n_b = m.run_batches(d, iter(batches), k)
        assert n_b == 3 and len(preps) == (3 if ahead else 0)
        assert all(p is not None and p.cn is not None for p in preps)
        for p, (pos, neg, _) in zip(preps, batches):             # the prepared lists, renumbered back, are the lists
            rowptr, col = heuristics.common_neighbour_lists(d.adj_t, torch.cat([pos, neg]))
            assert torch.equal(p.cn[0], rowptr) and torch.equal(p.ids[p.cn[1]], col)
        outs.append((float(tot), [p.detach().clone() for p in m.para_list]))
    assert outs[0][0] == outs[1][0]
    for a, b in zip(outs[0][1], outs[1][1]):
        assert torch.equal(a, b)


def _oracle_for(m, sets, encoder, loss, n, H, L, lr, clip):
    r = no.OracleNCNModel(sets, num_nodes=n, emb_hidden=H, gnn_hidden=H, mlp_hidden=H, gnn_layers=2, mlp_layers=L,
                          encoder=encoder, loss=loss, lr=lr, clip_norm=clip, dtype=torch.float64, optimizer="SGD")
    state = {"emb": m.emb.weight}
    state.update({"enc." + k[len("convs."):]: v for k, v in m.encoder.state_dict().items()})
    state.update({"pred." + k[len("lins."):]: v for k, v in m.predictor.state_dict().items()})
    assert set(state) == set(r.params)
    r.load({k: v.detach().cpu().double() for k, v in state.items()})
    return r


@pytest.mark.parametrize("loss", ["AUC", "HingeAUC"])
@pytest.mark.parametrize("encoder", ["SAGE", "GCN"])
def test_train_matches_oracle_trajectory(encoder, loss, monkeypatch):
    from plnlp_b200 import graph
    monkeypatch.setattr(graph, "DENSE_SPMM", False)
    n, H, L, B, k, lr, clip = 600, 16, 2, 48, 3, 0.01, 2.0
    d, o, ei = _data(encoder, n)
    torch.manual_seed(7)
    m = _model(encoder, loss, n, H, L, lr=lr, clip=clip)
    m.param_init()
    if encoder == "GCN":
        m.num_nodes = 10 ** 9                                   # batches restrict the last conv
    r = _oracle_for(m, no.sets_of(d.adj_t), encoder, loss, n, H, L, lr, clip)
    pos = ei.t()[:3 * B].contiguous()
    g = torch.Generator().manual_seed(11)
    negs = torch.randint(0, n, (pos.size(0), k, 2), generator=g)
    perms = [torch.arange(i * B, (i + 1) * B) for i in range(3)]
    got = m.train(d, {"train": {"edge": pos}}, B, "global", k, perms=perms, neg_edges=negs)
    want = r.train_epoch(None, o, pos, negs, perms, k)
    assert abs(got - want) <= TOL * abs(want), (got, want)
    named = {"emb": m.emb.weight}
    named.update({"enc." + k_[len("convs."):]: v for k_, v in m.encoder.named_parameters()})
    named.update({"pred." + k_[len("lins."):]: v for k_, v in m.predictor.named_parameters()})
    names = list(named)
    _params_close([named[k] for k in names], [r.params[k] for k in names], names)


def test_test_matches_metrics_of_oracle_scores():
    from plnlp_b200.utils import evaluate_hits, evaluate_mrr
    n, H, L = 600, 16, 2
    d, o, ei = _data("SAGE", n)
    torch.manual_seed(9)
    m = _model("SAGE", "AUC", n, H, L)
    m.param_init()
    g = torch.Generator().manual_seed(4)
    e = lambda P_: torch.randint(0, n, (P_, 2), generator=g)      # noqa: E731
    neg = e(400)
    neg[:20, 0] = -1                                               # the mean row
    split = {"train": {"edge": ei.t()[:10]}, "valid": {"edge": ei.t()[:200], "edge_neg": neg},
             "test": {"edge": ei.t()[200:400], "edge_neg": e(400)}}
    res = m.test(d, split, 64, None, "hits")
    m.encoder.eval(); m.predictor.eval()
    hg = m.encode_for_test(d)
    h = hg.cpu().double()
    lins = [(lin.weight.detach().cpu().double(), lin.bias.detach().cpu().double()) for lin in m.predictor.lins]
    sets = no.sets_of(d.adj_t)
    edges = (split["valid"]["edge"], split["valid"]["edge_neg"], split["test"]["edge"], split["test"]["edge_neg"])
    got = [m.batch_predict(hg, x, 64, adj_t=d.adj_t).cpu() for x in edges]
    ref = [no.score(h, x, no.lists(sets, x), lins) for x in edges]
    delta = 0.0
    for a, b in zip(got, ref):
        ok, msg = fp32_close(a, b.float(), b, TOL)
        assert ok, msg
        delta = max(delta, float((a.double() - b).abs().max()))
    # test() is evaluate_hits of those scores, exactly
    assert res == evaluate_hits(None, *got)
    # and against the oracle's scores a positive can change sides only where it lies within 2 delta of the K-th
    # negative (the threshold itself moves by at most delta)
    want = evaluate_hits(None, *[r.float() for r in ref])
    assert set(res) == set(want)
    for key in res:
        K = int(key.split("@")[1])
        for i, (pos, neg) in enumerate(((ref[0], ref[1]), (ref[2], ref[3]))):
            thr = torch.topk(neg, K).values[-1]
            near = int(((pos - thr).abs() <= 2 * delta).sum())
            assert abs(res[key][i] - want[key][i]) <= near / pos.numel() + 1e-12, (key, res[key], want[key], near)
    # MRR format: source / target / target_node_neg
    S = 100
    src = torch.randint(0, n, (S,), generator=g)
    msplit = {"train": {"source_node": src, "target_node": src}}
    for name in ("valid", "test"):
        msplit[name] = {"source_node": torch.randint(0, n, (S,), generator=g),
                        "target_node": torch.randint(0, n, (S,), generator=g),
                        "target_node_neg": torch.randint(0, n, (S, 20), generator=g)}
    res = m.test(d, msplit, 64, None, "mrr")
    got = []
    for name in ("valid", "test"):
        sp = msplit[name]
        pe = torch.stack([sp["source_node"], sp["target_node"]], 1)
        ne = torch.stack([sp["source_node"].repeat_interleave(20), sp["target_node_neg"].reshape(-1)], 1)
        for x in (pe, ne):
            a = m.batch_predict(hg, x, 64, adj_t=d.adj_t).cpu()
            b = no.score(h, x, no.lists(sets, x), lins)
            ok, msg = fp32_close(a, b.float(), b, TOL)
            assert ok, msg
            got.append(a)
    assert res == evaluate_mrr(None, *got)
    # batch_predict without the graph is refused
    with pytest.raises(ValueError):
        m.batch_predict(m.encode_for_test(d), split["valid"]["edge"], 64)


def test_unsupported_calls_raise():
    n, H = 300, 16
    d, _, ei = _data("SAGE", n)
    m = _model("SAGE", "AUC", n, H)
    m.param_init()
    q = torch.arange(5, device="cuda")
    with pytest.raises(NotImplementedError, match="NCN"):
        m.recommend(d, q, 10)
    with pytest.raises(NotImplementedError, match="NCN"):
        m.rank_against_all(d, torch.stack([q, q + 1], 1))
    m.partitioned = True
    pos = ei.t()[:8].contiguous().cuda()
    with pytest.raises(NotImplementedError, match="NCN"):
        m.train_batch(d, pos, pos, 1)
    with pytest.raises(NotImplementedError, match="NCN"):
        m.prepare_batch(d, pos, pos)
    with pytest.raises(NotImplementedError, match="NCN"):
        m.test(d, {"train": {"edge": pos}, "valid": {"edge": pos, "edge_neg": pos},
                   "test": {"edge": pos, "edge_neg": pos}}, 64, None, "hits")

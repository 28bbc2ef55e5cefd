"""The Transformer encoder on the row-partitioned model (-m gpu).

* ``plnlp_attn_score_csr_f32`` against ``plnlp_edge_dot_fwd_f32`` over the stacked table [q; k], bit for bit, and its
  argument checks.
* Virtual shards in one process (``TransformerConv.forward_block`` per shard, the gathered input shared, so autograd
  sums every shard's input gradient as the reduce-scatter would), R = 1, 2, 3 and a split with an empty block,
  against the single-GPU encoder with an fp64 oracle as the yardstick.
* One-rank NCCL runs (two ranks where two GPUs exist) of a training step (``selfcheck.partitioned_step``) for the
  Transformer, SAGE and WSAGE encoders, of ``encode_for_test`` and of ``recommend``.
"""
import ctypes
import math
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import plnlp_ref, sparse
from tests.helpers import fp32_close, rand_graph

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda")
TOL = 1e-5


# ----------------------------------------------------------------------------------------------- the score kernel
def _block(n_q, n_k, degrees, g):
    """CSR block [n_q, n_k] whose rows have the given numbers of entries (repeated over the rows)"""
    deg = torch.tensor([degrees[i % len(degrees)] for i in range(n_q)])
    rowptr = torch.zeros(n_q + 1, dtype=torch.int64)
    rowptr[1:] = torch.cumsum(deg, 0)
    col = torch.randint(0, n_k, (int(rowptr[-1]),), generator=g)
    return rowptr.to(DEV), col.to(DEV)


@pytest.mark.parametrize("F", [1, 7, 16, 50, 200, 256, 512])
def test_score_kernel_matches_edge_dot_on_the_stacked_table(F):
    from plnlp_b200 import _ops
    from plnlp_b200.graph import build_plan
    g = torch.Generator().manual_seed(F)
    n_q, n_k = 37, 211
    rowptr, col = _block(n_q, n_k, [0, 1, 33, 150, 5, 0, 64, 65], g)     # 150 > chunk: split across work items
    plan = build_plan(rowptr, col, None, n_q, n_k, chunk=64)
    assert plan.n_items > n_q
    row = torch.repeat_interleave(torch.arange(n_q, device=DEV), rowptr[1:] - rowptr[:-1])
    pairs = torch.stack([row, col + n_q], 1)
    for ld in (F, F + 3, ((F + 3) // 4) * 4 + 4):
        table = torch.randn(n_q + n_k, ld, generator=g).to(DEV)[:, :F]
        q, k = table[:n_q], table[n_q:]
        got = _ops.attn_score_raw(plan, q, k)
        want = _ops.edge_dot_raw(table, pairs)
        assert torch.equal(got, want), (F, ld)
        ref = (q.double()[row] * k.double()[col]).sum(1)
        assert float((got.double() - ref).abs().max()) <= 1e-5 * max(float(ref.abs().max()), 1.0)


def test_score_kernel_rejects_invalid_arguments():
    from plnlp_b200 import _lib
    from plnlp_b200.graph import build_plan
    lib = _lib.load()
    g = torch.Generator().manual_seed(1)
    rowptr, col = _block(8, 9, [3], g)
    plan = build_plan(rowptr, col, None, 8, 9)
    q, k, s = torch.randn(8, 16, device=DEV), torch.randn(9, 16, device=DEV), torch.empty(24, device=DEV)
    P = lambda t: t.data_ptr()  # noqa: E731
    args = [P(plan.item_ptr), P(plan.item_row), plan.n_items, P(plan.col), P(q), 16, P(k), 16, 16, P(s), None]
    fn = lib.plnlp_attn_score_csr_f32
    assert fn(*args) == 0
    torch.cuda.synchronize()
    for i in (0, 1, 3, 4, 6, 9):                                   # every pointer is required
        bad = list(args)
        bad[i] = None
        assert fn(*bad) == -1, i
    for i, v in ((2, -1), (8, 0), (8, -4), (5, 15), (7, 8)):       # negative sizes, F <= 0, ld < F
        bad = list(args)
        bad[i] = v
        assert fn(*bad) == -2, (i, v)
    empty = list(args)
    empty[2] = 0
    empty[0] = empty[1] = empty[3] = None
    assert fn(*empty) == 0                                          # nothing to do: no pointer needed


# ----------------------------------------------------------------------------------------------- virtual shards
def _graph(n, seed=9):
    from plnlp_b200.graph import CSRGraph
    ei, _ = rand_graph(n, 10 * n, seed=seed, hub=True)
    ei = ei[:, ei[0] != ei[1]]
    return CSRGraph.from_edge_index(torch.cat([ei, ei.flip(0)], 1).to(DEV), None, n).to_symmetric()


def test_block_attention_one_shard_is_the_single_gpu_composition():
    """same q, k, v: the R = 1 block attention (scores, weights, aggregate) equals EdgeDot -> SegmentSoftmax ->
    SpMMValues of the single-GPU conv bit for bit"""
    from plnlp_b200 import _ops, parallel
    from plnlp_b200.graph import CSRGraph, structure_of
    adj = _graph(301)
    local = parallel.shard_graph(adj, 0, 1, CSRGraph).local
    g = torch.Generator().manual_seed(2)
    for F in (16, 50, 200):
        q = torch.randn(301, F, generator=g).to(DEV)
        kv = torch.randn(301, 2 * F, generator=g).to(DEV)
        k, v = kv[:, :F], kv[:, F:]
        scale = 1.0 / math.sqrt(F)
        with torch.no_grad():
            s, alpha, agg = _ops.block_attention_fwd(q, k, v, structure_of(local), scale)
            st = structure_of(adj)
            s1 = _ops.EdgeDot.apply(torch.cat([q, k], 0), st.entry_pairs())
            a1 = _ops.SegmentSoftmax.apply(s1, st.rowptr, scale)
            agg1 = _ops.SpMMValues.apply(a1, v, adj)
        assert torch.equal(s, s1) and torch.equal(alpha, a1) and torch.equal(agg, agg1), F


def _virtual_encoder(enc, parts, adj, R):
    """the row-partitioned encoder played by one process: every shard runs ``forward_block`` on its rows, the gathered
    matrix of a layer is the concatenation of the shards' padded blocks -> [N, H]"""
    from plnlp_b200 import _ops, parallel
    from plnlp_b200.graph import CSRGraph
    n = adj.size(0)
    blk = parallel.block_size(n, R)
    locals_ = [parallel.shard_graph(adj, r, R, CSRGraph).local for r in range(R)]
    full = [parallel.pad_rows(p, R * blk) for p in parts]
    last = len(enc.convs) - 1
    for i, conv in enumerate(enc.convs):
        act = _ops.ACT_RELU if (i < last or enc.num_layers == 1) else _ops.ACT_NONE
        outs = [conv.forward_block([p[r * blk:(r + 1) * blk] for p in full], full, locals_[r], act) for r in range(R)]
        full = [torch.cat(outs, 0)]
    return full[0][:n]


def _oracle_encoder(enc, parts, adj):
    """fp64 oracle of the same encoder -> (out, {param name: grad}, grad of the first input block)"""
    rowptr, col, _ = adj.csr()
    o = sparse.SparseTensor(rowptr=rowptr.cpu(), col=col.cpu(), value=None, sparse_sizes=(adj.size(0), adj.size(1)),
                            is_sorted=True)
    layers = []
    for i, conv in enumerate(enc.convs):
        layers.append({k: v.detach().double().cpu().requires_grad_(True) for k, v in conv.named_parameters()})
    x0 = parts[0].detach().double().cpu().requires_grad_(True)
    x = torch.cat([x0] + [p.detach().double().cpu() for p in parts[1:]], 1)
    out = plnlp_ref.encoder_forward("TRANSFORMER", layers, x, o)
    return out, layers, x0


@pytest.mark.parametrize("R,N", [(1, 301), (2, 301), (3, 301), (8, 49)])      # (8, 49): blocks of 7, the last empty
@pytest.mark.parametrize("L", [1, 2])
@pytest.mark.parametrize("with_x", [False, True])
def test_virtual_shards_match_single_gpu(R, N, L, with_x):
    from plnlp_b200 import parallel
    from plnlp_b200.layer import Transformer, mark_constant
    if N == 49:
        assert parallel.row_block(N, R - 1, R) == (N, N)
    adj = _graph(N, seed=N)
    g = torch.Generator().manual_seed(L + 10 * R)
    emb = torch.randn(N, 12, generator=g).to(DEV).requires_grad_(True)
    parts = [emb] + ([mark_constant(torch.randn(N, 8, generator=g).to(DEV))] if with_x else [])
    torch.manual_seed(0)
    enc = Transformer(12 + (8 if with_x else 0), 32, 32, L, 0.0).to(DEV)
    gout = torch.randn(N, 32, generator=g).to(DEV)

    def run(fn):
        for p in enc.parameters():
            p.grad = None
        emb.grad = None
        y = fn()
        y.backward(gout)
        return y.detach(), emb.grad.clone(), {k: p.grad.clone() for k, p in enc.named_parameters()}

    y1, ge1, gp1 = run(lambda: enc(parts, adj))
    yv, gev, gpv = run(lambda: _virtual_encoder(enc, parts, adj, R))
    out64, layers64, x064 = _oracle_encoder(enc, parts, adj)
    out64.backward(gout.double().cpu())
    ok, msg = fp32_close(yv, y1, out64)
    assert ok, ("forward", msg)
    ok, msg = fp32_close(gev, ge1, x064.grad)
    assert ok, ("input grad", msg)
    # lin_key.bias moves every score of a row by the same amount, which the softmax ignores: its exact gradient is 0,
    # judged with the absolute floor of test_transformer_against_reference_golden
    floor = 2 * TOL * max(float(p.grad.abs().max()) for lay in layers64 for p in lay.values())
    for name, got in gpv.items():
        i, pname = name.split(".", 2)[1], name.split(".", 2)[2]
        ok, msg = fp32_close(got, gp1[name], layers64[int(i)][pname].grad, floor=floor)
        assert ok, (name, msg)


# ----------------------------------------------------------------------------------------------- NCCL runs
N_NODES, FEATS, EMB, HID, BATCH, K = 301, 8, 16, 32, 48, 2


class Data:
    pass


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _norm_graph(dev):
    from plnlp_b200.graph import CSRGraph
    from plnlp_b200.utils import gcn_normalization
    ei, _ = rand_graph(N_NODES, 3000, seed=9, hub=True)
    ei = ei[:, ei[0] != ei[1]]
    return gcn_normalization(CSRGraph.from_edge_index(torch.cat([ei, ei.flip(0)], 1).to(dev), None, N_NODES).to_symmetric())


def _models(rank, ws, dev, adj, predictor="MLP"):
    """a single-GPU Transformer model and its row-partitioned copy (same parameters) with their data objects"""
    from plnlp_b200 import parallel
    from plnlp_b200.graph import CSRGraph
    from plnlp_b200.model import BaseModel
    blk = parallel.block_size(N_NODES, ws)
    lo, hi = parallel.row_block(N_NODES, rank, ws)

    def make(n):
        torch.manual_seed(3)
        m = BaseModel(lr=0.01, dropout=0.0, grad_clip_norm=-1.0, gnn_num_layers=2, mlp_num_layers=2,
                      emb_hidden_channels=EMB, gnn_hidden_channels=HID, mlp_hidden_channels=HID, num_nodes=n,
                      num_node_feats=FEATS, gnn_encoder_name="Transformer", predictor_name=predictor, loss_func="AUC",
                      optimizer_name="Adam", device=dev, use_node_feats=True, train_node_emb=True)
        m.param_init()
        return m
    single, part = make(N_NODES), make(blk)
    with torch.no_grad():
        for a, b in zip(part.para_list, single.para_list):
            if a.shape == b.shape:
                a.copy_(b)
        part.emb.weight.zero_()
        part.emb.weight[: hi - lo].copy_(single.emb.weight[lo:hi])
    part.world_size, part.rank, part.partitioned = ws, rank, True
    part.num_nodes = N_NODES
    x = torch.randn(N_NODES, FEATS, generator=torch.Generator().manual_seed(4)).to(dev)
    d1, d2 = Data(), Data()
    d1.adj_t, d1.x, d1.edge_index = adj, x, None
    d2.adj_t, d2.edge_index = parallel.shard_graph(adj, rank, ws, CSRGraph), None
    d2.x = parallel.pad_rows(x[lo:hi].contiguous(), blk)
    return single, part, d1, d2


def _worker(rank, ws, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=ws, device_id=dev)
    try:
        from plnlp_b200 import selfcheck
        from plnlp_b200.graph import CSRGraph
        adj = _norm_graph(dev)
        out = {}
        for encoder in ("Transformer", "SAGE", "WSAGE"):
            for force_sparse in (False, True):
                errs = selfcheck.partitioned_step(rank, ws, dev, adj=CSRGraph(*adj.csr(), (N_NODES, N_NODES)),
                                                  feats=FEATS, emb=EMB, hid=HID, batch=BATCH, k=K, encoder=encoder,
                                                  force_sparse=force_sparse, keep=True)
                out[f"step/{encoder}/{force_sparse}"] = errs["_tensors"]
        single, part, d1, d2 = _models(rank, ws, dev, adj)
        for m in (single, part):
            m.encoder.eval()
            m.predictor.eval()
        out["encode"] = (part.encode_for_test(d2).cpu(), single.encode_for_test(d1).cpu())
        nodes = torch.randint(0, N_NODES, (23,), generator=torch.Generator().manual_seed(5)).to(dev)
        got = part.recommend(d2, nodes, 10, exclude="adj")
        want = single.recommend(d1, nodes, 10, exclude="adj")
        out["recommend"] = ([t.cpu() for t in got], [t.cpu() for t in want])
        ret[rank] = out
    finally:
        dist.destroy_process_group()


def _oracle_step(encoder, inputs, adj_csr):
    """fp64 CPU oracle of the step selfcheck.partitioned_step takes -> (loss, {name: grad})"""
    ref = plnlp_ref.OracleModel(num_nodes=N_NODES, emb_hidden=EMB, gnn_hidden=HID, mlp_hidden=HID, gnn_layers=2,
                                mlp_layers=2, encoder=encoder.upper(), predictor="MLP", loss="AUC", lr=0.01,
                                clip_norm=-1.0, num_node_feats=FEATS, use_node_feats=True, dtype=torch.float64)
    # the oracle's own initialisation names SAGE / GCN parameters only: take the model's, by name
    ref.params = {k: v.double().clone().requires_grad_(True) for k, v in inputs["state"].items()}
    ref._make_optimizer()
    rowptr, col, val = adj_csr
    adj = sparse.SparseTensor(rowptr=rowptr, col=col, value=val.double(), sparse_sizes=(N_NODES, N_NODES), is_sorted=True)
    rloss, _ = ref.step(inputs["x"].double(), adj, inputs["pos"], inputs["neg"], K, None, do_update=False)
    return float(rloss), {k: p.grad for k, p in ref.params.items()}


def _check(ret, ws):
    from plnlp_b200 import parallel
    adj_csr = tuple(t.cpu() for t in _norm_graph(torch.device("cuda", 0)).csr())
    for r in range(ws):
        lo, hi = parallel.row_block(N_NODES, r, ws)
        out = ret[r]
        for case, T in out.items():
            if not case.startswith("step/"):
                continue
            rloss, rg = _oracle_step(case.split("/")[1], T["inputs"], adj_csr)
            assert abs(T["part"]["loss"] - rloss) <= 1e-5 * abs(rloss), (case, T["part"]["loss"], rloss)
            floor = 2 * TOL * max(float(v.abs().max()) for v in rg.values())
            for name, got in T["part"].items():
                if name == "loss":
                    continue
                key = name if name == "emb" else name.replace("enc.convs.", "enc.").replace("pred.lins.", "pred.")
                want64 = rg[key][lo:hi] if name == "emb" else rg[key]
                ok, msg = fp32_close(got, T["single"][name], want64, floor=floor)
                assert ok, (r, case, name, msg)
        h_part, h_single = out["encode"]
        assert h_part.shape == h_single.shape
        assert float((h_part - h_single).abs().max()) <= 1e-5 * float(h_single.abs().max())
        (ids, scores), (ids1, scores1) = out["recommend"]
        assert ids.shape == ids1.shape == (23, 10)
        row_max = scores1.abs().amax(1, keepdim=True).clamp_min(1e-30)
        assert bool(((scores - scores1).abs() <= 1e-5 * row_max).all())


def test_partitioned_transformer_one_rank_nccl():
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(1, _free_port(), ret), nprocs=1, join=True)
    _check(ret, 1)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_partitioned_transformer_two_ranks_nccl():
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(2, _free_port(), ret), nprocs=2, join=True)
    _check(ret, 2)

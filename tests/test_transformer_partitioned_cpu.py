"""CPU tests (-m "not gpu") of the row-partitioned TransformerConv over torch.distributed gloo: the data flow of the
conv (all-gather of every input block, key / value over all gathered rows, queries and the skip term on the local
rows, reduce-scatter of the input gradients) with the dense linears and the block attention replaced by their
reference restatements in fp64 -- the CUDA kernels behind them are checked on the GPU
(tests/test_gpu_transformer_partitioned.py).  Parity target: ``oracle.plnlp_ref.conv_forward('TRANSFORMER', ...)`` on
the whole graph in one process."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import plnlp_ref, sparse
from tests.helpers import rand_graph, rel_err

EMB, FEATS, OUT = 5, 3, 4


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _oracle_graph(rowptr, col, val, sizes):
    return sparse.SparseTensor(rowptr=rowptr, col=col, value=val, sparse_sizes=sizes, is_sorted=True)


def _oracle_attention(q, kv, adj, scale):
    """oracle/pyg.py TransformerConv's attention on a rectangular row block: queries of the block's rows, keys and
    values of every column"""
    row, col, _ = adj.coo()
    F = q.size(1)
    k, v = kv[:, :F], kv[:, F:]
    score = (q[row] * k[col]).sum(-1) * scale
    n = q.size(0)
    mx = torch.full((n,), float("-inf"), dtype=score.dtype).scatter_reduce(0, row, score, "amax", include_self=True)
    e = torch.exp(score - mx[row])
    alpha = e / torch.zeros(n, dtype=score.dtype).index_add_(0, row, e)[row]
    return torch.zeros(n, F, dtype=q.dtype).index_add_(0, row, alpha.unsqueeze(-1) * v[col])


def _cpu_fused_linear(xs, ws, bias=None, act=0, drop_p=0.0, seed=0, addend=None):
    """what _ops.fused_linear computes, in torch on the CPU"""
    y = sum(x @ w.t() for x, w in zip(xs, ws))
    if bias is not None:
        y = y + bias
    if addend is not None:
        y = y + addend
    return torch.relu(y) if act == 1 else y


def _graph(N):
    ei, _ = rand_graph(N, 12 * N, seed=4, hub=True)
    return sparse.to_sparse_tensor(ei, None, N)               # the reference feeds the Transformer a value-less adj


def _inputs(N):
    g = torch.Generator().manual_seed(6)
    return (torch.randn(N, EMB, generator=g, dtype=torch.float64), torch.randn(N, FEATS, generator=g, dtype=torch.float64),
            torch.randn(N, OUT, generator=g, dtype=torch.float64))


def _conv():
    from plnlp_b200.layer import TransformerConv
    torch.manual_seed(0)
    return TransformerConv(EMB + FEATS, OUT).double()


def _worker(rank, ws, port, N, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=ws)
    try:
        from plnlp_b200 import _ops, layer, parallel
        _ops.fused_linear = _cpu_fused_linear                 # this process only
        gathers = []
        real_gather = parallel.all_gather_rows

        def counting_gather(x, group=None, name="", **kw):
            gathers.append(name)
            return real_gather(x, group, name=name, **kw)
        parallel.all_gather_rows = counting_gather

        E, X, G = _inputs(N)
        blk = parallel.block_size(N, ws)
        lo, hi = parallel.row_block(N, rank, ws)
        sadj = parallel.shard_graph(_graph(N), rank, ws, _oracle_graph)
        conv = _conv()
        emb = parallel.pad_rows(E[lo:hi].clone(), blk).requires_grad_(True)
        x = layer.mark_constant(parallel.pad_rows(X[lo:hi].clone(), blk))
        y = conv((emb, x), sadj, attention=_oracle_attention)
        assert y.shape == (blk, OUT)
        y.backward(parallel.pad_rows(G[lo:hi], blk))
        out = {"y": y.detach()[: hi - lo], "gemb": emb.grad[: hi - lo].clone(), "gpad": emb.grad[hi - lo:].clone(),
               "gparams": {k: p.grad.clone() for k, p in conv.named_parameters()}}
        # the constant block is gathered once and kept while it is unchanged ...
        const = [n for n in gathers if "constant" in n]
        full = layer._gather_input(x, sadj)
        conv((emb, x), sadj, attention=_oracle_attention)
        out["const_gathers_before_write"] = len([n for n in gathers if "constant" in n])
        out["same_object"] = layer._gather_input(x, sadj) is full
        # ... and gathered again after an in-place write
        x.mul_(2.0)
        again = layer._gather_input(x, sadj)
        out["const_gathers_after_write"] = len([n for n in gathers if "constant" in n])
        out["first_const_gathers"] = len(const)
        out["rewritten_rows"] = again[lo:hi].clone()
        ret[rank] = out
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("ws,N", [(2, 37), (3, 31), (3, 4)])       # (3, 4): blocks of 2, 2 and 0 rows
def test_partitioned_transformer_conv_matches_single_process_gloo(ws, N):
    from plnlp_b200 import parallel
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(ws, _free_port(), N, ret), nprocs=ws, join=True)
    E, X, G = _inputs(N)
    conv = _conv()
    p = {k: v.detach().clone().requires_grad_(True) for k, v in conv.named_parameters()}
    e = E.clone().requires_grad_(True)
    y = plnlp_ref.conv_forward("TRANSFORMER", p, torch.cat([e, X], 1), _graph(N))
    y.backward(G)
    for r in range(ws):
        lo, hi = parallel.row_block(N, r, ws)
        out = ret[r]
        assert rel_err(out["y"], y.detach()[lo:hi]) < 1e-12, r
        assert rel_err(out["gemb"], e.grad[lo:hi]) < 1e-12, r
        assert torch.all(out["gpad"] == 0), r                 # padding rows receive no gradient
        assert out["first_const_gathers"] == 1 and out["const_gathers_before_write"] == 1, out
        assert out["same_object"] and out["const_gathers_after_write"] == 2, out
        assert torch.equal(out["rewritten_rows"], 2.0 * X[lo:hi])
    # every rank holds its own share of each parameter gradient; their sum is the whole graph's (allreduce_grads)
    for name, want in p.items():
        got = sum(ret[r]["gparams"][name] for r in range(ws))
        assert rel_err(got, want.grad) < 1e-12 or float((got - want.grad).abs().max()) < 1e-12, name

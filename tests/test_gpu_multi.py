"""Multi-GPU parity (-m gpu, needs >= 2 GPUs; skipped otherwise): the row-partitioned SpMM with the CUDA
kernel as the local operator over NCCL, and one full training step of the partitioned / data-parallel
model, against the single-GPU result (SURVEY.md section 8e: index work identical, fp32 within
tolerance because the summation order changes).

Gradients are judged like the single-GPU parity tests judge theirs (``helpers.fp32_close``): within 1e-5 of an
fp64 oracle of the same step, or no further from it than a small multiple of the SINGLE-GPU run's own fp32
rounding error -- the yardstick for sums that cancel (the predictor-bias gradients of a pairwise loss whose
d loss / d score sums to zero), where "relative to the tensor's own magnitude" measures noise against noise."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests.helpers import fp32_close, rand_graph, rel_err

pytestmark = pytest.mark.gpu

N_NODES, FEATS, EMB, HID, BATCH, K = 301, 8, 16, 32, 48, 2


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _graph(dev):
    from plnlp_b200.graph import CSRGraph
    from plnlp_b200.utils import gcn_normalization
    ei, _ = rand_graph(N_NODES, 3000, seed=9, hub=True)
    ei = ei[:, ei[0] != ei[1]]
    return gcn_normalization(CSRGraph.from_edge_index(torch.cat([ei, ei.flip(0)], 1).to(dev), None, N_NODES).to_symmetric())


def _worker(rank, ws, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=ws, device_id=dev)
    try:
        from plnlp_b200 import _ops, parallel, selfcheck
        from plnlp_b200.graph import CSRGraph
        N, F = N_NODES, 24
        adj = _graph(dev)
        g = torch.Generator().manual_seed(1)
        x, gout = torch.randn(N, F, generator=g).to(dev), torch.randn(N, F, generator=g).to(dev)
        lo, hi = parallel.row_block(N, rank, ws)
        blk = parallel.block_size(N, ws)
        sadj = parallel.shard_graph(adj, rank, ws, CSRGraph)
        assert sadj.local_t is sadj.local                       # the prepared graph is bit-symmetric
        # ---- partitioned SpMM vs single GPU
        xr = x.clone().requires_grad_(True)
        y = _ops.spmm(adj, xr, "sum")
        y.backward(gout)
        xl = x[lo:hi].clone().requires_grad_(True)
        yl = _ops.spmm(sadj, xl, "sum")
        gl = torch.zeros(blk, F, device=dev)
        gl[: hi - lo] = gout[lo:hi]
        yl.backward(gl)
        out = {"spmm": {"fwd": rel_err(yl[: hi - lo], y[lo:hi]), "bwd": rel_err(xl.grad, xr.grad[lo:hi])}}
        # ---- one training step, every way the partitioned model can take it
        adj2 = CSRGraph(*adj.csr(), (N, N))                     # fresh object: no cached dense form
        cases = {"restricted": dict(force_sparse=True),          # union of endpoint rows, column-block partial products
                 "restricted_allreduce": dict(force_sparse=True),    # ... combined by all-reduce instead of RS + AG
                 "rows": dict(force_sparse=False),               # full last conv + compact endpoint-row exchange
                 "allgather": dict(force_sparse=False),          # full last conv + whole-matrix all-gather
                 "sparse_grad_only": dict(force_sparse=True),    # full last conv, row-sparse backward
                 "restricted_CE": dict(force_sparse=True, loss="CE")}   # a MEAN loss: gradients are averaged
        for name, kw in cases.items():
            parallel.EXCHANGE = "allgather" if name == "allgather" else "rows"
            parallel.RESTRICT_LAST = name != "sparse_grad_only"
            parallel.RESTRICT_COMBINE = "ar" if name == "restricted_allreduce" else "rs"
            errs = selfcheck.partitioned_step(rank, ws, dev, adj=adj2, feats=FEATS, emb=EMB, hid=HID, batch=BATCH,
                                              k=K, keep=True, **kw)
            out[name] = errs
        parallel.EXCHANGE, parallel.RESTRICT_LAST, parallel.RESTRICT_COMBINE = "rows", True, "rs"
        assert "_plnlp_agg_buffer" in adj2.__dict__
        ret[rank] = out
    finally:
        dist.destroy_process_group()


def _oracle_grads(inputs, adj_csr, loss):
    """fp64 CPU oracle of the same step -> {tensor name: gradient}"""
    from oracle import plnlp_ref, sparse
    ref = plnlp_ref.OracleModel(num_nodes=N_NODES, emb_hidden=EMB, gnn_hidden=HID, mlp_hidden=HID, gnn_layers=2,
                                mlp_layers=2, encoder="GCN", predictor="MLP", loss=loss, lr=0.01, clip_norm=-1.0,
                                num_node_feats=FEATS, use_node_feats=True, dtype=torch.float64)
    ref.load({k: v.double() for k, v in inputs["state"].items()})
    rowptr, col, val = adj_csr
    adj = sparse.SparseTensor(rowptr=rowptr, col=col, value=val.double(), sparse_sizes=(N_NODES, N_NODES), is_sorted=True)
    rloss, _ = ref.step(inputs["x"].double(), adj, inputs["pos"], inputs["neg"], K, None, do_update=False)
    return float(rloss), {k: p.grad for k, p in ref.params.items()}


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_partitioned_matches_single_gpu_nccl_ws2():
    from plnlp_b200 import parallel
    ws = 2
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(ws, _free_port(), ret), nprocs=ws, join=True)
    adj_csr = tuple(t.cpu() for t in _graph(torch.device("cuda", 0)).csr())
    report = []
    for r in range(ws):
        out = ret[r]
        assert out["spmm"]["fwd"] < 1e-6 and out["spmm"]["bwd"] < 2e-5, out["spmm"]
        lo, hi = parallel.row_block(N_NODES, r, ws)
        for case, errs in out.items():
            if case == "spmm":
                continue
            T = errs["_tensors"]
            loss = "CE" if case.endswith("_CE") else "AUC"
            rloss, rg = _oracle_grads(T["inputs"], adj_csr, loss)
            assert abs(T["part"]["loss"] - rloss) <= 1e-5 * abs(rloss), (case, T["part"]["loss"], rloss)
            floor = 1e-5 * max(float(v.abs().max()) for v in rg.values())
            for name, got in T["part"].items():
                if name == "loss":
                    continue
                key = name if name == "emb" else (name.replace("enc.convs.", "enc.").replace("pred.lins.", "pred."))
                want64 = rg[key][lo:hi] if name == "emb" else rg[key]
                ok, msg = fp32_close(got, T["single"][name], want64, floor=floor)
                report.append(f"rank {r} {case:18s} {name:24s} {msg}")
                assert ok, (r, case, name, msg)
    print("\n".join(report))          # per-tensor errors, shown with pytest -rP


def _dp_worker(rank, ws, port, ret):
    """data-parallel edge batches on a replicated encoder (ddi / collab shape): SAGE + MLP, a SUM loss and a MEAN loss"""
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=ws, device_id=dev)
    try:
        from plnlp_b200 import selfcheck
        from plnlp_b200.graph import CSRGraph
        ei, _ = rand_graph(N_NODES, 3000, seed=9, hub=True)
        adj = CSRGraph.from_edge_index(torch.cat([ei, ei.flip(0)], 1).to(dev), None, N_NODES)
        g = torch.Generator().manual_seed(3)
        pos_all = torch.randint(0, N_NODES, (ws * BATCH, 2), generator=g).to(dev)
        neg_all = torch.randint(0, N_NODES, (ws * BATCH, K, 2), generator=g).to(dev)
        out = {}
        for loss in ("AUC", "CE"):
            torch.manual_seed(11)
            single = selfcheck._model(N_NODES, 0, EMB, HID, dev, "SAGE", loss)
            torch.manual_seed(11)
            dp = selfcheck._model(N_NODES, 0, EMB, HID, dev, "SAGE", loss)
            dp.world_size, dp.rank = ws, rank
            d = selfcheck._Data()
            d.adj_t, d.x, d.edge_index = adj, None, None
            l1 = single.train_batch(d, pos_all, neg_all.reshape(-1, 2), K)
            sl = slice(rank * BATCH, (rank + 1) * BATCH)
            l2 = dp.train_batch(d, pos_all[sl], neg_all[sl].reshape(-1, 2), K).clone()
            dist.all_reduce(l2)
            if loss == "CE":
                l2 /= ws
            errs = {"loss": abs(float(l2) - float(l1)) / abs(float(l1))}
            scale = max(float(p.grad.abs().max()) for p in single.para_list)
            for a, b in zip(dp.para_list, single.para_list):
                errs[len(errs)] = float((a.grad - b.grad).abs().max()) / scale
            out[loss] = errs
        ret[rank] = out
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_data_parallel_edge_batches_sum_and_mean_losses_nccl_ws2():
    """ADVICE r1: a MEAN loss must be averaged over ranks, a SUM loss summed -- both then equal the single-GPU
    gradient of the global batch (errors on the model-wide gradient scale)"""
    ws = 2
    ret = mp.Manager().dict()
    mp.spawn(_dp_worker, args=(ws, _free_port(), ret), nprocs=ws, join=True)
    for r in range(ws):
        for loss, errs in ret[r].items():
            for k, v in errs.items():
                assert v < 2e-5, (r, loss, k, v)

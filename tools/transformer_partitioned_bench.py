"""Time the training step of the row-partitioned model with the Transformer encoder at the citation2 shape (2 x
TransformerConv 200, MLP head, 65 536 positives per global step, 3 local negatives each), built and partitioned the
way bench.measure does it.

Usage: torchrun --nproc_per_node R tools/transformer_partitioned_bench.py [--steps 5] [--out FILE]
(without torchrun: one rank, a one-rank NCCL group)

Prints one JSON line from rank 0: the card's name and power limit; ms per training step (CUDA events around
``--steps`` steps that end in a device synchronise, after a warm-up, the profiler off, max over ranks); the per-kernel
split of one instrumented step per rank (plnlp_b200.profiling spans: all-gathers of the conv inputs, the k|v GEMMs
forward and backward, the other GEMMs, the score kernel, softmax, the attention SpMMs, reduce-scatters, the rest); the
parity check of ``selfcheck.partitioned_step`` with this encoder.  On one rank the single-GPU Transformer step is timed
in the same call, alternating with the partitioned one."""
import argparse
import json
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
import bench  # noqa: E402
from plnlp_b200 import parallel, profiling, selfcheck  # noqa: E402
from plnlp_b200.graph import CSRGraph  # noqa: E402
from plnlp_b200.utils import gcn_normalization  # noqa: E402
from tools.recommend_bench import gpu_info  # noqa: E402


def split_of(spans, n_kv):
    """the per-kernel split of one instrumented step on this rank; ``n_kv``: the width of the stacked k|v (2F)"""
    keys = ("gather", "kv_gemm", "other_gemm", "score", "softmax", "attention_spmm", "reduce_scatter", "other")
    out = {k + "_ms": 0.0 for k in keys}
    for name, s in spans.items():
        if "all_gather" in name:
            k = "gather"
        elif "reduce_scatter" in name:
            k = "reduce_scatter"
        elif name.startswith("gemm"):
            dims = [int(d) for d in name.split()[1].split("x")]
            k = "kv_gemm" if n_kv in dims else "other_gemm"
        elif name.startswith("attn_score_csr"):
            k = "score"
        elif name.startswith("segment_softmax"):
            k = "softmax"
        elif name.startswith("spmm_csr"):
            k = "attention_spmm"
        else:
            k = "other"
        out[k + "_ms"] += s["ms"]
    out["total_instrumented_ms"] = sum(out.values())
    return {k: round(v, 3) for k, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the partitioned and single-GPU step (R = 1)")
    ap.add_argument("--out", default=None, help="also append the JSON line to this file (rank 0)")
    a = ap.parse_args()

    if "RANK" not in os.environ:
        os.environ.update(RANK="0", WORLD_SIZE="1", LOCAL_RANK="0", MASTER_ADDR="127.0.0.1", MASTER_PORT="29534")
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    try:
        info = gpu_info() if rank == 0 else None
        # parity first, on the small synthetic graph of bench.py's check, with this encoder
        errs = selfcheck.summarize(selfcheck.partitioned_step(rank, world, dev, encoder="Transformer"))
        parity = {}
        for key in ("loss_rel", "max_grad_rel", "max_grad_rel_per_tensor", "fp32_noise_floor"):
            t = torch.tensor([errs[key]], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            parity[key] = float(t)
        torch.cuda.empty_cache()

        cfg = dict(bench.WORKLOADS["citation2"], encoder="Transformer")     # value-less adjacency (main.py:181-184)
        N, B, k = cfg["N"], cfg["batch"], cfg["num_neg"]
        torch.manual_seed(0)
        data, split = bench.build_workload(cfg, dev, CSRGraph, gcn_normalization)
        full_adj, full_x = data.adj_t, data.x
        blk = parallel.block_size(N, world)
        lo, hi = parallel.row_block(N, rank, world)
        pdata = bench.Data()
        pdata.adj_t = parallel.shard_graph(full_adj, rank, world, CSRGraph, symmetric=True)
        pdata.x = parallel.pad_rows(full_x[lo:hi].contiguous(), blk)
        pdata.edge_index = data.edge_index
        torch.manual_seed(0)
        model = bench.make_model(dict(cfg, N=blk), dev)
        model.num_nodes, model.partitioned, model.world_size, model.rank = N, True, world, rank
        single = None
        if world == 1:
            torch.manual_seed(0)
            single = bench.make_model(cfg, dev)
        else:
            del full_adj, full_x
            data = None
        torch.cuda.empty_cache()
        pos_all = torch.stack([split["train"]["source_node"], split["train"]["target_node"]], 1)
        Bl = B // world
        g = torch.Generator(device=dev).manual_seed(1000 + rank)

        def batches(n):
            idx = torch.randint(0, pos_all.size(0), (n * Bl,), generator=g, device=dev)
            pos = pos_all[idx]
            neg = torch.stack([pos[:, :1].expand(-1, k), torch.randint(0, N, (n * Bl, k), generator=g, device=dev)], 2)
            return [(pos[i * Bl:(i + 1) * Bl], neg[i * Bl:(i + 1) * Bl].reshape(-1, 2)) for i in range(n)]

        def run(m, d, n):
            m.encoder.train()
            m.predictor.train()
            bs = batches(n)
            dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for pos, neg in bs:
                m.train_batch(d, pos, neg, k)
            e1.record()
            torch.cuda.synchronize()
            t = torch.tensor([e0.elapsed_time(e1) / n], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t)

        run(model, pdata, a.warmup)
        if single is not None:
            run(single, data, a.warmup)
        part_ms, single_ms = [], []
        for _ in range(a.rounds if single is not None else 1):
            part_ms.append(run(model, pdata, a.steps))
            if single is not None:
                single_ms.append(run(single, data, a.steps))
        profiling.enable()
        run(model, pdata, 1)
        split_part = split_of(profiling.disable(), 2 * cfg["hid"])
        splits = [None] * world
        dist.all_gather_object(splits, split_part)
        split_single = None
        if single is not None:
            profiling.enable()
            run(single, data, 1)
            split_single = {k_: round(v["ms"], 3) for k_, v in sorted(profiling.disable().items(),
                                                                        key=lambda kv: -kv[1]["ms"])[:12]}
        if rank == 0:
            res = {"workload": "citation2-shape Transformer", "N": N, "nnz": int(pdata.adj_t.local.nnz()) if world == 1
                   else None, "ranks": world, "block_rows": blk, "encoder": "2 x TransformerConv 200, MLP head",
                   "global_batch": B, "num_neg": k, "gpu": info,
                   "partitioned_ms_per_step": [round(x, 2) for x in part_ms],
                   "timing": f"CUDA events around {a.steps} training steps after {a.warmup} warm-up steps, profiler "
                             "off, max over ranks",
                   "split_one_instrumented_step_per_rank": splits,
                   "parity_check": dict(parity, what="selfcheck.partitioned_step(encoder='Transformer'): one step on a "
                                                     "60 000-node graph vs the single-GPU model; max over ranks")}
            if single is not None:
                res["single_gpu_ms_per_step"] = [round(x, 2) for x in single_ms]
                res["single_gpu_alternated"] = "the two step kinds alternate, one list entry per round"
                res["single_gpu_top_spans_ms"] = split_single
            line = json.dumps(res)
            print(line, flush=True)
            if a.out:
                os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
                with open(a.out, "a") as f:
                    f.write(line + "\n")
    finally:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

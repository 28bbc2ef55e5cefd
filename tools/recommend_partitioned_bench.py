"""Time candidate-sharded link recommendation (BaseModel.recommend / rank_against_all on a row-partitioned model) at
the citation2 shape, built and partitioned the way bench.measure does it.

Usage: torchrun --nproc_per_node R tools/recommend_partitioned_bench.py [--runs DOT:100:1000,MLP:100:20]
       [--candidates COUNT] [--out FILE]
(without torchrun: one rank, a one-rank NCCL group)

Prints one JSON line per run from rank 0: the card's name and power limit, ms per query of both calls (CUDA events
around calls that end in a device synchronise, after a warm-up, the profiler off), and per rank the split of one
instrumented ``recommend`` call (plnlp_b200.profiling spans): score GEMM / fused MLP (ms, TFLOP/s), mask + select,
exclusion build, exchange (query rows, all-gather of the top-k lists) and merge, encode of the row block.
``--candidates COUNT`` restricts every run to COUNT distinct random nodes (the same on every rank); the lines then
gain a "candidates" field."""
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
from plnlp_b200 import parallel, profiling, recommend  # noqa: E402
from plnlp_b200.graph import CSRGraph  # noqa: E402
from plnlp_b200.utils import gcn_normalization  # noqa: E402
from tools.recommend_bench import gpu_info, timed  # noqa: E402


def split_of(spans, nb):
    """the per-kernel split of one instrumented call on this rank"""
    out = {"score_ms": 0.0, "score_flops": 0, "select_ms": 0.0, "mask_ms": 0.0, "merge_ms": 0.0, "exclusion_ms": 0.0,
           "exchange_ms": 0.0, "encode_ms": 0.0}
    for name, s in spans.items():
        if name.startswith("edge_mlp_fwd_fused") or (name.startswith("gemm") and f"x{nb}x" in name):
            out["score_ms"] += s["ms"]
            out["score_flops"] += s["flops"]
        elif name.startswith("topk_rows_f32"):
            out["select_ms"] += s["ms"]
        elif name.startswith("score_mask_f32"):
            out["mask_ms"] += s["ms"]
        elif name.startswith("topk_merge_f32"):
            out["merge_ms"] += s["ms"]
        elif name == "recommend: exclusion CSR":
            out["exclusion_ms"] += s["ms"]
        elif name.startswith("recommend: exchange"):
            out["exchange_ms"] += s["ms"]
        elif name == "recommend: encode (row block)":
            out["encode_ms"] += s["ms"]
    out["score_tflops"] = round(out.pop("score_flops") / max(out["score_ms"], 1e-9) / 1e9, 1)
    return {k: round(v, 3) for k, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", default="DOT:100:1000,DOT:100:8000,MLP:100:20",
                    help="comma-separated PREDICTOR:K:QUERIES")
    ap.add_argument("--exclude", default="adj", choices=["adj", "none"])
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--candidates", type=int, default=None, help="restrict to this many random nodes")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file (rank 0)")
    a = ap.parse_args()

    if "RANK" not in os.environ:
        os.environ.update(RANK="0", WORLD_SIZE="1", LOCAL_RANK="0", MASTER_ADDR="127.0.0.1", MASTER_PORT="29533")
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    try:
        cfg = dict(bench.WORKLOADS["citation2"])
        N = cfg["N"]
        torch.manual_seed(0)
        data, _ = bench.build_workload(cfg, dev, CSRGraph, gcn_normalization)
        blk = parallel.block_size(N, world)
        lo, hi = parallel.row_block(N, rank, world)
        data.adj_t = parallel.shard_graph(data.adj_t, rank, world, CSRGraph, symmetric=True)
        data.x = parallel.pad_rows(data.x[lo:hi].contiguous(), blk)
        torch.cuda.empty_cache()
        exclude = None if a.exclude == "none" else "adj"
        info = gpu_info() if rank == 0 else None
        for run in a.runs.split(","):
            predictor, k, Q = run.split(":")
            k, Q = int(k), int(Q)
            model = bench.make_model(dict(cfg, N=blk, predictor=predictor), dev)
            model.num_nodes, model.partitioned, model.world_size, model.rank = N, True, world, rank
            g = torch.Generator(device=dev).manual_seed(3)       # the same queries on every rank
            nodes = torch.randint(0, N, (Q,), generator=g, device=dev)
            edges = torch.stack([nodes, torch.randint(0, N, (Q,), generator=g, device=dev)], 1)
            cand, width = None, hi - lo
            if a.candidates is not None:
                cand = torch.unique(torch.randperm(N, generator=g, device=dev)[:a.candidates])
                x, y = recommend.candidate_slices(cand, [(lo, hi)])[0]
                width = y - x
            rec = lambda: model.recommend(data, nodes, k, exclude=exclude, candidates=cand)          # noqa: E731
            rnk = lambda: model.rank_against_all(data, edges, exclude=exclude, candidates=cand)      # noqa: E731
            rec()                                                                    # warm-up
            rnk()
            dist.barrier()
            rec_ms, (ids, _) = timed(rec, a.reps)
            dist.barrier()
            rank_ms, _ = timed(rnk, a.reps)
            profiling.enable()
            rec()
            split = split_of(profiling.disable(), width)
            splits = [None] * world
            dist.all_gather_object(splits, split)
            times = torch.tensor([rec_ms, rank_ms], dtype=torch.float64, device=dev)
            dist.all_reduce(times, op=dist.ReduceOp.MAX)
            if rank == 0:
                res = {"workload": cfg["name"], "N": N, "ranks": world, "block_rows": blk, "predictor": predictor,
                       "queries": Q, "k": k, "exclude": a.exclude, "gpu": info,
                       "recommend": {"ms": round(float(times[0]), 3), "ms_per_query": round(float(times[0]) / Q, 5)},
                       "rank_against_all": {"ms": round(float(times[1]), 3),
                                            "ms_per_query": round(float(times[1]) / Q, 5)},
                       "timing": f"CUDA events on rank 0 around {a.reps} calls, max over ranks",
                       "split_one_recommend_call_per_rank": splits,
                       "valid_ids_first_row": int((ids[0] >= 0).sum())}
                if cand is not None:
                    res["candidates"] = cand.numel()
                line = json.dumps(res)
                print(line, flush=True)
                if a.out:
                    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
                    with open(a.out, "a") as f:
                        f.write(line + "\n")
            del model
            torch.cuda.empty_cache()
    finally:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

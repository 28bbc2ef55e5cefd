"""Time link recommendation over all nodes (BaseModel.recommend / rank_against_all) at the BASELINE graph shapes.

Usage: python tools/recommend_bench.py [citation2|ddi|collab] --predictor DOT|MLP --queries Q --k K
       [--candidates COUNT] [--out FILE]

Prints one JSON line: ms per query and candidate pairs/s of both calls (timed with CUDA events after a warm-up, the
profiler off), then the per-kernel split of one instrumented ``recommend`` call (plnlp_b200.profiling spans): the
score GEMM's TFLOP/s and the select kernel's GB/s and share of the HBM copy peak (bytes = passes x Q x N x 4; the
select reads each score row once).  The card's name and power limit come from a read-only nvidia-smi query.  With the
MLP head at citation2 shape every query costs 2 H H1 FLOP per candidate: the run times the given sample of queries and
the all-nodes figure is an extrapolation, labelled as such.  ``--candidates COUNT`` restricts both calls to COUNT
distinct random nodes (seeded): pairs, GEMM width and select bytes then count |C| candidates per query, and the line
gains a "candidates" field."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from plnlp_b200 import profiling  # noqa: E402
from plnlp_b200.graph import CSRGraph  # noqa: E402
from plnlp_b200.utils import full_rank_metrics, gcn_normalization  # noqa: E402

HBM_PEAK_GBS = 7700.0          # HGX B200 data sheet, one GPU
SELECT_PASSES = 1              # plnlp_topk_rows_f32 reads each score row once


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:      # the numbers still stand; say that the card could not be read
        return {"error": repr(e)}


def timed(fn, reps):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("workload", nargs="?", default="citation2", choices=sorted(bench.WORKLOADS))
    ap.add_argument("--predictor", default="DOT", choices=["DOT", "MLP"])
    ap.add_argument("--queries", type=int, default=1000)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--exclude", default="adj", choices=["adj", "none"])
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--candidates", type=int, default=None, help="restrict to this many random nodes")
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    a = ap.parse_args()

    dev = torch.device("cuda")
    cfg = dict(bench.WORKLOADS[a.workload], predictor=a.predictor)
    torch.manual_seed(0)
    data, _ = bench.build_workload(cfg, dev, CSRGraph, gcn_normalization)
    model = bench.make_model(cfg, dev)
    N, Q = cfg["N"], a.queries
    exclude = None if a.exclude == "none" else "adj"
    g = torch.Generator(device=dev).manual_seed(3)
    nodes = torch.randint(0, N, (Q,), generator=g, device=dev)
    edges = torch.stack([nodes, torch.randint(0, N, (Q,), generator=g, device=dev)], 1)
    cand, W = None, N
    if a.candidates is not None:
        cand = torch.randperm(N, generator=g, device=dev)[:a.candidates]
        W = cand.numel()

    rec = lambda: model.recommend(data, nodes, a.k, exclude=exclude, candidates=cand)          # noqa: E731
    rank = lambda: model.rank_against_all(data, edges, exclude=exclude, candidates=cand)      # noqa: E731
    rec()                                                                    # warm-up: every shape the timing uses
    rank()
    enc_ms, _ = timed(lambda: model.encode_for_test(data), a.reps)
    rec_ms, (ids, _) = timed(rec, a.reps)
    rank_ms, ranks = timed(rank, a.reps)

    profiling.enable()
    rec()
    spans = profiling.disable()
    gemm = {"ms": 0.0, "flops": 0}
    select = {"ms": 0.0, "n": 0}
    other = {}
    for name, s in spans.items():
        if name.startswith("gemm") or name.startswith("edge_mlp_fwd_fused"):
            if "x{}x".format(W) in name or name.startswith("edge_mlp_fwd_fused"):   # the score chunks, not the encoder
                gemm["ms"] += s["ms"]
                gemm["flops"] += s["flops"]
                continue
        if name.startswith("topk_rows_f32"):
            select["ms"] += s["ms"]
            select["n"] += s["n"]
            continue
        other[name] = round(s["ms"], 3)
    sel_bytes = SELECT_PASSES * Q * W * 4
    res = {
        "workload": cfg["name"], "N": N, "predictor": a.predictor, "queries": Q, "k": a.k, "exclude": a.exclude,
        "gpu": gpu_info(),
        "encode_ms": round(enc_ms, 3),
        "recommend": {"ms": round(rec_ms, 3), "ms_per_query": round(rec_ms / Q, 5),
                      "pairs_per_s": round(Q * W / rec_ms * 1e3)},
        "rank_against_all": {"ms": round(rank_ms, 3), "ms_per_query": round(rank_ms / Q, 5),
                             "pairs_per_s": round(Q * W / rank_ms * 1e3),
                             "metrics_random_targets": {k: round(v, 6) for k, v in full_rank_metrics(ranks).items()}},
        "split_one_recommend_call": {
            "score_ms": round(gemm["ms"], 3), "score_ms_per_query": round(gemm["ms"] / Q, 5),
            "score_tflops": round(gemm["flops"] / max(gemm["ms"], 1e-9) / 1e9, 1),
            "select_ms": round(select["ms"], 3), "select_ms_per_query": round(select["ms"] / Q, 5),
            "select_passes": SELECT_PASSES, "select_gbs": round(sel_bytes / max(select["ms"], 1e-9) / 1e6, 1),
            "select_frac_hbm_peak": round(sel_bytes / max(select["ms"], 1e-9) / 1e6 / HBM_PEAK_GBS, 3),
            "hbm_peak_gbs_datasheet": HBM_PEAK_GBS, "other_ms": other},
        "all_nodes_extrapolated_s": {"recommend": round(rec_ms / Q * N / 1e3, 1),
                                     "rank_against_all": round(rank_ms / Q * N / 1e3, 1),
                                     "note": f"extrapolated from {Q} timed queries to all {N} nodes"},
        "valid_ids_first_row": int((ids[0] >= 0).sum()),
    }
    if cand is not None:
        res["candidates"] = W
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

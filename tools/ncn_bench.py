"""Time the NCN predictor (layer.NCNPredictor, heuristics.common_neighbour_lists) against the MLP head on a BASELINE
graph shape.

Usage: python tools/ncn_bench.py [citation2|collab|ddi] [--steps K] [--warmup W] [--eval-sources S] [--out FILE]

The graph, encoder and hyper-parameters are bench.py's (``build_workload``, ``make_model``); only the predictor
changes.  One seeded set of training batches (bench's batch size, uniform positives, negatives as the workload's
sampler draws them) is fed to both models through ``BaseModel.run_batches``.  Prints one JSON line:
  * the card's name and power limit (a read-only nvidia-smi query);
  * ms per training step with MLP and with NCN (W warm-up steps, then K timed steps between CUDA events; the MLP
    is timed again after NCN, so the spread of the same code is visible);
  * the per-kernel split of the NCN head for one batch (plnlp_b200.profiling spans: count, fill, plan build,
    aggregate SpMM forward and backward, the MLP GEMMs and the rest), from a separate instrumented pass;
  * common-neighbour list entries per batch, and the rows the restricted last conv computes with and without them;
  * ``BaseModel.test`` pairs/s on the eval splits of tools/heuristics_bench.py (citation2-shape: the first S
    sources of each split, labelled);
  * a bit-for-bit check of the lists of a seeded sample of batch pairs against Python sets built from the raw
    stored rows of the adjacency."""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
from heuristics_bench import build_splits  # noqa: E402
from plnlp_b200 import heuristics, model as M, profiling  # noqa: E402
from plnlp_b200.graph import CSRGraph  # noqa: E402
from plnlp_b200.utils import gcn_normalization  # noqa: E402
from recommend_bench import gpu_info  # noqa: E402

SAMPLE = 2000


def make_batches(cfg, split, n_batches, dev):
    tr = split["train"]
    pos_all = tr["edge"] if "edge" in tr else torch.stack([tr["source_node"], tr["target_node"]], 1)
    g = torch.Generator(device=dev).manual_seed(5)
    B, k, N = cfg["batch"], cfg["num_neg"], cfg["N"]
    out = []
    for _ in range(n_batches):
        pos = pos_all[torch.randint(0, pos_all.size(0), (B,), generator=g, device=dev)].to(dev)
        dst = torch.randint(0, N, (B * k,), generator=g, device=dev)
        if cfg["sampler"] == "local":
            src = pos[:, 0].repeat_interleave(k)
        else:
            src = torch.randint(0, N, (B * k,), generator=g, device=dev)
        out.append((pos, torch.stack([src, dst], 1), None))
    return out


def time_steps(m, data, batches, warmup, k):
    m.encoder.train(); m.predictor.train()
    m.run_batches(data, iter(batches[:warmup]), k)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    m.run_batches(data, iter(batches[warmup:]), k)
    e1.record()
    torch.cuda.synchronize()
    return round(e0.elapsed_time(e1) / (len(batches) - warmup), 3)


def head_split(m, data, batch):
    """profiling spans of the NCN head alone on one batch: lists, then forward + backward of score_edges on the
    encoder output"""
    with torch.no_grad():
        h = m.encoder(m.input_parts(data), data.adj_t)
    h = h.detach().requires_grad_(True)
    e = torch.cat([batch[0], batch[1]], 0)
    torch.cuda.synchronize()
    profiling.enable()
    with profiling.span("NCN head total (lists + forward + backward)"):
        cn = heuristics.common_neighbour_lists(data.adj_t, e)
        m.predictor.score_edges(h, e, cn).sum().backward()
    spans = profiling.disable()
    return {name: {"n": v["n"], "ms": round(v["ms"], 3)} for name, v in sorted(spans.items())}, cn


def check_lists(adj, e, cn, dev):
    g = torch.Generator(device=dev).manual_seed(8)
    idx = torch.randint(0, e.size(0), (SAMPLE,), generator=g, device=dev)
    rowptr, col, _ = adj.csr()
    rowptr, col = rowptr.cpu().tolist(), col.cpu().tolist()
    r, c = cn[0].cpu().tolist(), cn[1].cpu().tolist()
    nb = lambda u: set(col[rowptr[u]:rowptr[u + 1]]) - {u}      # noqa: E731
    equal = nonempty = 0
    for p, (u, v) in zip(idx.tolist(), e[idx].cpu().tolist()):
        want = sorted(nb(u) & nb(v))
        equal += c[r[p]:r[p + 1]] == want
        nonempty += bool(want)
    return {"pairs": SAMPLE, "bit_equal": equal, "nonempty": nonempty}


def eval_rate(m, data, which, N, dev, S):
    split, metric = build_splits(which, N, dev)
    label = "full splits"
    if which == "citation2":
        for name in ("valid", "test"):
            split[name] = {k: v[:S] for k, v in split[name].items()}
        label = f"first {S} sources x 1000 negatives of each split"
    split["train"] = {"source_node": None} if metric == "mrr" else {"edge": None}     # selects the split format
    if metric == "mrr":
        pairs = sum(split[s]["source_node"].numel() + split[s]["target_node_neg"].numel() for s in ("valid", "test"))
    else:
        pairs = sum(split[s]["edge"].size(0) + split[s]["edge_neg"].size(0) for s in ("valid", "test"))
    m.test(data, split, 65536, None, metric)                   # warm-up
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    res = m.test(data, split, 65536, None, metric)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    return {"splits": label, "pairs": pairs, "ms": round(ms, 1), "pairs_per_s": round(pairs / ms * 1e3),
            "result": res}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("workload", nargs="?", default="citation2", choices=sorted(bench.WORKLOADS))
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--eval-sources", type=int, default=8192)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda")
    cfg = dict(bench.WORKLOADS[args.workload])
    torch.manual_seed(0)
    data, split = bench.build_workload(cfg, dev, CSRGraph, gcn_normalization)
    batches = make_batches(cfg, split, args.warmup + args.steps, dev)
    out = {"tool": "ncn_bench", "workload": bench.workload_label(cfg), "gpu": gpu_info(),
           "steps": args.steps, "warmup": args.warmup}
    models = {}
    for pred in ("MLP", "NCN"):
        torch.manual_seed(0)
        models[pred] = bench.make_model(dict(cfg, predictor=pred), dev)
    k = cfg["num_neg"]
    t = {"MLP": time_steps(models["MLP"], data, batches, args.warmup, k),
         "NCN": time_steps(models["NCN"], data, batches, args.warmup, k)}
    t["MLP_again"] = time_steps(models["MLP"], data, batches, args.warmup, k)
    out["ms_per_step"] = t
    out["ncn_over_mlp"] = round(t["NCN"] / min(t["MLP"], t["MLP_again"]), 3)
    m = models["NCN"]
    split_spans, cn = head_split(m, data, batches[0])
    out["ncn_head_split_one_batch"] = split_spans
    e = torch.cat([batches[0][0], batches[0][1]], 0)
    out["pairs_per_batch"] = e.size(0)
    out["cn_entries_per_batch"] = int(cn[0][-1])
    ends = torch.unique(e.reshape(-1)).numel()
    ids, _, _ = M.ncn_restrict(e, cn)
    out["restricted_rows"] = {"endpoints": ends, "endpoints_and_common_neighbours": ids.numel(),
                              "row_sparse_batch": m._sparse_rows(batches[0][0], batches[0][1]),
                              "num_nodes": cfg["N"]}
    out["list_check"] = check_lists(data.adj_t, e, cn, dev)
    out["test"] = {p: eval_rate(models[p], data, args.workload, cfg["N"], dev, args.eval_sources)
                   for p in ("MLP", "NCN")}
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

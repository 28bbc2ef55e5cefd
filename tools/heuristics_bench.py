"""Time the common-neighbour link heuristics (plnlp_b200/heuristics.py) on the eval splits of a BASELINE graph shape.

Usage: python tools/heuristics_bench.py [citation2|collab|ddi] --method CN|AA|RA [--reps R]

The graph and the valid / test splits are built as tools/eval_bench.py builds them: citation2-shape = 86 596 sources
x 1 000 negatives per split (MRR), the others 133 489 positives + 100 000 negatives per split (Hits@K).  Prints one
JSON line:
  * the card's name and power limit (a read-only nvidia-smi query);
  * the neighbour-table build time (cleaned CSR + weights, the cache cleared before each of R builds; median);
  * per split, the scoring time of all its pairs (positives and negatives, CUDA events, median of R after a warm-up)
    and pairs/s, plus one ``heuristics.test`` call end to end with its result;
  * the index bytes the pairs touch, from the degrees of the cleaned table: per pair 16 B of edge, 32 B of row
    pointers and 4 B per entry of both neighbour lists (all of them on the merge path; an upper bound where the
    kernel binary-searches the longer list);
  * the agreement with the oracle's rules (oracle/heuristics.py) on a seeded sample of 10 000 test pairs, recomputed
    on the CPU from the raw stored rows of the adjacency: how many are bit-equal, and the largest difference in fp32
    ulps."""
import argparse
import json
import math
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
from oracle import heuristics as oh  # noqa: E402
from plnlp_b200 import heuristics  # noqa: E402
from plnlp_b200.graph import CSRGraph  # noqa: E402
from plnlp_b200.utils import gcn_normalization, get_pos_neg_edges  # noqa: E402
from recommend_bench import gpu_info, timed  # noqa: E402

SAMPLE = 10000


def build_splits(which, N, dev):
    """the eval splits of tools/eval_bench.py -> (split dict, metric)"""
    g = torch.Generator(device=dev).manual_seed(3)
    split = {}
    if which == "citation2":
        S, K = 86596, 1000
        for name in ("valid", "test"):
            split[name] = {"source_node": torch.randint(0, N, (S,), generator=g, device=dev),
                           "target_node": torch.randint(0, N, (S,), generator=g, device=dev),
                           "target_node_neg": torch.randint(0, N, (S, K), generator=g, device=dev)}
        return split, "mrr"
    P, Q = 133489, 100000
    for name in ("valid", "test"):
        split[name] = {"edge": torch.randint(0, N, (P, 2), generator=g, device=dev),
                       "edge_neg": torch.randint(0, N, (Q, 2), generator=g, device=dev)}
    return split, "hits"


def oracle_sample(adj, edges, method):
    """fp32 [S]: the oracle's rules on the CPU for the pairs ``edges``, from the raw stored rows of ``adj``"""
    rowptr, col, _ = adj.csr()
    rowptr, col = rowptr.cpu().numpy(), col.cpu().numpy()

    def nbrs(u):
        return set(col[rowptr[u]:rowptr[u + 1]].tolist()) - {u}
    out = []
    for u, v in edges.cpu().tolist():
        common = nbrs(u) & nbrs(v)
        out.append(math.fsum(oh.term(method, len(nbrs(w))) for w in sorted(common)))
    return torch.from_numpy(np.array(out, dtype=np.float64).astype(np.float32))


def two_hop_pairs(table, dev):
    """SAMPLE seeded pairs (u, v) with v a neighbour of a neighbour of u: pairs that do share neighbours"""
    g = torch.Generator(device=dev).manual_seed(6)
    has = torch.nonzero(table.deg > 0).reshape(-1)
    u = has[torch.randint(0, has.numel(), (SAMPLE,), generator=g, device=dev)]

    def step(x):
        off = (torch.rand(SAMPLE, generator=g, device=dev) * table.deg[x]).to(torch.int64)
        return table.col[table.rowptr[x] + off].to(torch.int64)
    x = step(u)
    return torch.stack([u, step(x)], 1)


def agreement(adj, edges, method):
    got = heuristics.score_edges(adj, edges, method).cpu()
    want = oracle_sample(adj, edges, method)
    ulp = (got.view(torch.int32).to(torch.int64) - want.view(torch.int32).to(torch.int64)).abs()
    return {"pairs": edges.size(0), "bit_equal": int((ulp == 0).sum()), "max_ulp": int(ulp.max()),
            "nonzero_scores": int((want != 0).sum())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("workload", nargs="?", default="citation2", choices=["citation2", "collab", "ddi"])
    ap.add_argument("--method", default="CN", choices=list(heuristics.METHODS))
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    dev = torch.device("cuda")
    cfg = dict(bench.WORKLOADS[args.workload])
    torch.manual_seed(0)
    data, split = bench.build_workload(cfg, dev, CSRGraph, gcn_normalization)
    N = cfg["N"]
    eval_split, metric = build_splits(args.workload, N, dev)
    split.update(eval_split)
    adj = data.adj_t

    builds = []
    for _ in range(args.reps + 1):
        heuristics._CACHE.clear()
        ms, table = timed(lambda: heuristics.neighbour_table(adj).weight(args.method), 1)
        builds.append(ms)
    table = heuristics.neighbour_table(adj)

    res = {"workload": cfg["name"], "gpu": gpu_info(), "method": args.method, "N": N,
           "table": {"build_ms_median": round(float(np.median(builds[1:])), 2), "build_ms_first": round(builds[0], 2),
                     "stored_entries": adj.nnz(), "cleaned_entries": table.col.numel()},
           "splits": {}}
    deg = table.deg
    for name in ("valid", "test"):
        pos, neg = get_pos_neg_edges(name, split, device=dev)
        e = torch.cat([pos, neg.reshape(-1, 2)])
        heuristics.score_edges(adj, e, args.method)                    # warm-up
        times = [timed(lambda: heuristics.score_edges(adj, e, args.method), 1)[0] for _ in range(args.reps)]
        ms = float(np.median(times))
        d = deg[e[:, 0]] + deg[e[:, 1]]
        index_bytes = int(e.size(0)) * (16 + 32) + 4 * int(d.sum())
        res["splits"][name] = {"pairs": int(e.size(0)), "ms_median": round(ms, 3), "ms_all": [round(t, 3) for t in times],
                               "pairs_per_s": round(e.size(0) / ms * 1e3), "index_bytes": index_bytes,
                               "index_GB_per_s": round(index_bytes / ms / 1e6, 1)}
    ms, out = timed(lambda: heuristics.test(data, split, args.method, None, None, metric), 1)
    res["test_call"] = {"ms": round(ms, 2), "result": {k: [round(v, 5) for v in vs] for k, vs in out.items()}}

    pos, neg = get_pos_neg_edges("test", split, device=dev)
    e = torch.cat([pos, neg.reshape(-1, 2)])
    pick = torch.randint(0, e.size(0), (SAMPLE,), generator=torch.Generator(device=dev).manual_seed(5), device=dev)
    res["oracle_sample"] = agreement(adj, e[pick], args.method)
    res["oracle_sample_two_hop"] = agreement(adj, two_hop_pairs(table, dev), args.method)
    print(json.dumps(res))


if __name__ == "__main__":
    main()

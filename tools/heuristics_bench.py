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
    ulps.

With ``--queries Q [--k K]`` it times heuristic recommendation instead (``heuristics.recommend`` with exclude='adj'
on Q seeded query nodes, and ``heuristics.rank_against_all`` on the first Q (source, target) pairs of the test split)
and prints one JSON line with: the first call including the table builds (cleaned CSR, transpose, weights) and the
median of R cached calls (CUDA events); the per-kernel split of one instrumented call of each (plnlp_b200.profiling
spans: mark, score, mask, select); the marked (two-hop) pairs per query -- the pairs the score kernel intersects,
against N pairs per query for ``score_edges`` over every (u, j); the time of that pair-by-pair workaround for
``--pair-queries`` of the queries, timed in the same call; and a bit-for-bit check of a sample of the returned scores
against ``score_edges``.  ``--partitioned`` (under torchrun; one rank without it) runs the collective calls on
``parallel.shard_graph`` and checks them against the single-GPU calls on the same rank.

With ``--method Katz|PPR`` (``--beta/--hops`` or ``--alpha/--iters``) it times the path-based scores (paths.py) and
prints one JSON line with: per hop of one block of 256 sources, the kernel time (CUDA events), the live-row fraction
of the state it reads, the bytes it gathers (the live rows' state entries, every column index and live byte, the
output) and those bytes/s against the 7.7 TB/s data-sheet peak; the eval-split pairs/s of ``score_edges`` over the
pairs of ``--sources`` distinct test sources (a labelled subset; the full-split time is extrapolated linearly and
labelled so); ``recommend`` per-query time on 256 queries with its kernel split; and the agreement of a sample of
scores with the fp64 series computed on the CPU with scipy from the cleaned reach table.  ``--partitioned`` runs the
collective calls as above and checks them against one GPU."""
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
from plnlp_b200 import _ops, heuristics, profiling  # noqa: E402
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


_POPCOUNT = None


def marked_pairs(table, nodes, chunk=64):
    """the bits the mark kernel sets for ``nodes`` over all columns: the (query, j) pairs the score kernel
    intersects"""
    global _POPCOUNT
    if _POPCOUNT is None:
        _POPCOUNT = torch.tensor([bin(i).count("1") for i in range(256)], dtype=torch.int64, device=nodes.device)
    rr, rc = table.reach()
    total = 0
    for i in range(0, nodes.numel(), chunk):
        bm = _ops.two_hop_mark_raw(table.rowptr, table.col, rr, rc, nodes[i:i + chunk], table.n)
        total += int(_POPCOUNT[bm.view(torch.uint8).to(torch.int64)].sum())
    return total


def split_of(spans):
    return {name: {"n": v["n"], "ms": round(v["ms"], 3)} for name, v in sorted(spans.items())}


def recommend_main(args, cfg, data, split, dev):
    import torch.distributed as dist
    N = cfg["N"]
    adj = data.adj_t
    graph = adj
    if args.partitioned:
        from plnlp_b200 import parallel
        if "RANK" not in os.environ:
            os.environ.update(RANK="0", WORLD_SIZE="1", LOCAL_RANK="0", MASTER_ADDR="127.0.0.1", MASTER_PORT="29541")
        dist.init_process_group("nccl", device_id=dev)
        graph = parallel.shard_graph(adj, dist.get_rank(), dist.get_world_size(), CSRGraph, symmetric=True)
    g = torch.Generator(device=dev).manual_seed(7)
    nodes = torch.randint(0, N, (args.queries,), generator=g, device=dev)
    pos, _ = get_pos_neg_edges("test", split, device=dev)
    edges = pos[:args.queries].contiguous()
    m, k = args.method, args.k
    rec = lambda: heuristics.recommend(graph, nodes, k, m, "adj")           # noqa: E731
    rank = lambda: heuristics.rank_against_all(graph, edges, m, "adj")      # noqa: E731
    res = {"workload": cfg["name"], "gpu": gpu_info(), "method": m, "N": N, "queries": args.queries, "k": k,
           "exclude": "adj", "partitioned": bool(args.partitioned),
           "ranks": dist.get_world_size() if args.partitioned else 1}
    for name, fn in (("recommend", rec), ("rank_against_all", rank)):
        heuristics._CACHE.clear()
        first, out = timed(fn, 1)
        times = [timed(fn, 1)[0] for _ in range(args.reps)]
        profiling.enable()
        fn()
        spans = profiling.disable()
        res[name] = {"first_call_ms_with_table_builds": round(first, 2), "ms_median": round(float(np.median(times)), 2),
                     "ms_all": [round(t, 2) for t in times],
                     "ms_per_query": round(float(np.median(times)) / args.queries, 4), "split": split_of(spans)}
        res[name + "_out"] = out
    ids, scores = res.pop("recommend_out")
    ranks = res.pop("rank_against_all_out")
    res["rank_against_all"]["mrr"] = round(float((1.0 / ranks).mean()), 5)
    res["rank_against_all"]["targets_scoring_0"] = int((heuristics.score_edges(graph, edges, m) == 0).sum())
    table = heuristics.neighbour_table(adj)
    marked = marked_pairs(table, nodes)
    res["two_hop"] = {"marked_pairs_per_query": round(marked / args.queries, 1), "all_pairs_per_query": N,
                      "share": round(marked / args.queries / N, 6)}
    # the returned scores against score_edges, bit for bit
    sample = min(args.queries, 64)
    live = ids[:sample] >= 0
    pairs = torch.stack([nodes[:sample, None].expand(-1, k)[live], ids[:sample][live]], 1)
    want = heuristics.score_edges(graph, pairs, m)
    res["score_edges_check"] = {"pairs": int(pairs.size(0)),
                                "bit_equal": int((want.view(torch.int32) == scores[:sample][live].view(torch.int32)).sum())}
    if args.partitioned:
        si, ss = heuristics.recommend(adj, nodes, k, m, "adj")
        sr = heuristics.rank_against_all(adj, edges, m, "adj")
        res["single_gpu_check"] = {"ids_equal": bool(torch.equal(si, ids)), "scores_equal": bool(torch.equal(ss, scores)),
                                   "ranks_equal": bool(torch.equal(sr, ranks))}
    else:
        # the pair-by-pair workaround: score_edges over every (u, j), then the same top-k select, for a few queries
        Qp = min(args.pair_queries, args.queries)
        j = torch.arange(N, device=dev)

        def pairwise():
            out = []
            for u in nodes[:Qp].tolist():
                S = heuristics.score_edges(adj, torch.stack([torch.full_like(j, u), j], 1), m).reshape(1, N)
                out.append(_ops.topk_rows_raw(S, k)[0])
            return out
        pairwise()
        ms, _ = timed(pairwise, 1)
        res["pairwise_workaround"] = {"queries": Qp, "ms": round(ms, 2), "ms_per_query": round(ms / Qp, 3),
                                      "note": "score_edges over all N pairs plus the select, no exclusion mask"}
    if not args.partitioned or dist.get_rank() == 0:
        print(json.dumps(res))
    if args.partitioned:
        dist.destroy_process_group()


PEAK_BYTES_PER_S = 7.7e12      # HBM3e, NVIDIA HGX B200 data sheet, one GPU


def fp64_series(table_rowptr, table_col, inv_deg, method, sources):
    """fp64 [N, S] on the CPU (scipy): the truncated series of ``method`` for the sources, hop by hop from the
    cleaned reach rows R(j), with no fp32 rounding"""
    import scipy.sparse as sp
    from plnlp_b200 import paths
    rp, col = table_rowptr.cpu().numpy(), table_col.cpu().numpy()
    n = rp.size - 1
    Rm = sp.csr_matrix((np.ones(col.size), col, rp), shape=(n, n))
    wt = inv_deg.cpu().numpy()[:, None]
    E = np.zeros((n, len(sources)))
    E[np.asarray(sources), np.arange(len(sources))] = 1.0
    x = E.copy()
    for c, b, weighted in paths.hops(method):
        x = c * (Rm @ (wt * x if weighted else x)) + b * E
    return x


def path_main(args, cfg, data, split, dev):
    import torch.distributed as dist
    from plnlp_b200 import parallel, paths
    N, adj = cfg["N"], data.adj_t
    m = heuristics.Katz(args.beta, args.hops) if args.method == "Katz" else heuristics.PPR(args.alpha, args.iters)
    graph = adj
    if args.partitioned:
        if "RANK" not in os.environ:
            os.environ.update(RANK="0", WORLD_SIZE="1", LOCAL_RANK="0", MASTER_ADDR="127.0.0.1", MASTER_PORT="29541")
        dist.init_process_group("nccl", device_id=dev)
        graph = parallel.shard_graph(adj, dist.get_rank(), dist.get_world_size(), CSRGraph, symmetric=True)
    res = {"workload": cfg["name"], "gpu": gpu_info(), "method": repr(m), "N": N, "partitioned": bool(args.partitioned),
           "ranks": dist.get_world_size() if args.partitioned else 1}
    ms, shard = timed(lambda: paths.path_shard(adj).plan(), 1)
    shard = paths.path_shard(adj)
    res["table"] = {"build_ms_first": round(ms, 2), "reach_entries": int(shard.col.numel())}
    pos, neg = get_pos_neg_edges("test", split, device=dev)
    e_all = torch.cat([pos, neg.reshape(-1, 2)])
    us = torch.unique(e_all[:, 0])
    # per hop of one block of 256 sources
    B = 256
    src = us[:B].contiguous()
    x, live = shard.start(src)
    nnz = int(shard.col.numel())
    per_hop = []
    for h, (c, b, w) in enumerate(paths.hops(m)):
        shard.hop(x, live, src, c, b, w)                                   # warm-up of this hop's inputs
        ms, (y, lv) = timed(lambda: shard.hop(x, live, src, c, b, w), 1)
        live_entries = int(live[shard.col.long()].sum())
        nbytes = live_entries * B * 4 + nnz * 5 + N * B * 4 + N
        per_hop.append({"hop": h + 1, "ms": round(ms, 3), "live_row_fraction_in": round(float(live.float().mean()), 5),
                        "gathered_GB": round(nbytes / 1e9, 3), "GB_per_s": round(nbytes / ms / 1e6, 1),
                        "share_of_7.7TB_per_s": round(nbytes / ms / 1e-3 / PEAK_BYTES_PER_S, 3)})
        x, live = y, lv
    res["hops_B256"] = per_hop
    res["block_B256_ms"] = round(sum(h["ms"] for h in per_hop), 2)
    # eval split: the pairs of a subset of the distinct test sources
    S = min(args.sources, us.numel())
    keep = torch.isin(e_all[:, 0], us[:S])
    e = e_all[keep].contiguous()
    heuristics.score_edges(graph, e[:1000], m)
    times = [timed(lambda: heuristics.score_edges(graph, e, m), 1)[0] for _ in range(args.reps)]
    ms = float(np.median(times))
    res["eval_split_subset"] = {"subset": f"pairs of the first {S} of {us.numel()} distinct test sources",
                                "sources": S, "pairs": int(e.size(0)), "ms_median": round(ms, 1),
                                "pairs_per_s": round(e.size(0) / ms * 1e3),
                                "extrapolated_full_split_s": round(ms * us.numel() / S / 1e3, 1),
                                "extrapolation": "linear in distinct sources (blocks of 256); not measured"}
    out = heuristics.score_edges(graph, e, m)
    # recommend on 256 queries
    g = torch.Generator(device=dev).manual_seed(7)
    nodes = torch.randint(0, N, (256,), generator=g, device=dev)
    fn = lambda: heuristics.recommend(graph, nodes, args.k, m, "adj")      # noqa: E731
    fn()
    times = [timed(fn, 1)[0] for _ in range(args.reps)]
    profiling.enable()
    ids, sc = fn()
    spans = profiling.disable()
    res["recommend"] = {"queries": 256, "k": args.k, "exclude": "adj", "ms_median": round(float(np.median(times)), 2),
                        "ms_per_query": round(float(np.median(times)) / 256, 4), "split": split_of(spans)}
    if args.partitioned:
        si, ss = heuristics.recommend(adj, nodes, args.k, m, "adj")
        res["single_gpu_check"] = {"ids_equal": bool(torch.equal(si, ids)), "scores_equal": bool(torch.equal(ss, sc)),
                                   "scores_edges_equal": bool(torch.equal(heuristics.score_edges(adj, e, m), out))}
    # oracle sample: the fp64 series for 8 sources against the kernel's scores of their pairs
    pick = us[:S][torch.randperm(S, generator=torch.Generator().manual_seed(5))[:8].to(dev)].sort().values
    ref = fp64_series(shard.rowptr, shard.col, shard.inv_deg, m, pick.cpu().numpy())
    sel = torch.isin(e[:, 0], pick)
    pe, got = e[sel].cpu(), out[sel].cpu().double().numpy()
    want = ref[pe[:, 1].numpy(), torch.searchsorted(pick.cpu(), pe[:, 0]).numpy()]
    rel = np.abs(got - want) / np.maximum(np.abs(want), 1e-300)
    res["oracle_sample"] = {"pairs": int(pe.size(0)), "sources": 8, "within_1e-5_rel": int((rel <= 1e-5).sum()),
                            "max_rel_err": float(rel.max()) if rel.size else 0.0,
                            "nonzero": int((want > 0).sum())}
    res["gpu_after"] = gpu_info()
    if not args.partitioned or dist.get_rank() == 0:
        print(json.dumps(res))
    if args.partitioned:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("workload", nargs="?", default="citation2", choices=["citation2", "collab", "ddi"])
    ap.add_argument("--method", default="CN", choices=list(heuristics.METHODS) + list(heuristics.PATH_METHODS))
    ap.add_argument("--beta", type=float, default=0.005)
    ap.add_argument("--hops", type=int, default=3)
    ap.add_argument("--alpha", type=float, default=0.15)
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--sources", type=int, default=2048, help="path methods: distinct test sources to time")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--queries", type=int, default=0, help="time recommend / rank_against_all on this many queries")
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--pair-queries", type=int, default=4)
    ap.add_argument("--partitioned", action="store_true")
    args = ap.parse_args()
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(dev)
    cfg = dict(bench.WORKLOADS[args.workload])
    torch.manual_seed(0)
    data, split = bench.build_workload(cfg, dev, CSRGraph, gcn_normalization)
    N = cfg["N"]
    eval_split, metric = build_splits(args.workload, N, dev)
    split.update(eval_split)
    if args.method in heuristics.PATH_METHODS:
        return path_main(args, cfg, data, split, dev)
    if args.queries > 0:
        return recommend_main(args, cfg, data, split, dev)
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

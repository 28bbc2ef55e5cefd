"""Common-neighbour link heuristics on the GPU: Common Neighbours (CN), Adamic-Adar (AA) and Resource Allocation (RA),
the non-learned baselines every OGB link-prediction table prints beside a model.  An extension: the reference has
no heuristics.

Semantics (restated on the CPU in oracle/heuristics.py):
  * N(u) is the set of distinct column ids of stored row u of ``adj_t``, without u itself.  Values are ignored,
    duplicates merged and the diagonal entry dropped, so ``data.adj_t`` gives the same neighbour sets before and
    after ``gcn_normalization`` or ``set_diag``.  On a non-symmetric adjacency N(u) is row u, as stored.
    d(w) = |N(w)|.
  * CN(u, v) = |N(u) & N(v)|.
  * AA(u, v) = sum over w in N(u) & N(v) of 1 / ln d(w); a term with d(w) < 2 contributes 0.
  * RA(u, v) = sum over w in N(u) & N(v) of 1 / d(w); a term with d(w) = 0 (only possible on a non-symmetric
    adjacency) contributes 0.
  * Every sum is accumulated in fp64 and rounded to fp32 once.  Pairs (u, u) are allowed.

``score_edges`` builds a neighbour table once per adjacency object -- the cleaned CSR (int64 row pointers, sorted
distinct diagonal-free int32 columns) from the graph-construction kernels of ``graph.py``, plus the per-node fp64
weights 1 / ln d and 1 / d -- and caches it, so per-epoch evaluation builds it once.  The pairs then go through one
kernel, csrc/heuristic.cu, which intersects the two sorted neighbour lists of each pair with one warp.

On a row-partitioned graph (``adj_t`` a ``parallel.ShardedAdj``) ``score_edges`` is collective: every rank passes
the same edges and gets the full result.  The work is split by the intermediate node w, which is what the partition
owns: rank r sums over w in N(u) & N(v) & [lo, hi).  For any u the set N(u) & [lo, hi) is row u of the column block
A[:, lo:hi], the transpose of the rank's row block of A^T (``ShardedAdj.local_t``), cleaned by the same kernels into
a CSR with one row per node of the graph.  The weights of the rank's own w come from its own rows of A
(``ShardedAdj.local``), so no degree crosses the interconnect.  The same kernel produces the fp64 partials, one fp64
all-reduce sums them and the result is rounded to fp32 once.  ``Shard`` is the per-rank step, with no collective.
"""
from __future__ import annotations

import torch

from . import _ops, graph, parallel, recommend
from .utils import evaluate_hits, evaluate_mrr, get_pos_neg_edges

METHODS = ("CN", "AA", "RA")


def clean_csr(row, col, n):
    """(rowptr int64 [n + 1], col int32) of the entries (row, col) of an [n, n] matrix: every row sorted, duplicates
    merged, diagonal entries dropped -- one radix sort of the keys row * n + col (graph-construction kernels)"""
    keys, pos = graph._gb_make_keys(row, col, n, both=False, drop_diag=True)
    n_dead = int((row == col).sum())
    keys, pos = graph._gb_sort(keys, pos, n, n, has_dead=n_dead > 0)
    keys, _ = graph._gb_unique(keys[:keys.numel() - n_dead], pos, None, row.numel())
    rowptr, c = graph._gb_keys_to_csr(keys, n, n)
    return rowptr, c.to(torch.int32)


def weight_table(deg, method):
    """fp64 [n]: the term a common neighbour w adds, from its degree -- 1 / ln d (AA), 1 / d (RA); None for CN"""
    if method == "CN":
        return None
    d = deg.to(torch.float64)
    if method == "AA":
        return torch.where(deg >= 2, 1.0 / torch.log(d.clamp_min(2.0)), torch.zeros_like(d))
    return torch.where(deg >= 1, 1.0 / d.clamp_min(1.0), torch.zeros_like(d))


class NeighbourTable:
    """the cleaned CSR the kernel intersects (``rowptr`` int64 [n + 1], ``col`` int32) and the degree d(w) of every
    node whose weight it may read (``deg`` int64 [n]); the weight tables are built on first use"""

    def __init__(self, rowptr, col, deg=None):
        self.rowptr, self.col = rowptr, col
        self.n = rowptr.numel() - 1
        self.deg = rowptr[1:] - rowptr[:-1] if deg is None else deg
        self._weights = {}

    def weight(self, method):
        if method not in self._weights:
            self._weights[method] = weight_table(self.deg, method)
        return self._weights[method]


def _rows_of(rowptr, nb):
    """(local row of every entry of the first nb rows, entry count)"""
    deg = rowptr[1:nb + 1] - rowptr[:nb]
    e = int(rowptr[nb])
    return torch.repeat_interleave(torch.arange(nb, device=rowptr.device), deg, output_size=e), e


def shard_table(local, local_t, lo, hi, n, clean=None):
    """the ``NeighbourTable`` of the block [lo, hi) of intermediate nodes: row u lists N(u) & [lo, hi) (the column
    block A[:, lo:hi]: entry (i, u) of ``local_t``, the rows [lo, hi) of A^T, is entry (u, lo + i) of A), and ``deg``
    holds d(w) for w in [lo, hi) (from ``local``, the rows [lo, hi) of A) and 0 elsewhere"""
    clean = clean or clean_csr
    nb = hi - lo
    t_rowptr, t_col, _ = local_t.csr()
    i, e = _rows_of(t_rowptr, nb)
    rowptr, col = clean(t_col[:e].to(torch.int64), lo + i, n)
    l_rowptr, l_col, _ = local.csr()
    i, e = _rows_of(l_rowptr, nb)
    own_ptr, _ = clean(lo + i, l_col[:e].to(torch.int64), n)
    return NeighbourTable(rowptr, col, own_ptr[1:] - own_ptr[:-1])


_CACHE = {}


def neighbour_table(adj):
    """the cached ``NeighbourTable`` of an adjacency object (CSRGraph, torch_sparse.SparseTensor) or of this rank's
    block of a ``parallel.ShardedAdj``"""
    hit = _CACHE.get(id(adj))
    if hit is not None and hit[0] is adj:
        return hit[1]
    if isinstance(adj, parallel.ShardedAdj):
        lo, hi = parallel.row_block(adj.n_global, adj.rank, adj.world_size)
        table = shard_table(adj.local, adj.local_t, lo, hi, adj.n_global)
    else:
        if adj.size(0) != adj.size(1):
            raise ValueError(f"link heuristics need a square adjacency, got {adj.size(0)} x {adj.size(1)}")
        row, col, _ = adj.coo()
        table = NeighbourTable(*clean_csr(row.to(torch.int64), col.to(torch.int64), adj.size(0)))
    if len(_CACHE) > 16:
        _CACHE.clear()
    _CACHE[id(adj)] = (adj, table)
    return table


def _check_method(method):
    if method not in METHODS:
        raise ValueError(f"method must be one of {METHODS}, got {method!r}")


class Shard:
    """the per-rank step of the collective ``score_edges``: fp64 partial sums over the rank's block of intermediate
    nodes.  Runs no collective, so one process can play every shard; ``op`` (default ``_ops.link_heuristic_raw``)
    can be replaced by a reference."""

    def __init__(self, table, op=None):
        self.table, self.op = table, op

    def partial(self, edges, method):
        op = self.op or _ops.link_heuristic_raw
        return op(self.table.rowptr, self.table.col, self.table.weight(method), edges)


def _batches(P, batch_size):
    bs = int(batch_size) if batch_size else max(P, 1)
    if bs < 1:
        raise ValueError("batch_size must be positive")
    return range(0, P, bs), bs


def _score_sharded(sadj, edges, method, batch_size):
    import torch.distributed as dist
    dev = sadj.local.csr()[1].device
    e = torch.as_tensor(edges)
    try:
        recommend._agree(sadj.group, dev, [4, e.numel(), METHODS.index(method) if method in METHODS else -1,
                                           int(batch_size or 0)])
    except ValueError as err:
        raise ValueError("heuristics.score_edges on a row-partitioned graph is collective: every rank must pass "
                         "the same number of edges, method and batch_size") from err
    _check_method(method)
    e = recommend._edge_ids(e, sadj.n_global).to(dev)
    shard = Shard(neighbour_table(sadj))
    out = torch.empty(e.size(0), dtype=torch.float32, device=dev)
    starts, bs = _batches(e.size(0), batch_size)
    for i in starts:
        part = shard.partial(e[i:i + bs], method)
        dist.all_reduce(part, group=sadj.group)
        out[i:i + bs] = part.to(torch.float32)
    return out


def score_edges(adj_t, edges, method, batch_size=None):
    """-> fp32 [P] on the adjacency's device: the ``method`` heuristic ('CN', 'AA' or 'RA', see the module
    docstring) of every pair edges[p] = (u, v), an int64 [P, 2] tensor of node ids in [0, n).  ``batch_size``: pairs
    per kernel launch (default: all).  Raises ValueError for another method, dtype or shape, or ids out of range.
    ``adj_t`` a ``parallel.ShardedAdj``: a collective call, every rank passes the same arguments and gets the full
    result."""
    if isinstance(adj_t, parallel.ShardedAdj):
        return _score_sharded(adj_t, edges, method, batch_size)
    _check_method(method)
    e = recommend._edge_ids(edges, adj_t.size(0))
    table = neighbour_table(adj_t)
    e = e.to(table.rowptr.device)
    out = torch.empty(e.size(0), dtype=torch.float32, device=e.device)
    shard = Shard(table)
    starts, bs = _batches(e.size(0), batch_size)
    for i in starts:
        out[i:i + bs] = shard.partial(e[i:i + bs], method).to(torch.float32)
    return out


def test(data, split_edge, method, batch_size, evaluator, eval_metric):
    """``BaseModel.test`` for a heuristic: score the valid and test splits of ``split_edge`` on ``data.adj_t`` ->
    {'Hits@20'|'Hits@50'|'Hits@100'|'MRR': (valid, test)}, through the same ``get_pos_neg_edges``,
    ``evaluate_hits`` and ``evaluate_mrr`` as a model.  Collective on a row-partitioned graph."""
    adj = data.adj_t
    dev = (adj.local if isinstance(adj, parallel.ShardedAdj) else adj).csr()[1].device
    preds = []
    for split in ("valid", "test"):
        for e in get_pos_neg_edges(split, split_edge, device=dev):
            preds.append(score_edges(adj, e.reshape(-1, 2), method, batch_size))
    if eval_metric == 'hits':
        return evaluate_hits(evaluator, *preds)
    return evaluate_mrr(evaluator, *preds)

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

``recommend`` and ``rank_against_all`` rank every node (or a candidate set) for a query, with the interface, tie rule
and filtering of the model's calls in recommend.py.  A node outside the two-hop set of the query shares no neighbour
with it and scores exactly +0.0, so only that set is scored: a chunk of queries against W columns is a zeroed fp32
matrix S [Qc, W]; the mark kernel sets a bit for every j in R(w) for w in N(u) (R the transposed table, cached with
the table), and the score kernel intersects N(u) and N(j) for every set bit with the device routine of
``score_edges``.  Every entry therefore equals ``score_edges`` of its pair bit for bit, for every ``batch_size`` and
on every run.  The mask and select kernels of recommend.py then run unchanged.

On a row-partitioned graph both calls are collective and split the work by intermediate node as ``score_edges``
does: rank r computes the fp64 partial of every column over w in [lo, hi), sends column block s to rank s
(``all_to_all_single``), adds the R partials it receives in rank order 0..R-1 in fp64 and rounds once; the model's
sharded mask, select and merge follow.  CN is exact and R = 1 is bit-identical to one GPU; AA and RA lie within one
fp32 ulp of one GPU (and, at R >= 3, may differ by an ulp from the partitioned ``score_edges``, whose all-reduce
sums in another order).  ``RankShard`` is the per-rank step, with no collective.

``common_neighbour_lists`` returns the common neighbours themselves, one ascending list per pair: the count kernel
of ``score_edges`` (CN) gives the lengths, their running sum the offsets, and a fill kernel with the same
intersection routine writes the lists.  The NCN predictor (layer.py) sums the embeddings of these nodes.

The path-based scores Katz and Personalized PageRank (``Katz``, ``PPR``, ``PATH_METHODS``) go through the same four
calls and are run by paths.py, which documents their semantics.
"""
from __future__ import annotations

import math
import numbers
from dataclasses import dataclass
from typing import ClassVar

import torch

from . import _ops, graph, parallel, profiling
from . import recommend as rec
from .utils import evaluate_hits, evaluate_mrr, get_pos_neg_edges

METHODS = ("CN", "AA", "RA")
PATH_METHODS = ("Katz", "PPR")         # path-based scores, run by paths.py; the strings mean the default parameters
PATH_CODES = {"Katz": 10, "PPR": 11}   # their method words in the collective argument check
MAX_KATZ_HOPS = 32
MAX_PPR_ITERS = 1000


def _int_param(v, name, hi):
    if isinstance(v, bool) or not isinstance(v, numbers.Integral) or not 1 <= int(v) <= hi:
        raise ValueError(f"{name} must be an integer in [1, {hi}], got {v!r}")
    return int(v)


def _real_param(v, name):
    if isinstance(v, bool) or not isinstance(v, numbers.Real) or not math.isfinite(float(v)):
        raise ValueError(f"{name} must be a finite real number, got {v!r}")
    return float(v)


@dataclass(frozen=True)
class Katz:
    """Katz index truncated at ``hops`` = L: sum over l = 1 .. L of beta^l * (number of length-l walks from u to v
    along N).  beta finite and > 0, 1 <= hops <= MAX_KATZ_HOPS; anything else raises ValueError."""
    beta: float = 0.005
    hops: int = 3
    name: ClassVar[str] = "Katz"

    def __post_init__(self):
        beta = _real_param(self.beta, "Katz beta")
        if not beta > 0.0:
            raise ValueError(f"Katz beta must be > 0, got {self.beta!r}")
        object.__setattr__(self, "beta", beta)
        object.__setattr__(self, "hops", _int_param(self.hops, "Katz hops", MAX_KATZ_HOPS))


@dataclass(frozen=True)
class PPR:
    """Personalized PageRank of v for the source u after ``iters`` = T power iterations x <- (1 - alpha) P^T x +
    alpha e_u from x = e_u, P the row-stochastic walk on N (a walker at a node without neighbours is dropped).
    0 < alpha < 1, 1 <= iters <= MAX_PPR_ITERS; anything else raises ValueError."""
    alpha: float = 0.15
    iters: int = 30
    name: ClassVar[str] = "PPR"

    def __post_init__(self):
        alpha = _real_param(self.alpha, "PPR alpha")
        if not 0.0 < alpha < 1.0:
            raise ValueError(f"PPR alpha must lie in (0, 1), got {self.alpha!r}")
        object.__setattr__(self, "alpha", alpha)
        object.__setattr__(self, "iters", _int_param(self.iters, "PPR iters", MAX_PPR_ITERS))


def path_method(method):
    """the ``Katz`` / ``PPR`` parameters of a path method ('Katz', 'PPR' or an instance), or None for any other
    method"""
    if isinstance(method, (Katz, PPR)):
        return method
    if isinstance(method, str) and method in PATH_METHODS:
        return Katz() if method == "Katz" else PPR()
    return None


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
    node whose weight it may read (``deg`` int64 [n]); the weight tables and the transpose are built on first use.
    ``clean``: the cleaning function for the transpose (default ``clean_csr``)."""

    def __init__(self, rowptr, col, deg=None, clean=None):
        self.rowptr, self.col = rowptr, col
        self.n = rowptr.numel() - 1
        self.deg = rowptr[1:] - rowptr[:-1] if deg is None else deg
        self._weights = {}
        self._clean = clean
        self._reach = None

    def weight(self, method):
        if method not in self._weights:
            self._weights[method] = weight_table(self.deg, method)
        return self._weights[method]

    def reach(self):
        """(rowptr int64 [n + 1], col int32) of the transpose R(w) = {j : w in N(j)}: ``clean_csr`` of the swapped
        pairs.  Equal to the table itself on a symmetric graph; on any graph, j shares a neighbour with u exactly
        when j lies in R(w) for some w in N(u)."""
        if self._reach is None:
            i, e = _rows_of(self.rowptr, self.n)
            self._reach = (self._clean or clean_csr)(self.col[:e].to(torch.int64), i, self.n)
        return self._reach


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
    return NeighbourTable(rowptr, col, own_ptr[1:] - own_ptr[:-1], clean)


_CACHE = {}


def cached_table(adj):
    """the ``NeighbourTable`` of ``adj`` if ``neighbour_table`` has built it, else None"""
    hit = _CACHE.get(id(adj))
    return hit[1] if hit is not None and hit[0] is adj else None


def neighbour_table(adj):
    """the cached ``NeighbourTable`` of an adjacency object (CSRGraph, torch_sparse.SparseTensor) or of this rank's
    block of a ``parallel.ShardedAdj``"""
    hit = cached_table(adj)
    if hit is not None:
        return hit
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
        rec._agree(sadj.group, dev, [4, e.numel(), METHODS.index(method) if method in METHODS else -1,
                                           int(batch_size or 0)])
    except ValueError as err:
        raise ValueError("heuristics.score_edges on a row-partitioned graph is collective: every rank must pass "
                         "the same number of edges, method and batch_size") from err
    _check_method(method)
    e = rec._edge_ids(e, sadj.n_global).to(dev)
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
    result.  ``method`` may also be a path method, 'Katz', 'PPR', ``Katz(...)`` or ``PPR(...)`` (paths.py); then
    ``batch_size`` is the number of sources propagated together (see ``recommend``)."""
    pm = path_method(method)
    if pm is not None:
        from . import paths
        return paths.score_edges(adj_t, edges, pm, batch_size)
    if isinstance(adj_t, parallel.ShardedAdj):
        return _score_sharded(adj_t, edges, method, batch_size)
    _check_method(method)
    e = rec._edge_ids(edges, adj_t.size(0))
    table = neighbour_table(adj_t)
    e = e.to(table.rowptr.device)
    out = torch.empty(e.size(0), dtype=torch.float32, device=e.device)
    shard = Shard(table)
    starts, bs = _batches(e.size(0), batch_size)
    for i in starts:
        out[i:i + bs] = shard.partial(e[i:i + bs], method).to(torch.float32)
    return out


def _pair_ids(edges, n):
    """``edges`` checked for ``common_neighbour_lists``: an int64 [P, 2] tensor with ids in [-1, n)"""
    e = torch.as_tensor(edges)
    if e.dtype != torch.int64:
        raise ValueError("edges must be int64")
    if e.dim() != 2 or e.size(1) != 2:
        raise ValueError("edges must have shape [P, 2]")
    if e.numel():
        lo, hi = torch.stack([e.min(), e.max()]).tolist()          # one host read
        if lo < -1 or hi >= n:
            raise ValueError(f"edges: node ids must lie in [-1, {n})")
    return e


def common_neighbour_lists(adj_t, edges):
    """-> (rowptr int64 [P + 1], col int64 [nnz]) on the adjacency's device: the common neighbours N(u) & N(v) of
    every pair edges[p] = (u, v) at col[rowptr[p] .. rowptr[p + 1]), in ascending id order (N as in the module
    docstring; global ids in and out).  ``edges``: int64 [P, 2] with ids in [-1, n); -1 (the mean row of
    ``BaseModel.encode_for_test``) has no neighbours, and (u, u) lists N(u).  The list lengths are the CN counts of
    ``score_edges``.  Two host reads: the id range check and the list total.  Raises ValueError for another dtype or shape or an id out of range,
    NotImplementedError on a row-partitioned graph."""
    if isinstance(adj_t, parallel.ShardedAdj):
        raise NotImplementedError("common_neighbour_lists (the NCN predictor) is not implemented on a "
                                  "row-partitioned graph")
    e = _pair_ids(edges, _n_nodes(adj_t))
    table = neighbour_table(adj_t)
    e = e.to(table.rowptr.device)
    P = e.size(0)
    rowptr = torch.zeros(P + 1, dtype=torch.int64, device=e.device)
    if P:
        with profiling.span("heuristics: common-neighbour counts"):
            rowptr[1:] = torch.cumsum(_ops.link_heuristic_raw(table.rowptr, table.col, None, e).to(torch.int64), 0)
    with profiling.span("heuristics: common-neighbour lists"):
        col = _ops.common_neighbour_list_raw(table.rowptr, table.col, e, rowptr)
    return rowptr, col.to(torch.int64)


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


# ---------------------------------------------------------------------------------------------------------------------
# Recommendation and full ranking by a heuristic
# ---------------------------------------------------------------------------------------------------------------------

def query_bytes(W):
    """device bytes one query row of a one-GPU chunk costs: the fp32 score row and its bitmap"""
    return 4 * W + W // 8


def sharded_query_bytes(W, width, R):
    """the same for one rank of a row-partitioned graph: the fp64 partial row over all W columns, its bitmap, the
    padded send and receive rows [R, width] (fp64) and the fp32 block row"""
    return 8 * W + W // 8 + 16 * R * width + 4 * width


def _chunk_rows(batch_size, row_bytes):
    bs = int(batch_size) if batch_size else max(1, rec.CHUNK_BYTES // max(row_bytes, 1))
    if bs < 1:
        raise ValueError("batch_size must be positive")
    return bs


class Ranker:
    """score chunks of query nodes against W columns -- the nodes [col0, col0 + W), or the candidate set ``cand``
    (strictly ascending) -- with the table ``table``: mark the two-hop set of every query, then intersect only there.
    ``dtype`` fp32 gives the rounded scores, fp64 a shard's partial sums.  Runs no collective."""

    def __init__(self, table, method, W, col0=0, cand=None, dtype=torch.float32):
        self.table, self.method, self.W, self.col0, self.cand, self.dtype = table, method, W, col0, cand, dtype

    def chunk(self, q):
        """S [len(q), W] in ``dtype``: the heuristic of (q[a], column c's node); exactly 0 outside the two-hop set"""
        t = self.table
        rrowptr, rcol = t.reach()
        with profiling.span("heuristics: mark"):
            bitmap = _ops.two_hop_mark_raw(t.rowptr, t.col, rrowptr, rcol, q, self.W, self.col0, self.cand)
        with profiling.span("heuristics: score"):
            return _ops.two_hop_score_raw(t.rowptr, t.col, t.weight(self.method), q, bitmap, self.W, self.col0,
                                          self.cand, self.dtype)

    def target_values(self, S, q, tgt):
        """[len(q)] in S's dtype: the entry of the unmasked chunk S for (q[a], tgt[a]), or, for a target that is not
        a column (outside ``cand``), the same value from ``link_heuristic_raw`` -- the same device routine"""
        if self.cand is None:
            return S.gather(1, (tgt - self.col0).reshape(-1, 1)).reshape(-1)
        pos = torch.searchsorted(self.cand, tgt).clamp_max(max(self.W - 1, 0))
        if self.W:
            ts = S.gather(1, pos.reshape(-1, 1)).reshape(-1)
            hit = self.cand[pos] == tgt
        else:
            ts = torch.zeros(q.numel(), dtype=self.dtype, device=q.device)
            hit = torch.zeros(q.numel(), dtype=torch.bool, device=q.device)
        miss = torch.nonzero(~hit).reshape(-1)
        if miss.numel():
            t = self.table
            pairs = torch.stack([q[miss], tgt[miss]], 1)
            ts[miss] = _ops.link_heuristic_raw(t.rowptr, t.col, t.weight(self.method), pairs).to(self.dtype)
        return ts


def _mask(S, q, rowptr, col, exclude_self, col0=0, cand=None):
    with profiling.span("heuristics: mask"):
        if cand is not None:
            return _ops.score_mask_raw(S, q, rowptr, col, exclude_self, cand=cand)
        return _ops.score_mask_raw(S, q, rowptr, col, exclude_self, col0=col0)


def _select(S, k, t=None, ts=None, col0=0, cand=None):
    with profiling.span("heuristics: select"):
        if cand is not None:
            return _ops.topk_rows_raw(S, k, target=t, target_score=ts, cand=cand)
        return _ops.topk_rows_raw(S, k, target=t, target_score=ts, col0=col0)


def _n_nodes(adj_t):
    if adj_t.size(0) != adj_t.size(1):
        raise ValueError(f"link heuristics need a square adjacency, got {adj_t.size(0)} x {adj_t.size(1)}")
    return adj_t.size(0)


def _exclude_edges(exclude, n, device):
    """``exclude`` checked: None, 'adj' or an int64 [E, 2] edge tensor on the device"""
    if exclude is None or isinstance(exclude, str):
        if exclude is not None and exclude != "adj":
            raise ValueError(f"exclude: expected None, 'adj' or an int64 [E, 2] edge tensor, got {exclude!r}")
        return exclude
    e = rec._node_ids(exclude, n, "exclude").to(device)
    if e.dim() != 2 or e.size(1) != 2:
        raise ValueError("exclude edges must have shape [E, 2]")
    return e


class RankShard:
    """the per-rank step of the collective ``recommend`` / ``rank_against_all`` on a row-partitioned graph: rank
    ``rank`` of ``R`` owns the intermediate nodes and the columns [lo, hi) (blocks of ``blk``), ``table`` is its
    ``shard_table``, ``rowptr`` / ``col`` its known links (``recommend.shard_exclude_csr``).  ``cand``: the whole
    candidate set (sorted); the rank then owns its slice of it.  Runs no collective: ``partial`` gives the fp64
    partial of every column, laid out per owner for ``all_to_all_single``; ``combine`` adds what the rank receives
    in rank order; ``topk`` / ``counts`` are the model's sharded tail on the rank's block."""

    def __init__(self, table, method, n, rank, R, rowptr=None, col=None, exclude_self=True, cand=None):
        from . import parallel
        self.n, self.rank, self.R = n, rank, R
        self.blk = parallel.block_size(n, R)
        self.lo, self.hi = parallel.row_block(n, rank, R)
        self.rowptr, self.col, self.exclude_self = rowptr, col, exclude_self
        self.cand = cand
        if cand is None:
            self.mine, self.width, self.own = None, self.blk, self.hi - self.lo
            self.ranker = Ranker(table, method, R * self.blk, dtype=torch.float64)
        else:
            self.slices = rec.candidate_slices(cand, [parallel.row_block(n, r, R) for r in range(R)])
            a, b = self.slices[rank]
            self.mine, self.own = cand[a:b], b - a
            self.width = max(y - x for x, y in self.slices)
            self.ranker = Ranker(table, method, cand.numel(), cand=cand, dtype=torch.float64)

    def batch_size(self, batch_size):
        return _chunk_rows(batch_size, sharded_query_bytes(self.ranker.W, self.width, self.R))

    def partial(self, q):
        """(P fp64 [Qc, W], send fp64 [R, Qc, width]): the rank's partial sums over its intermediate nodes for every
        column, and the same laid out as one padded column block per owner"""
        P = self.ranker.chunk(q)
        Qc = q.numel()
        if self.cand is None:
            return P, P.view(Qc, self.R, self.blk).transpose(0, 1).contiguous()
        send = torch.zeros(self.R, Qc, self.width, dtype=torch.float64, device=q.device)
        for r, (a, b) in enumerate(self.slices):
            send[r, :, :b - a] = P[:, a:b]
        return P, send

    def combine(self, recv):
        """fp32 [Qc, own]: the R partials of the rank's columns (recv [R, Qc, width], from ranks 0 .. R-1) added in
        rank order in fp64 and rounded once"""
        acc = recv[0].clone()
        for r in range(1, self.R):
            acc += recv[r]
        return acc[:, :self.own].to(torch.float32).contiguous()

    @staticmethod
    def target_scores(parts):
        """fp32 [Qc] from the all-gathered target partials [R, Qc], added in rank order like ``combine``"""
        acc = parts[0].clone()
        for r in range(1, parts.size(0)):
            acc += parts[r]
        return acc.to(torch.float32)

    def topk(self, S, q, k):
        """-> (ids int64 [Qc, k] global, scores [Qc, k]): the best k of the rank's block"""
        if self.own == 0:
            return rec._no_candidates(q.numel(), k, q.device)
        _mask(S, q, self.rowptr, self.col, self.exclude_self, self.lo, self.mine)
        ids, sc, _, _ = _select(S, k, col0=self.lo, cand=self.mine)
        return ids, sc

    def counts(self, S, q, t, ts):
        """-> int32 [2, Qc]: the rank's gt / ge counts against the target scores"""
        if self.own == 0:
            return torch.zeros(2, q.numel(), dtype=torch.int32, device=q.device)
        _mask(S, q, self.rowptr, self.col, self.exclude_self, self.lo, self.mine)
        _, _, gt, ge = _select(S, 0, t, ts, col0=self.lo, cand=self.mine)
        return torch.stack([gt, ge])


def _sharded_setup(sadj, call, n_items, k, method, exclude, exclude_self, batch_size, candidates):
    """the argument check every rank runs before any other collective -> (device, candidate set or None)"""
    dev = sadj.local.csr()[1].device
    try:
        rec._agree(sadj.group, dev, [call, n_items, int(k), int(batch_size or 0), int(bool(exclude_self)),
                                           *rec._exclude_kind(exclude), rec._n_candidates(candidates),
                                           METHODS.index(method) if method in METHODS else -1])
    except ValueError as err:
        raise ValueError("heuristics.recommend / rank_against_all on a row-partitioned graph are collective: every "
                         "rank must pass the same number of queries, k, method, exclude, exclude_self, batch_size "
                         "and number of candidates") from err
    _check_method(method)
    return dev, rec.candidate_set(candidates, sadj.n_global, dev)


def _rank_shard(sadj, method, exclude, exclude_self, cand, dev):
    n = sadj.n_global
    e = _exclude_edges(exclude, n, dev)
    lo, hi = parallel.row_block(n, sadj.rank, sadj.world_size)
    rowptr, col = rec.shard_exclude_csr(e, lo, hi, n, sadj.local_t)
    return RankShard(neighbour_table(sadj), method, n, sadj.rank, sadj.world_size, rowptr, col, exclude_self, cand)


def _exchange(shard, q, group):
    """the rank's fp64 partial P and its fp32 block of summed scores"""
    import torch.distributed as dist
    P, send = shard.partial(q)
    recv = torch.empty_like(send)
    with profiling.span("heuristics: exchange (all_to_all partials)"):
        dist.all_to_all_single(recv, send, group=group)
    return P, shard.combine(recv)


@torch.no_grad()
def _recommend_sharded(sadj, nodes, k, method, exclude, exclude_self, batch_size, candidates):
    import torch.distributed as dist
    nodes = torch.as_tensor(nodes)
    dev, cand = _sharded_setup(sadj, 1, nodes.numel(), k, method, exclude, exclude_self, batch_size, candidates)
    k = rec._check_k(k)
    nodes = rec._node_ids(nodes, sadj.n_global, "nodes").reshape(-1).to(dev)
    if cand is not None and cand.numel() == 0:
        return rec._no_candidates(nodes.numel(), k, dev)
    shard = _rank_shard(sadj, method, exclude, exclude_self, cand, dev)
    bs = shard.batch_size(batch_size)
    R, Q = shard.R, nodes.numel()
    ids = torch.empty(Q, k, dtype=torch.int64, device=dev)
    scores = torch.empty(Q, k, dtype=torch.float32, device=dev)
    for i in range(0, Q, bs):
        q = nodes[i:i + bs]
        _, S = _exchange(shard, q, sadj.group)
        mine_i, mine_s = shard.topk(S, q, k)
        with profiling.span("heuristics: exchange (all_gather top-k)"):
            all_i = torch.empty(R * q.numel(), k, dtype=torch.int64, device=dev)
            all_s = torch.empty(R * q.numel(), k, dtype=torch.float32, device=dev)
            dist.all_gather_into_tensor(all_i, mine_i, group=sadj.group)
            dist.all_gather_into_tensor(all_s, mine_s, group=sadj.group)
        ids[i:i + bs], scores[i:i + bs] = _ops.topk_merge_raw(all_i.view(R, -1, k), all_s.view(R, -1, k), k)
    return ids, scores


@torch.no_grad()
def _rank_sharded(sadj, edges, method, exclude, exclude_self, batch_size, candidates):
    import torch.distributed as dist
    edges = torch.as_tensor(edges)
    dev, cand = _sharded_setup(sadj, 2, edges.numel(), 0, method, exclude, exclude_self, batch_size, candidates)
    edges = rec._edge_ids(edges, sadj.n_global).to(dev)
    if cand is not None and cand.numel() == 0:
        return torch.ones(edges.size(0), dtype=torch.float32, device=dev)
    shard = _rank_shard(sadj, method, exclude, exclude_self, cand, dev)
    bs = shard.batch_size(batch_size)
    src, tgt = edges[:, 0].contiguous(), edges[:, 1].contiguous()
    ranks = torch.empty(edges.size(0), dtype=torch.float32, device=dev)
    for i in range(0, edges.size(0), bs):
        q, t = src[i:i + bs], tgt[i:i + bs]
        P, S = _exchange(shard, q, sadj.group)
        mine = shard.ranker.target_values(P, q, t)
        with profiling.span("heuristics: exchange (all_gather target partials)"):
            parts = torch.empty(shard.R * q.numel(), dtype=torch.float64, device=dev)
            dist.all_gather_into_tensor(parts, mine, group=sadj.group)
        c = shard.counts(S, q, t, shard.target_scores(parts.view(shard.R, -1)))
        with profiling.span("heuristics: exchange (all_reduce counts)"):
            dist.all_reduce(c, group=sadj.group)
        ranks[i:i + bs] = 0.5 * (c[0].to(torch.float32) + c[1].to(torch.float32)) + 1.0
    return ranks


@torch.no_grad()
def recommend(adj_t, nodes, k, method, exclude=None, exclude_self=True, batch_size=None, candidates=None):
    """-> (ids int64 [Q, k], scores fp32 [Q, k]) on the adjacency's device: row q holds the k nodes j with the largest
    ``method`` heuristic of (nodes[q], j) ('CN', 'AA' or 'RA', the semantics of ``score_edges``, bit for bit), by
    score descending then id ascending; excluded nodes (and nodes[q] itself when ``exclude_self``) never appear.
    Every node outside the two-hop set of the query scores exactly +0.0 and is a candidate like any other, so where
    fewer than k nodes score above 0 the row is filled with score-0 nodes in ascending id order; a row runs short,
    ending in (-1, -inf), only when fewer than k nodes are left at all.  ``exclude``: None, 'adj' (the stored rows
    of ``adj_t``) or an int64 [E, 2] tensor of known links (src, dst).  ``batch_size``: queries per chunk (default:
    a chunk of about 1 GiB); results do not depend on it.  ``candidates``: an int64 tensor of node ids (a set); only
    those nodes are recommended, as if every other node were an excluded link of every query.  1 <= k <= 1024.  A
    bad method, k, dtype or shape, an id out of range, a bad exclude or candidate set raises ValueError.  ``adj_t`` a
    ``parallel.ShardedAdj``: a collective call, every rank passes the same arguments and gets the full result.

    Path methods ('Katz', 'PPR', ``Katz(...)``, ``PPR(...)``; paths.py): the query's column of the propagated state
    is its score row, a node the walks never reach scores +0.0, and the rules above are unchanged.  ``batch_size``
    is then the number of queries propagated together, rounded up to 32, 64, 128 or 256 (default:
    as many as fit ``paths.PATH_BYTES``); results do not depend on it."""
    pm = path_method(method)
    if pm is not None:
        from . import paths
        return paths.recommend(adj_t, nodes, k, pm, exclude, exclude_self, batch_size, candidates)
    if isinstance(adj_t, parallel.ShardedAdj):
        return _recommend_sharded(adj_t, nodes, k, method, exclude, exclude_self, batch_size, candidates)
    _check_method(method)
    k = rec._check_k(k)
    n = _n_nodes(adj_t)
    dev = adj_t.csr()[1].device
    nodes = rec._node_ids(nodes, n, "nodes").reshape(-1).to(dev)
    cand = rec.candidate_set(candidates, n, dev)
    e = _exclude_edges(exclude, n, dev)
    W = n if cand is None else cand.numel()
    bs = _chunk_rows(batch_size, query_bytes(W))
    if W == 0:
        return rec._no_candidates(nodes.numel(), k, dev)
    rowptr, col = rec.exclude_csr(adj_t, e, n, dev)
    ranker = Ranker(neighbour_table(adj_t), method, W, cand=cand)
    Q = nodes.numel()
    ids = torch.empty(Q, k, dtype=torch.int64, device=dev)
    scores = torch.empty(Q, k, dtype=torch.float32, device=dev)
    for i in range(0, Q, bs):
        q = nodes[i:i + bs]
        S = _mask(ranker.chunk(q), q, rowptr, col, exclude_self, cand=cand)
        ids[i:i + bs], scores[i:i + bs], _, _ = _select(S, k, cand=cand)
    return ids, scores


@torch.no_grad()
def rank_against_all(adj_t, edges, method, exclude=None, exclude_self=True, batch_size=None, candidates=None):
    """-> fp32 [P]: the filtered rank of each target edges[p, 1] among all nodes (or the ``candidates`` plus the
    target) for the source edges[p, 0] under the ``method`` heuristic, 1 + (gt + ge) / 2, where gt (ge) counts the
    candidates j != target that are not excluded and score > (>=) the target.  The target is never excluded.  A
    target outside the two-hop set of its source scores 0 and gets the mean tie rank among all score-0 candidates --
    the true filtered rank, and a common case for CN on a sparse graph.  Arguments and errors as ``recommend``;
    collective on a row-partitioned graph.  Path methods as in ``recommend``."""
    pm = path_method(method)
    if pm is not None:
        from . import paths
        return paths.rank_against_all(adj_t, edges, pm, exclude, exclude_self, batch_size, candidates)
    if isinstance(adj_t, parallel.ShardedAdj):
        return _rank_sharded(adj_t, edges, method, exclude, exclude_self, batch_size, candidates)
    _check_method(method)
    n = _n_nodes(adj_t)
    dev = adj_t.csr()[1].device
    edges = rec._edge_ids(edges, n).to(dev)
    cand = rec.candidate_set(candidates, n, dev)
    e = _exclude_edges(exclude, n, dev)
    W = n if cand is None else cand.numel()
    bs = _chunk_rows(batch_size, query_bytes(W))
    if W == 0:
        return torch.ones(edges.size(0), dtype=torch.float32, device=dev)
    rowptr, col = rec.exclude_csr(adj_t, e, n, dev)
    ranker = Ranker(neighbour_table(adj_t), method, W, cand=cand)
    src, tgt = edges[:, 0].contiguous(), edges[:, 1].contiguous()
    ranks = torch.empty(edges.size(0), dtype=torch.float32, device=dev)
    for i in range(0, edges.size(0), bs):
        q, t = src[i:i + bs], tgt[i:i + bs]
        S = ranker.chunk(q)
        ts = ranker.target_values(S, q, t)          # read before the mask: the target is never excluded
        _, _, gt, ge = _select(_mask(S, q, rowptr, col, exclude_self, cand=cand), 0, t, ts, cand=cand)
        ranks[i:i + bs] = 0.5 * (gt.to(torch.float32) + ge.to(torch.float32)) + 1.0
    return ranks

"""Path-based link scores on the GPU: Katz and Personalized PageRank (PPR), the non-learned rows link-prediction
tables print beside Common Neighbours, Adamic-Adar and Resource Allocation.  Unlike those they also score pairs with
no common neighbour.  The public surface is in heuristics.py (``heuristics.Katz``, ``heuristics.PPR``, and the
``method`` argument of ``score_edges``, ``test``, ``recommend`` and ``rank_against_all``); this module runs them.

Semantics (restated on the CPU in tests/path_oracle.py):
  * N(u), d(w) = |N(w)| and R(j) = {w : j in N(w)} are those of the common-neighbour heuristics (values, duplicates
    and the diagonal do not matter); R is ``NeighbourTable.reach()``.
  * The state has one fp32 column x per source u, and every hop is
        y[j] = fp32(c * s_j + b * [j == u]),   s_j = sum over w in R(j) of wt(w) * x[w]
    with fp64 products and sums rounded to nearest (no contraction) and one rounding to fp32.  s_j is summed over
    R(j) in ascending w, cut into items of PROP_CHUNK entries: each item in order, then the item partials in order.
  * Katz(beta, L): wt = 1, c = beta; from x = e_u, L hops with b = 1 on hops 1 .. L-1 and b = 0 on hop L -- Horner's
    form of sum over l = 1 .. L of beta^l * (number of length-l walks from u to v along N).
  * PPR(alpha, T): wt(w) = 1 / d(w) (0 when d(w) = 0), c = 1 - alpha, b = alpha; from x = e_u, T hops.
  * The score of (u, v) is x[v] of u's column.

A block of B sources (B = 32, 64, 128 or 256) is propagated together as a node-major state [N, B] by
csrc/propagate.cu, one launch per hop; the columns are independent, so every score is the same for every B.  A
uint8 live map marks the rows of the state that have a non-zero entry; the kernel skips the rest, which changes no
bit since every value is >= 0.

On a row-partitioned graph (``parallel.ShardedAdj``) the calls are collective.  Rank r owns the state rows
[lo, hi): per hop it all-gathers the state blocks and the live map (``parallel.all_gather_rows``) and runs the kernel
on its cleaned reach rows (from ``local_t``), with the arithmetic of one GPU, so every score is bit-identical to one
GPU at every R.  PPR's 1 / d vector over all N is all-gathered once per adjacency and cached.  The rank's final
rows are its shard's columns of the score chunk, so the sharded mask / select / merge tail of the common-neighbour
calls follows unchanged.  ``PathShard`` is the per-rank hop step, with no collective.
"""
from __future__ import annotations

import struct

import torch

from . import _ops, graph, parallel, profiling
from . import heuristics as H
from . import recommend as rec

PROP_CHUNK = 256               # entries of R(j) per work item: fixes the summation order on every graph
MAX_BLOCK = 256                # sources propagated together at most
WIDTHS = (32, 64, 128, 256)    # the block widths the kernel takes: each of 32 lanes owns 1, 2, 4 or 8 columns
PATH_BYTES = 8 << 30           # default budget of the per-block buffers (see ``block_width``)


def hops(method):
    """[(c, b, weighted)] of every hop of a ``heuristics.Katz`` / ``heuristics.PPR``"""
    if isinstance(method, H.Katz):
        return [(float(method.beta), 1.0 if h < method.hops else 0.0, False) for h in range(1, method.hops + 1)]
    return [(1.0 - float(method.alpha), float(method.alpha), True)] * method.iters


def agree_params(method):
    """int64 words that identify a path method and its parameters (compared across ranks with ``recommend._agree``)"""
    bits = lambda v: struct.unpack("<q", struct.pack("<d", float(v)))[0]  # noqa: E731
    if isinstance(method, H.Katz):
        return [H.PATH_CODES["Katz"], bits(method.beta), int(method.hops)]
    return [H.PATH_CODES["PPR"], bits(method.alpha), int(method.iters)]


def block_width(batch_size, col_bytes):
    """sources per block, one of the kernel's widths 32, 64, 128 and 256: ``batch_size`` rounded up to the next of
    them (capped at MAX_BLOCK), or, for None, the widest whose ``col_bytes`` per source fit PATH_BYTES (at least 32).
    Raises ValueError for batch_size < 1."""
    if batch_size:
        bs = int(batch_size)
        if bs < 1:
            raise ValueError("batch_size must be positive")
        return next((w for w in WIDTHS if w >= bs), MAX_BLOCK)
    fit = PATH_BYTES // max(col_bytes, 1)
    return max([w for w in WIDTHS if w <= fit] or [WIDTHS[0]])


def column_bytes(n, W):
    """device bytes one source costs on one GPU: two fp32 state columns over n nodes and its fp32 score row over
    W columns"""
    return 4 * (2 * n + W)


def sharded_column_bytes(n, blk, W):
    """the same for one rank of a row-partitioned graph: the gathered state column, two block columns, the score row"""
    return 4 * (n + 2 * blk + W) + n


def _hop_gpu(shard, x, live, src, c, b, weight):
    return _ops.propagate_raw(shard.plan(), weight, x, src, c, b, live, shard.lo)


class PathShard:
    """the state rows [lo, hi) of a graph of n nodes: ``rowptr`` (int64 [hi - lo + 1]) / ``col`` (int32) the cleaned
    reach rows R(j) for j in [lo, hi), ``inv_deg`` fp64 [n] the PPR weight 1 / d (or 0) of every node (needed for PPR
    only), ``blk`` the padded block height (a state block has blk rows, zero past hi - lo).  ``hop`` is one hop of
    these rows from the full state; it runs no collective, so one process can play every shard.  ``op`` (default: the
    CUDA kernel) can be replaced by a reference; ``live = False`` reads every row."""

    def __init__(self, rowptr, col, lo, hi, n, blk=None, inv_deg=None, op=None, live=True):
        self.rowptr, self.col, self.lo, self.hi, self.n = rowptr, col, lo, hi, n
        self.blk = hi - lo if blk is None else blk
        self.inv_deg, self.op, self.live = inv_deg, op, live
        self._plan = None

    def plan(self):
        if self._plan is None:
            self._plan = graph.build_plan(self.rowptr, self.col, None, self.hi - self.lo, self.n, chunk=PROP_CHUNK)
        return self._plan

    def start(self, src):
        """(x fp32 [blk, B], live uint8 [blk]): the block of x = e_src[a] in column a (src int64 [B], -1 padding)"""
        B, dev = src.numel(), src.device
        x = torch.zeros(self.blk, B, dtype=torch.float32, device=dev)
        live = torch.zeros(self.blk, dtype=torch.uint8, device=dev)
        a = torch.nonzero((src >= self.lo) & (src < self.hi)).reshape(-1)
        x[src[a] - self.lo, a] = 1.0
        live[src[a] - self.lo] = 1
        return x, live

    def hop(self, x, live, src, c, b, weighted):
        """(y fp32 [blk, B], live uint8 [blk]): one hop of the rows [lo, hi) from the full state x [>= n, B] and its
        live map"""
        if weighted and self.inv_deg is None:
            raise RuntimeError("PathShard: a weighted hop needs inv_deg")
        y, lv = (self.op or _hop_gpu)(self, x, live if self.live else None, src, c, b,
                                      self.inv_deg if weighted else None)
        rows = self.hi - self.lo
        if self.blk > rows:
            y = torch.cat([y, y.new_zeros(self.blk - rows, y.size(1))])
            lv = torch.cat([lv, lv.new_zeros(self.blk - rows)])
        return y, lv


def propagate(shard, src, method, group=None, sharded=False):
    """(x fp32 [blk, B], live): the final state block of the sources src (int64 [B], -1 padding) after every hop of
    ``method``; ``sharded``: the blocks of every rank of ``group`` are all-gathered before each hop (collective)"""
    x, live = shard.start(src)
    for c, b, weighted in hops(method):
        if sharded:
            with profiling.span("paths: all-gather state"):
                xf = parallel.all_gather_rows(x, group, name="nccl all_gather (path state)", tag="path_state")
                lf = parallel.all_gather_rows(live.view(-1, 1), group, name="nccl all_gather (path live)",
                                              tag="path_live").view(-1)
        else:
            xf, lf = x, live
        with profiling.span("paths: hop"):
            x, live = shard.hop(xf, lf, src, c, b, weighted)
    return x, live


def padded(src, B):
    """src int64 [<= B] padded to [B] with -1"""
    if src.numel() == B:
        return src.contiguous()
    return torch.cat([src, src.new_full((B - src.numel(),), -1)])


def source_blocks(u, B):
    """[(sources int64 [<= B], sel, column)]: the distinct ids of u in ascending order, cut into blocks of B; sel are
    the positions p of u with u[p] in the block, and column[i] is the block column of u[sel[i]]"""
    if u.numel() == 0:
        return []
    us, inv = torch.unique(u, return_inverse=True)
    order = torch.argsort(inv, stable=True)
    n_blk = (us.numel() + B - 1) // B
    cut = torch.searchsorted(inv[order], torch.arange(n_blk + 1, device=u.device) * B).tolist()
    out = []
    for i in range(n_blk):
        sel = order[cut[i]:cut[i + 1]]
        out.append((us[i * B:(i + 1) * B], sel, inv[sel] - i * B))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# tables: one GPU and row-partitioned
# ---------------------------------------------------------------------------------------------------------------------

def reach_rows(local, local_t, lo, hi, n, clean=None):
    """(rowptr int64 [hi - lo + 1], col int32, deg int64 [hi - lo]): the cleaned reach rows R(j) for j in [lo, hi)
    (``local_t`` holds the rows [lo, hi) of A^T: entry (i, w) says lo + i is in N(w)), and d(j) = |N(j)| of the same
    nodes (from ``local``, the rows [lo, hi) of A)"""
    clean = clean or H.clean_csr
    nb = hi - lo
    t_rowptr, t_col, _ = local_t.csr()
    i, e = H._rows_of(t_rowptr, nb)
    rp, col = clean(lo + i, t_col[:e].to(torch.int64), n)
    l_rowptr, l_col, _ = local.csr()
    i, e = H._rows_of(l_rowptr, nb)
    own, _ = clean(lo + i, l_col[:e].to(torch.int64), n)
    return rp[lo:hi + 1] - rp[lo], col, own[lo + 1:hi + 1] - own[lo:hi]


_CACHE = {}


def _cached(adj, build):
    hit = _CACHE.get(id(adj))
    if hit is not None and hit[0] is adj:
        return hit[1]
    value = build()
    if len(_CACHE) > 16:
        _CACHE.clear()
    _CACHE[id(adj)] = (adj, value)
    return value


def path_shard(adj):
    """the cached ``PathShard`` of all rows of an adjacency object (one GPU), with its PPR weights"""
    def build():
        t = H.neighbour_table(adj)
        rowptr, col = t.reach()
        return PathShard(rowptr, col, 0, t.n, t.n, inv_deg=t.weight("RA"))
    return _cached(adj, build)


def sharded_path_shard(sadj):
    """this rank's cached ``PathShard`` of a ``parallel.ShardedAdj``; building it is collective (the 1 / d vector
    over all nodes is all-gathered once)"""
    def build():
        n, R = sadj.n_global, sadj.world_size
        lo, hi = parallel.row_block(n, sadj.rank, R)
        rowptr, col, deg = reach_rows(sadj.local, sadj.local_t, lo, hi, n)
        inv = torch.zeros(sadj.blk, 1, dtype=torch.float64, device=deg.device)
        inv[:hi - lo, 0] = H.weight_table(deg, "RA")
        inv = parallel.all_gather_rows(inv, sadj.group, name="nccl all_gather (path 1/d)", tag="path_inv_deg")
        return PathShard(rowptr, col, lo, hi, n, sadj.blk, inv.reshape(-1)[:n].contiguous())
    return _cached(sadj, build)


# ---------------------------------------------------------------------------------------------------------------------
# the four calls
# ---------------------------------------------------------------------------------------------------------------------

def _agree(group, dev, head, method, what):
    try:
        rec._agree(group, dev, head)
        rec._agree(group, dev, agree_params(method))
    except ValueError as err:
        raise ValueError(f"heuristics.{what} on a row-partitioned graph is collective: every rank must pass the same "
                         "arguments, method and method parameters") from err


def score_edges(adj_t, edges, method, batch_size=None):
    """``heuristics.score_edges`` for a path method (already parsed)"""
    if isinstance(adj_t, parallel.ShardedAdj):
        return _score_sharded(adj_t, edges, method, batch_size)
    n = H._n_nodes(adj_t)
    dev = adj_t.csr()[1].device
    e = rec._edge_ids(edges, n).to(dev)
    B = block_width(batch_size, column_bytes(n, 0))
    shard = path_shard(adj_t)
    out = torch.empty(e.size(0), dtype=torch.float32, device=dev)
    for srcs, sel, col in source_blocks(e[:, 0], B):
        x, _ = propagate(shard, padded(srcs, B), method)
        out[sel] = x[e[sel, 1], col]
    return out


def _score_sharded(sadj, edges, method, batch_size):
    import torch.distributed as dist
    dev = sadj.local.csr()[1].device
    e = torch.as_tensor(edges)
    _agree(sadj.group, dev, [4, e.numel(), H.PATH_CODES[method.name], int(batch_size or 0)], method, "score_edges")
    e = rec._edge_ids(e, sadj.n_global).to(dev)
    n = sadj.n_global
    B = block_width(batch_size, sharded_column_bytes(n, sadj.blk, 0))
    shard = sharded_path_shard(sadj)
    out = torch.zeros(e.size(0), dtype=torch.float32, device=dev)
    for srcs, sel, col in source_blocks(e[:, 0], B):
        x, _ = propagate(shard, padded(srcs, B), method, sadj.group, sharded=True)
        v = e[sel, 1]
        own = (v >= shard.lo) & (v < shard.hi)
        out[sel[own]] = x[v[own] - shard.lo, col[own]]     # the owner of v writes the score
    with profiling.span("paths: all_reduce scores"):
        dist.all_reduce(out, group=sadj.group)              # + exact zeros from every other rank
    return out


def _prepare(exclude, candidates, dev, n):
    return rec.candidate_set(candidates, n, dev), H._exclude_edges(exclude, n, dev)


def _chunk(x, nq, cand, lo=0):
    """S fp32 [nq, W]: the state rows of the chunk's columns (all rows of the block, or the candidates), transposed"""
    with profiling.span("paths: transpose"):
        rows = x if cand is None else x[cand - lo]
        return rows[:, :nq].t().contiguous()


@torch.no_grad()
def recommend(adj_t, nodes, k, method, exclude=None, exclude_self=True, batch_size=None, candidates=None):
    """``heuristics.recommend`` for a path method (already parsed)"""
    if isinstance(adj_t, parallel.ShardedAdj):
        return _recommend_sharded(adj_t, nodes, k, method, exclude, exclude_self, batch_size, candidates)
    k = rec._check_k(k)
    n = H._n_nodes(adj_t)
    dev = adj_t.csr()[1].device
    nodes = rec._node_ids(nodes, n, "nodes").reshape(-1).to(dev)
    cand, e = _prepare(exclude, candidates, dev, n)
    W = n if cand is None else cand.numel()
    B = block_width(batch_size, column_bytes(n, W))
    if W == 0:
        return rec._no_candidates(nodes.numel(), k, dev)
    rowptr, col = rec.exclude_csr(adj_t, e, n, dev)
    shard = path_shard(adj_t)
    Q = nodes.numel()
    ids = torch.empty(Q, k, dtype=torch.int64, device=dev)
    scores = torch.empty(Q, k, dtype=torch.float32, device=dev)
    for i in range(0, Q, B):
        q = nodes[i:i + B]
        x, _ = propagate(shard, padded(q, B), method)
        S = H._mask(_chunk(x, q.numel(), cand), q, rowptr, col, exclude_self, cand=cand)
        ids[i:i + B], scores[i:i + B], _, _ = H._select(S, k, cand=cand)
    return ids, scores


@torch.no_grad()
def rank_against_all(adj_t, edges, method, exclude=None, exclude_self=True, batch_size=None, candidates=None):
    """``heuristics.rank_against_all`` for a path method (already parsed)"""
    if isinstance(adj_t, parallel.ShardedAdj):
        return _rank_sharded(adj_t, edges, method, exclude, exclude_self, batch_size, candidates)
    n = H._n_nodes(adj_t)
    dev = adj_t.csr()[1].device
    edges = rec._edge_ids(edges, n).to(dev)
    cand, e = _prepare(exclude, candidates, dev, n)
    W = n if cand is None else cand.numel()
    B = block_width(batch_size, column_bytes(n, W))
    if W == 0:
        return torch.ones(edges.size(0), dtype=torch.float32, device=dev)
    rowptr, col = rec.exclude_csr(adj_t, e, n, dev)
    shard = path_shard(adj_t)
    src, tgt = edges[:, 0].contiguous(), edges[:, 1].contiguous()
    ranks = torch.empty(edges.size(0), dtype=torch.float32, device=dev)
    for i in range(0, edges.size(0), B):
        q, t = src[i:i + B], tgt[i:i + B]
        x, _ = propagate(shard, padded(q, B), method)
        ts = x[t, torch.arange(q.numel(), device=dev)]      # read from the state: the target is never excluded
        S = H._mask(_chunk(x, q.numel(), cand), q, rowptr, col, exclude_self, cand=cand)
        _, _, gt, ge = H._select(S, 0, t, ts, cand=cand)
        ranks[i:i + B] = 0.5 * (gt.to(torch.float32) + ge.to(torch.float32)) + 1.0
    return ranks


def _sharded_setup(sadj, call, n_items, k, method, exclude, exclude_self, batch_size, candidates):
    dev = sadj.local.csr()[1].device
    _agree(sadj.group, dev, [call, n_items, int(k), int(batch_size or 0), int(bool(exclude_self)),
                             *rec._exclude_kind(exclude), rec._n_candidates(candidates), H.PATH_CODES[method.name]],
           method, "recommend / rank_against_all")
    n = sadj.n_global
    cand = rec.candidate_set(candidates, n, dev)
    e = H._exclude_edges(exclude, n, dev)
    lo, hi = parallel.row_block(n, sadj.rank, sadj.world_size)
    rowptr, col = rec.shard_exclude_csr(e, lo, hi, n, sadj.local_t)
    # the common-neighbour calls' per-rank tail (mask, select, counts on the rank's columns); its ranker is unused
    tail = H.RankShard(None, "CN", n, sadj.rank, sadj.world_size, rowptr, col, exclude_self, cand)
    width = sadj.blk if cand is None else tail.width
    B = block_width(batch_size, sharded_column_bytes(n, sadj.blk, width))
    return dev, cand, tail, B


def _rank_chunk(x, nq, tail):
    """S fp32 [nq, own]: the rank's columns of the chunk from its state block"""
    if tail.cand is None:
        return _chunk(x[:tail.own], nq, None)
    return _chunk(x, nq, tail.mine, tail.lo)


@torch.no_grad()
def _recommend_sharded(sadj, nodes, k, method, exclude, exclude_self, batch_size, candidates):
    import torch.distributed as dist
    nodes = torch.as_tensor(nodes)
    dev, cand, tail, B = _sharded_setup(sadj, 1, nodes.numel(), k, method, exclude, exclude_self, batch_size,
                                        candidates)
    k = rec._check_k(k)
    nodes = rec._node_ids(nodes, sadj.n_global, "nodes").reshape(-1).to(dev)
    if cand is not None and cand.numel() == 0:
        return rec._no_candidates(nodes.numel(), k, dev)
    shard = sharded_path_shard(sadj)
    R, Q = sadj.world_size, nodes.numel()
    ids = torch.empty(Q, k, dtype=torch.int64, device=dev)
    scores = torch.empty(Q, k, dtype=torch.float32, device=dev)
    for i in range(0, Q, B):
        q = nodes[i:i + B]
        x, _ = propagate(shard, padded(q, B), method, sadj.group, sharded=True)
        mine_i, mine_s = tail.topk(_rank_chunk(x, q.numel(), tail), q, k)
        with profiling.span("paths: exchange (all_gather top-k)"):
            all_i = torch.empty(R * q.numel(), k, dtype=torch.int64, device=dev)
            all_s = torch.empty(R * q.numel(), k, dtype=torch.float32, device=dev)
            dist.all_gather_into_tensor(all_i, mine_i, group=sadj.group)
            dist.all_gather_into_tensor(all_s, mine_s, group=sadj.group)
        ids[i:i + B], scores[i:i + B] = _ops.topk_merge_raw(all_i.view(R, -1, k), all_s.view(R, -1, k), k)
    return ids, scores


@torch.no_grad()
def _rank_sharded(sadj, edges, method, exclude, exclude_self, batch_size, candidates):
    import torch.distributed as dist
    edges = torch.as_tensor(edges)
    dev, cand, tail, B = _sharded_setup(sadj, 2, edges.numel(), 0, method, exclude, exclude_self, batch_size,
                                        candidates)
    edges = rec._edge_ids(edges, sadj.n_global).to(dev)
    if cand is not None and cand.numel() == 0:
        return torch.ones(edges.size(0), dtype=torch.float32, device=dev)
    shard = sharded_path_shard(sadj)
    src, tgt = edges[:, 0].contiguous(), edges[:, 1].contiguous()
    ranks = torch.empty(edges.size(0), dtype=torch.float32, device=dev)
    for i in range(0, edges.size(0), B):
        q, t = src[i:i + B], tgt[i:i + B]
        x, _ = propagate(shard, padded(q, B), method, sadj.group, sharded=True)
        own = (t >= shard.lo) & (t < shard.hi)
        at = (t - shard.lo).clamp(0, x.size(0) - 1)
        ts = torch.where(own, x[at, torch.arange(q.numel(), device=dev)], torch.zeros((), device=dev))
        with profiling.span("paths: exchange (all_reduce target scores)"):
            dist.all_reduce(ts, group=sadj.group)            # the owner's score + exact zeros
        c = tail.counts(_rank_chunk(x, q.numel(), tail), q, t, ts)
        with profiling.span("paths: exchange (all_reduce counts)"):
            dist.all_reduce(c, group=sadj.group)
        ranks[i:i + B] = 0.5 * (c[0].to(torch.float32) + c[1].to(torch.float32)) + 1.0
    return ranks

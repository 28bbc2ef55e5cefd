"""Link recommendation over all nodes: ``BaseModel.recommend`` (top-k candidates per query node) and
``BaseModel.rank_against_all`` (filtered full-ranking evaluation).  An extension: the reference only scores explicit
pairs (model.py:175-182).

Queries are processed in chunks.  A chunk is a dense score matrix S [Qc, N] -- row q holds the eval-mode predictor
score of (nodes[q], j) for every node j, the query as the source -- produced by the kernels the package already has:

  DOT                  S = h[q] . h^T                       one GEMM
  BIL                  S = bilin(h)[q] . h^T                 bilin(h) once per call, as ``score_edges`` does
  MLPDOT / MLPBIL      z = mlp(h) once per call; S = z[q] . z^T or bilin(z)[q] . z^T
  MLP (2-layer head)   the fused edge-MLP kernel over the explicit pairs (q, j) of the chunk: 2 H H1 FLOP per
                       candidate, there is no algebraic shortcut for a Hadamard-product MLP
  anything else        ``predictor.score_edges`` over explicit pairs, in pieces of a fixed size (correct, not fast)

then known links are set to -inf in place (csrc/topk.cu, plnlp_score_mask_f32) and one pass of
plnlp_topk_rows_f32 selects the top k per row, or counts the candidates that beat the target.  Every GEMM and pair
piece runs with a configuration fixed by the graph and the model alone, so results are bit-identical for every
``batch_size``.

On a row-partitioned model (``data.adj_t`` a ``parallel.ShardedAdj``) both calls are collective: every rank of the
group calls them with the same arguments and gets the full result.  The CANDIDATES are sharded by the partition the
model already has: rank r encodes its row block [lo, hi) without an all-gather, fetches the query rows it needs from
their owners (``parallel.fetch_rows``) and scores every query against its own block only (``Shard``); the select
works on global ids (col0 = lo), so the per-shard top-k lists merge exactly (plnlp_topk_merge_f32) and the per-shard
rank counts add up.  Only k candidates per query and rank, or two counts, cross the interconnect.
"""
from __future__ import annotations

import torch

from . import _ops, graph, profiling
from .layer import BilinearPredictor, DotPredictor, MLPBilPredictor, MLPDotPredictor, MLPPredictor

CHUNK_BYTES = 1 << 30          # default budget of one chunk's score matrix (plus its pair list on the fused MLP path)
PAIR_PIECE = 1 << 16           # pairs per predictor.score_edges call on the generic path (padded: fixed GEMM shapes)
MAX_K = 1024


def query_bytes(n_cand, path, n_partials=0):
    """device bytes one query row of a chunk costs: the fp32 score row, plus on the fused MLP path the int64 pair
    list, the kernel's ``n_partials`` partial scores and their sum per candidate"""
    if path == "fused_mlp":
        return n_cand * (4 + 16 + 4 * n_partials + 4)
    return n_cand * 4


def default_batch_size(n_cand, path, n_partials=0, budget=CHUNK_BYTES):
    """queries per chunk: as many as fit ``budget`` bytes, at least one"""
    return max(1, budget // max(query_bytes(n_cand, path, n_partials), 1))


def gemm_backend(n_cand, width):
    """the GEMM kernel for S = A . B^T with B [n_cand, width], chosen from the B side alone: the CUDA-core kernel where
    ``_ops.gemm_raw`` would pick it for a one-row chunk or where the tall-skinny TMA kernel could take over, the
    tensor-core default everywhere else -- never a choice that depends on the chunk's row count"""
    if width < 32 or n_cand <= 512 or n_cand * width < (1 << 20):
        return "ffma"
    return _ops.GEMM_BACKEND


class _Scorer:
    """score chunks S [Qc, hi - lo]: query nodes against the candidates [lo, hi) of a graph of ``n`` nodes, from
    ``h`` whose row i is the encoded row lo + i (rows past hi - lo may follow: the mean row, padding).  By default
    the whole graph: h [N + 1, H] with the mean row last."""

    def __init__(self, model, h, lo=0, hi=None, n=None):
        pred = model.predictor
        self.lo = lo
        self.hi = h.size(0) - 1 if hi is None else hi
        self.nb = nb = self.hi - lo
        self.n = nb if n is None else n
        self.h = h
        self.path = "pairs"
        self.n_partials = 0
        self.table = h                      # the per-node rows a query reads: what other shards fetch from this one
        if isinstance(pred, DotPredictor):
            self.path, self.dst = "gemm", h[:nb]
        elif isinstance(pred, BilinearPredictor):
            self.path, self.table, self.dst = "gemm", pred.bilin(h), h[:nb]
        elif isinstance(pred, (MLPDotPredictor, MLPBilPredictor)) and pred._node_level():
            z = pred._mlp(h)
            self.table = pred.bilin(z) if isinstance(pred, MLPBilPredictor) else z
            self.path, self.dst = "gemm", z[:nb]
        elif (isinstance(pred, MLPPredictor) and pred.lins[-1].out_features == 1
              and _ops.fused_edge_mlp_ok(h, pred.flat_params())):
            self.path, self.params = "fused_mlp", pred.flat_params()
            self.n_partials = 2 * ((self.params[0].size(0) + 255) // 256)
        self.pred = pred
        self._pair_table = None
        if self.path == "gemm":
            self.backend = gemm_backend(self.n, self.dst.size(1))

    def default_batch_size(self):
        return default_batch_size(self.nb, self.path, self.n_partials)

    def _pairs(self, q, j0, j1):
        """int64 [len(q) * (j1 - j0), 2]: (q[a], j) for j in [j0, j1), query-major"""
        cand = torch.arange(j0, j1, dtype=torch.int64, device=q.device)
        return torch.stack([q.repeat_interleave(j1 - j0), cand.repeat(q.numel())], 1)

    def _pair_rows(self, q, rows):
        """(table, query row numbers) for the pair paths: h itself, or ``[h[:nb] ; rows]`` with the query rows
        appended (kept for the call: the block is copied once)"""
        if rows is None:
            return self.h, q
        Qc = rows.size(0)
        t = self._pair_table
        if t is None or t.size(0) < self.nb + Qc:
            t = self._pair_table = torch.empty(self.nb + Qc, self.h.size(1), dtype=self.h.dtype, device=self.h.device)
            t[:self.nb] = self.h[:self.nb]
        t[self.nb:self.nb + Qc] = rows
        return t[:self.nb + Qc], torch.arange(self.nb, self.nb + Qc, dtype=torch.int64, device=q.device)

    def chunk(self, q, rows=None):
        """S [len(q), hi - lo] for the query nodes q (int64, on the device).  ``rows``: the rows of ``table`` of the
        queries, fetched from their owners (default: read from this scorer's own table)"""
        Qc, N = q.numel(), self.nb
        if self.path == "gemm":
            A = _ops.gather_rows_idx_raw(self.table, q) if rows is None else rows
            return _ops.gemm_raw(A, self.dst, transb=True, split_k=1, backend=self.backend, fixed_backend=True)
        table, qi = self._pair_rows(q, rows)
        if self.path == "fused_mlp":
            W1, b1, w2, b2 = self.params
            score, _ = _ops.edge_mlp_fwd_raw(table, self._pairs(qi, 0, N), W1, b1, w2, b2, 0.0, 0, need_a1=False)
            return score.reshape(Qc, N)
        # generic path: every score_edges call sees exactly PAIR_PIECE pairs (the tail is padded with pair (0, 0))
        S = torch.empty(Qc * N, dtype=torch.float32, device=q.device)
        flat_q = qi.repeat_interleave(N)
        cand = torch.arange(N, dtype=torch.int64, device=q.device).repeat(Qc)
        for p0 in range(0, Qc * N, PAIR_PIECE):
            p1 = min(p0 + PAIR_PIECE, Qc * N)
            pairs = torch.zeros(PAIR_PIECE, 2, dtype=torch.int64, device=q.device)
            pairs[:p1 - p0, 0] = flat_q[p0:p1]
            pairs[:p1 - p0, 1] = cand[p0:p1]
            S[p0:p1] = self.pred.score_edges(table, pairs).reshape(-1)[:p1 - p0]
        return S.reshape(Qc, N)


class Shard:
    """the per-shard step of the candidate-sharded calls: the candidates [lo, hi) of a graph of ``n`` nodes, ``h``
    their encoded rows (row i = node lo + i; padding rows may follow), ``rowptr`` / ``col`` their known links
    (``shard_exclude_csr``).  Needs no collective: the caller brings the query rows (``table`` rows of the queries,
    from every shard) and combines the shards' results.  An empty block (hi == lo) scores nothing."""

    def __init__(self, model, h, lo, hi, n, rowptr=None, col=None, exclude_self=True):
        self.lo, self.hi = lo, hi
        self.scorer = _Scorer(model, h, lo, hi, n)
        self.rowptr, self.col, self.exclude_self = rowptr, col, exclude_self

    @property
    def table(self):
        return self.scorer.table

    def _masked(self, S, q):
        return _ops.score_mask_raw(S, q, self.rowptr, self.col, self.exclude_self, col0=self.lo)

    def topk(self, q, rows, k):
        """-> (ids int64 [Qc, k] global, scores [Qc, k]): the shard's k best candidates per query"""
        if self.hi == self.lo:
            return (torch.full((q.numel(), k), -1, dtype=torch.int64, device=q.device),
                    torch.full((q.numel(), k), float("-inf"), device=q.device))
        ids, sc, _, _ = _ops.topk_rows_raw(self._masked(self.scorer.chunk(q, rows), q), k, col0=self.lo)
        return ids, sc

    def target_scores(self, q, rows, t):
        """-> (S [Qc, hi - lo] or None, fp32 [Qc]): the unmasked score chunk and the score of every target this shard
        owns (0 for the others: summed over the shards, every target gets its score)"""
        if self.hi == self.lo:
            return None, torch.zeros(q.numel(), dtype=torch.float32, device=q.device)
        S = self.scorer.chunk(q, rows)
        own = (t >= self.lo) & (t < self.hi)
        ts = S.gather(1, (t - self.lo).clamp(0, self.hi - self.lo - 1).reshape(-1, 1)).reshape(-1)
        return S, torch.where(own, ts, torch.zeros_like(ts))

    def counts(self, S, q, t, ts):
        """-> int32 [2, Qc]: the shard's gt / ge counts against the target scores ``ts`` (summed over shards)"""
        if S is None:
            return torch.zeros(2, q.numel(), dtype=torch.int32, device=q.device)
        _, _, gt, ge = _ops.topk_rows_raw(self._masked(S, q), 0, target=t, target_score=ts, col0=self.lo)
        return torch.stack([gt, ge])


def _sharded_adj(model, data):
    """the model's ``parallel.ShardedAdj`` on a row-partitioned model, else None"""
    if not model.partitioned:
        return None
    from . import parallel
    if not isinstance(data.adj_t, parallel.ShardedAdj):
        raise NotImplementedError("recommend / rank_against_all on a row-partitioned model need data.adj_t to be the "
                                  "parallel.ShardedAdj of its partition")
    return data.adj_t


def _node_ids(t, n, what):
    t = torch.as_tensor(t)
    if t.dtype != torch.int64:
        raise ValueError(f"{what} must be int64")
    if t.numel() and (int(t.min()) < 0 or int(t.max()) >= n):
        raise ValueError(f"{what}: node ids must lie in [0, {n})")
    return t


def exclude_csr(data, exclude, n, device):
    """the known links to filter, as (rowptr int64 [n + 1], col int32) on the device, or (None, None):
    ``None``; ``'adj'``: the stored rows of data.adj_t; an int64 [E, 2] edge tensor: row q lists the dst of every
    edge whose src is q (built with CSRGraph.from_edge_index)"""
    if exclude is None:
        return None, None
    if isinstance(exclude, str):
        if exclude != "adj":
            raise ValueError(f"exclude: expected None, 'adj' or an int64 [E, 2] edge tensor, got {exclude!r}")
        adj = data.adj_t
        if adj.size(0) != n:
            raise ValueError(f"exclude='adj': the adjacency has {adj.size(0)} rows, the graph {n} nodes")
        st = _ops.structure_of(adj)
        return st.rowptr, st.fwd.col
    e = _node_ids(exclude, n, "exclude").to(device)
    if e.dim() != 2 or e.size(1) != 2:
        raise ValueError("exclude edges must have shape [E, 2]")
    # from_edge_index stores edge (a, b) in row b: hand it (dst, src) so that row q holds the dst of q's edges
    g = graph.CSRGraph.from_edge_index(e.flip(1).t().contiguous(), None, n)
    rowptr, col, _ = g.csr()
    return rowptr, col.to(torch.int32)


def _csr(src, dst, n):
    """CSR (rowptr int64 [n + 1], col int32) of the pairs (src, dst): row q lists the dst of every pair with src q"""
    order = torch.argsort(src, stable=True)
    rowptr = torch.zeros(n + 1, dtype=torch.int64, device=src.device)
    if src.numel():
        rowptr[1:] = torch.cumsum(torch.bincount(src, minlength=n), 0)
    return rowptr, dst[order].to(torch.int32)


def shard_exclude_csr(exclude, lo, hi, n, local_t=None):
    """the known links among the candidates [lo, hi), as (rowptr int64 [n + 1], col int32) with rows = global query
    id and col = global candidate id in [lo, hi), or (None, None).  ``'adj'``: ``local_t`` holds the rows [lo, hi) of
    A^T (``ShardedAdj.local_t``), i.e. the columns [lo, hi) of A -- transposed here, right for non-symmetric graphs
    too; an int64 [E, 2] edge tensor: its edges whose dst lies in [lo, hi).  The union over the shards of a
    partition is the CSR ``exclude_csr`` builds."""
    if exclude is None:
        return None, None
    if isinstance(exclude, str):
        rowptr, col, _ = local_t.csr()
        nb = hi - lo
        deg = rowptr[1:nb + 1] - rowptr[:nb]
        src = col[int(rowptr[0]):int(rowptr[nb])]
        dst = lo + torch.repeat_interleave(torch.arange(nb, device=col.device), deg, output_size=src.numel())
    else:
        keep = (exclude[:, 1] >= lo) & (exclude[:, 1] < hi)
        src, dst = exclude[keep, 0], exclude[keep, 1]
    return _csr(src, dst, n)


def _encode(model, data):
    model.encoder.eval()
    model.predictor.eval()
    return model.encode_for_test(data)


def _check_k(k):
    k = int(k)
    if not 1 <= k <= MAX_K:
        raise ValueError(f"k must lie in [1, {MAX_K}]")
    return k


def _exclude_kind(exclude):
    if exclude is None:
        return 0, 0
    if isinstance(exclude, str):
        return (1 if exclude == "adj" else 3), 0
    return 2, int(torch.as_tensor(exclude).numel())


def _agree(group, device, vals):
    """every rank all-gathers the call's arguments before any other collective: a mismatch raises ValueError on
    every rank instead of leaving the others waiting in a collective"""
    import torch.distributed as dist
    mine = torch.tensor(vals, dtype=torch.int64, device=device)
    every = torch.empty(dist.get_world_size(group), mine.numel(), dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(every, mine, group=group)
    if not bool((every == mine).all()):
        raise ValueError("recommend / rank_against_all on a row-partitioned model are collective: every rank must "
                         f"pass the same arguments (per rank [call, Q, k, batch_size, exclude_self, exclude kind, E]: "
                         f"{every.tolist()})")


def _local_shard(model, data, sadj, exclude, exclude_self):
    """this rank's ``Shard``: its row block encoded without an all-gather, its known links"""
    from . import parallel
    n = sadj.n_global
    lo, hi = parallel.row_block(n, sadj.rank, sadj.world_size)
    model.encoder.eval()
    model.predictor.eval()
    with profiling.span("recommend: encode (row block)"):
        h = model.encoder(model.input_parts(data), sadj)
    if isinstance(exclude, str) or exclude is None:
        if exclude is not None and exclude != "adj":
            raise ValueError(f"exclude: expected None, 'adj' or an int64 [E, 2] edge tensor, got {exclude!r}")
        e = exclude
    else:
        e = _node_ids(exclude, n, "exclude").to(h.device)
        if e.dim() != 2 or e.size(1) != 2:
            raise ValueError("exclude edges must have shape [E, 2]")
    with profiling.span("recommend: exclusion CSR"):
        rowptr, col = shard_exclude_csr(e, lo, hi, n, sadj.local_t)
    return Shard(model, h, lo, hi, n, rowptr, col, exclude_self)


def _fetch(shard, q, group):
    """the ``table`` rows of the query nodes q from their owners"""
    from . import parallel
    uq, inv = torch.unique(q, return_inverse=True)
    return _ops.gather_rows_idx_raw(parallel.fetch_rows(shard.table, uq, group), inv)


def _sharded_batch_size(sadj, shard, batch_size):
    """queries per chunk: from the padded block size, the same on every rank"""
    s = shard.scorer
    return int(batch_size) if batch_size else default_batch_size(sadj.blk, s.path, s.n_partials)


@torch.no_grad()
def _recommend_sharded(model, data, sadj, nodes, k, exclude, exclude_self, batch_size):
    import torch.distributed as dist
    group, dev = sadj.group, model.device
    nodes = torch.as_tensor(nodes)
    _agree(group, dev, [1, nodes.numel(), int(k), int(batch_size or 0), int(bool(exclude_self)),
                        *_exclude_kind(exclude)])
    k = _check_k(k)
    nodes = _node_ids(nodes, sadj.n_global, "nodes").reshape(-1).to(dev)
    shard = _local_shard(model, data, sadj, exclude, exclude_self)
    bs = _sharded_batch_size(sadj, shard, batch_size)
    R, Q = dist.get_world_size(group), nodes.numel()
    ids = torch.empty(Q, k, dtype=torch.int64, device=dev)
    scores = torch.empty(Q, k, dtype=torch.float32, device=dev)
    for i in range(0, Q, bs):
        q = nodes[i:i + bs]
        with profiling.span("recommend: exchange (query rows)"):
            rows = _fetch(shard, q, group)
        mine_i, mine_s = shard.topk(q, rows, k)
        with profiling.span("recommend: exchange (all_gather top-k)"):
            all_i = torch.empty(R * q.numel(), k, dtype=torch.int64, device=dev)
            all_s = torch.empty(R * q.numel(), k, dtype=torch.float32, device=dev)
            dist.all_gather_into_tensor(all_i, mine_i, group=group)
            dist.all_gather_into_tensor(all_s, mine_s, group=group)
        ids[i:i + bs], scores[i:i + bs] = _ops.topk_merge_raw(all_i.view(R, -1, k), all_s.view(R, -1, k), k)
    return ids, scores


@torch.no_grad()
def _rank_sharded(model, data, sadj, edges, exclude, exclude_self, batch_size):
    import torch.distributed as dist
    group, dev = sadj.group, model.device
    edges = torch.as_tensor(edges)
    _agree(group, dev, [2, edges.numel(), 0, int(batch_size or 0), int(bool(exclude_self)), *_exclude_kind(exclude)])
    edges = _node_ids(edges, sadj.n_global, "edges").to(dev)
    if edges.dim() != 2 or edges.size(1) != 2:
        raise ValueError("edges must have shape [P, 2]")
    shard = _local_shard(model, data, sadj, exclude, exclude_self)
    bs = _sharded_batch_size(sadj, shard, batch_size)
    src, tgt = edges[:, 0].contiguous(), edges[:, 1].contiguous()
    ranks = torch.empty(edges.size(0), dtype=torch.float32, device=dev)
    for i in range(0, edges.size(0), bs):
        q, t = src[i:i + bs], tgt[i:i + bs]
        with profiling.span("recommend: exchange (query rows)"):
            rows = _fetch(shard, q, group)
        S, ts = shard.target_scores(q, rows, t)
        with profiling.span("recommend: exchange (all_reduce target scores)"):
            dist.all_reduce(ts, group=group)     # before the counts: the target score comes from its owner
        c = shard.counts(S, q, t, ts)
        with profiling.span("recommend: exchange (all_reduce counts)"):
            dist.all_reduce(c, group=group)
        ranks[i:i + bs] = 0.5 * (c[0].to(torch.float32) + c[1].to(torch.float32)) + 1.0
    return ranks


@torch.no_grad()
def recommend(model, data, nodes, k, exclude=None, exclude_self=True, batch_size=None):
    """-> (ids int64 [Q, k], scores fp32 [Q, k]) on the device: row q holds the k candidates j in [0, N) with the
    largest score of the pair (nodes[q], j), by score descending then id ascending; excluded candidates (and
    nodes[q] itself when ``exclude_self``) and NaN scores never appear; a row with fewer than k candidates ends
    in (-1, -inf).  ``batch_size``: queries per chunk (default: a chunk of about 1 GiB).  Row-partitioned model:
    a collective call, see the module docstring."""
    sadj = _sharded_adj(model, data)
    if sadj is not None:
        return _recommend_sharded(model, data, sadj, nodes, k, exclude, exclude_self, batch_size)
    k = _check_k(k)
    h = _encode(model, data)
    n, dev = h.size(0) - 1, h.device
    nodes = _node_ids(nodes, n, "nodes").reshape(-1).to(dev)
    rowptr, col = exclude_csr(data, exclude, n, dev)
    scorer = _Scorer(model, h)
    bs = int(batch_size) if batch_size else scorer.default_batch_size()
    Q = nodes.numel()
    ids = torch.empty(Q, k, dtype=torch.int64, device=dev)
    scores = torch.empty(Q, k, dtype=torch.float32, device=dev)
    for i in range(0, Q, bs):
        q = nodes[i:i + bs]
        S = scorer.chunk(q)
        _ops.score_mask_raw(S, q, rowptr, col, exclude_self)
        ids[i:i + bs], scores[i:i + bs], _, _ = _ops.topk_rows_raw(S, k)
    return ids, scores


@torch.no_grad()
def rank_against_all(model, data, edges, exclude=None, exclude_self=True, batch_size=None):
    """-> fp32 [P]: the rank of each target among all nodes for its source, 1 + (gt + ge) / 2, where gt (ge) counts
    the candidates j != target that are not excluded and score > (>=) the target (the tie rule of utils.mrr_list).
    The target itself is never excluded, even when it is a known link (the filtered setting).  Row-partitioned
    model: a collective call, see the module docstring."""
    sadj = _sharded_adj(model, data)
    if sadj is not None:
        return _rank_sharded(model, data, sadj, edges, exclude, exclude_self, batch_size)
    h = _encode(model, data)
    n, dev = h.size(0) - 1, h.device
    edges = _node_ids(edges, n, "edges").to(dev)
    if edges.dim() != 2 or edges.size(1) != 2:
        raise ValueError("edges must have shape [P, 2]")
    rowptr, col = exclude_csr(data, exclude, n, dev)
    scorer = _Scorer(model, h)
    bs = int(batch_size) if batch_size else scorer.default_batch_size()
    src, tgt = edges[:, 0].contiguous(), edges[:, 1].contiguous()
    ranks = torch.empty(edges.size(0), dtype=torch.float32, device=dev)
    for i in range(0, edges.size(0), bs):
        q, t = src[i:i + bs], tgt[i:i + bs]
        S = scorer.chunk(q)
        ts = S.gather(1, t.reshape(-1, 1)).reshape(-1)       # read before the mask: the target is never excluded
        _ops.score_mask_raw(S, q, rowptr, col, exclude_self)
        _, _, gt, ge = _ops.topk_rows_raw(S, 0, target=t, target_score=ts)
        ranks[i:i + bs] = 0.5 * (gt.to(torch.float32) + ge.to(torch.float32)) + 1.0
    return ranks

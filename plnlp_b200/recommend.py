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

``candidates`` restricts both calls to a set C of nodes (the items of a bipartite graph, an evaluation pool).  C is
sorted and made unique once per call, so column j of a chunk is the j-th smallest candidate and keys on the column
break ties exactly as keys on the global id would.  The GEMM heads score against dst[C], gathered once per call,
with the backend ``gemm_backend`` picks for the whole graph; the pair paths score the pairs (q, C[j]).  Every score
is therefore the one the all-node call computes, bit for bit.  The mask and the select find a node's column by binary
search in C (plnlp_score_mask_cand_f32, plnlp_topk_rows_cand_f32).  A target outside C is scored as one more pair
through the same path.  On a row-partitioned model rank r takes C_r = C & [lo, hi), a contiguous slice of the sorted
C, and reports global ids, so the merge is unchanged.
"""
from __future__ import annotations

import torch

from . import _ops, graph, profiling
from .layer import BilinearPredictor, DotPredictor, MLPBilPredictor, MLPDotPredictor, MLPPredictor, NCNPredictor

CHUNK_BYTES = 1 << 30          # default budget of one chunk's score matrix (plus its pair list on the fused MLP path)
PAIR_PIECE = 1 << 16           # pairs per predictor.score_edges call on the generic path (padded: fixed GEMM shapes)
DIAG_PIECE = 256               # query rows per [p, p] GEMM whose diagonal scores (query, target) pairs on the GEMM path
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
    the whole graph: h [N + 1, H] with the mean row last.  ``cand``: strictly ascending global ids in [lo, hi); the
    chunk's columns are then those nodes only, S [Qc, len(cand)]."""

    def __init__(self, model, h, lo=0, hi=None, n=None, cand=None):
        pred = model.predictor
        self.lo = lo
        self.hi = h.size(0) - 1 if hi is None else hi
        self.nb = nb = self.hi - lo
        self.n = nb if n is None else n
        self.h = h
        self.cols = None if cand is None else cand - lo         # block rows of the candidates
        self.width = nb if cand is None else cand.numel()        # columns of a chunk
        self.path = "pairs"
        self.n_partials = 0
        self.table = h                      # the per-node rows a query reads: what other shards fetch from this one
        dst = None
        if isinstance(pred, NCNPredictor):
            raise NotImplementedError("recommend / rank_against_all are not implemented for the NCN predictor (its "
                                      "score of a pair needs the pair's common neighbours)")
        if isinstance(pred, DotPredictor):
            self.path, dst = "gemm", h[:nb]
        elif isinstance(pred, BilinearPredictor):
            self.path, self.table, dst = "gemm", pred.bilin(h), h[:nb]
        elif isinstance(pred, (MLPDotPredictor, MLPBilPredictor)) and pred._node_level():
            z = pred._mlp(h)
            self.table = pred.bilin(z) if isinstance(pred, MLPBilPredictor) else z
            self.path, dst = "gemm", z[:nb]
        elif (isinstance(pred, MLPPredictor) and pred.lins[-1].out_features == 1
              and _ops.fused_edge_mlp_ok(h, pred.flat_params())):
            self.path, self.params = "fused_mlp", pred.flat_params()
            self.n_partials = 2 * ((self.params[0].size(0) + 255) // 256)
        self.pred = pred
        self._pair_table = None
        if self.path == "gemm":
            self.dst_block = dst
            self.dst = dst if self.cols is None or not self.width else _ops.gather_rows_idx_raw(dst, self.cols)
            # the graph's N, not the chunk's width: a candidate chunk runs the kernel of the all-node call
            self.backend = gemm_backend(self.n, dst.size(1))

    def default_batch_size(self):
        return default_batch_size(self.width, self.path, self.n_partials)

    def _col_rows(self, device):
        """int64 [width]: the block row of every column"""
        if self.cols is not None:
            return self.cols
        return torch.arange(self.nb, dtype=torch.int64, device=device)

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

    def _score_pairs(self, table, flat_q, flat_c):
        """fp32 [P]: the pair paths' score of the pairs (flat_q[p], flat_c[p]), rows of ``table``"""
        if self.path == "fused_mlp":
            W1, b1, w2, b2 = self.params
            score, _ = _ops.edge_mlp_fwd_raw(table, torch.stack([flat_q, flat_c], 1), W1, b1, w2, b2, 0.0, 0,
                                             need_a1=False)
            return score
        # generic path: every score_edges call sees exactly PAIR_PIECE pairs (the tail is padded with pair (0, 0))
        P = flat_q.numel()
        S = torch.empty(P, dtype=torch.float32, device=flat_q.device)
        for p0 in range(0, P, PAIR_PIECE):
            p1 = min(p0 + PAIR_PIECE, P)
            pairs = torch.zeros(PAIR_PIECE, 2, dtype=torch.int64, device=flat_q.device)
            pairs[:p1 - p0, 0] = flat_q[p0:p1]
            pairs[:p1 - p0, 1] = flat_c[p0:p1]
            S[p0:p1] = self.pred.score_edges(table, pairs).reshape(-1)[:p1 - p0]
        return S

    def chunk(self, q, rows=None):
        """S [len(q), width] for the query nodes q (int64, on the device).  ``rows``: the rows of ``table`` of the
        queries, fetched from their owners (default: read from this scorer's own table)"""
        Qc, N = q.numel(), self.width
        if self.path == "gemm":
            A = _ops.gather_rows_idx_raw(self.table, q) if rows is None else rows
            return _ops.gemm_raw(A, self.dst, transb=True, split_k=1, backend=self.backend, fixed_backend=True)
        table, qi = self._pair_rows(q, rows)
        return self._score_pairs(table, qi.repeat_interleave(N), self._col_rows(q.device).repeat(Qc)).reshape(Qc, N)

    def pair_scores(self, q, t, rows=None):
        """fp32 [len(q)]: the score of (q[a], block row t[a]) through the chunk's own path and kernel, so it equals
        that pair's chunk entry bit for bit.  The GEMM path takes the diagonal of [p, p] products."""
        if self.path != "gemm":
            table, qi = self._pair_rows(q, rows)
            return self._score_pairs(table, qi, t)
        A = _ops.gather_rows_idx_raw(self.table, q) if rows is None else rows
        B = _ops.gather_rows_idx_raw(self.dst_block, t)
        out = torch.empty(q.numel(), dtype=torch.float32, device=q.device)
        for p0 in range(0, q.numel(), DIAG_PIECE):
            p1 = min(p0 + DIAG_PIECE, q.numel())
            out[p0:p1] = _ops.gemm_raw(A[p0:p1], B[p0:p1], transb=True, split_k=1, backend=self.backend,
                                       fixed_backend=True).diagonal()
        return out

    def target_scores(self, S, q, t, rows=None):
        """fp32 [len(q)]: the score of (q[a], t[a]) for every global target t[a] in [lo, hi) (garbage for the others):
        read from the unmasked chunk S when t[a] is one of its columns, else scored as a pair"""
        if self.cols is None:
            return S.gather(1, (t - self.lo).clamp(0, self.nb - 1).reshape(-1, 1)).reshape(-1)
        tl = t - self.lo
        own = (tl >= 0) & (tl < self.nb)
        pos = torch.searchsorted(self.cols, tl).clamp_max(max(self.width - 1, 0))
        if self.width:
            ts = S.gather(1, pos.reshape(-1, 1)).reshape(-1)
            hit = self.cols[pos] == tl
        else:
            ts = torch.zeros(q.numel(), dtype=torch.float32, device=q.device)
            hit = torch.zeros_like(own)
        miss = torch.nonzero(own & ~hit).reshape(-1)
        if miss.numel():
            ts[miss] = self.pair_scores(q[miss], tl[miss], None if rows is None else rows[miss])
        return ts


def _no_candidates(Q, k, device):
    return (torch.full((Q, k), -1, dtype=torch.int64, device=device),
            torch.full((Q, k), float("-inf"), device=device))


class Shard:
    """the per-shard step of the candidate-sharded calls: the candidates [lo, hi) of a graph of ``n`` nodes, ``h``
    their encoded rows (row i = node lo + i; padding rows may follow), ``rowptr`` / ``col`` their known links
    (``shard_exclude_csr``).  ``cand``: the shard's slice of a candidate set (strictly ascending global ids in
    [lo, hi)); the shard then scores those nodes only.  Needs no collective: the caller brings the query rows
    (``table`` rows of the queries, from every shard) and combines the shards' results.  An empty block (hi == lo)
    scores nothing; a block with an empty candidate slice scores only the targets it owns."""

    def __init__(self, model, h, lo, hi, n, rowptr=None, col=None, exclude_self=True, cand=None):
        self.lo, self.hi, self.cand = lo, hi, cand
        self.scorer = _Scorer(model, h, lo, hi, n, cand)
        self.rowptr, self.col, self.exclude_self = rowptr, col, exclude_self

    @property
    def table(self):
        return self.scorer.table

    def _masked(self, S, q):
        if self.cand is not None:
            return _ops.score_mask_raw(S, q, self.rowptr, self.col, self.exclude_self, cand=self.cand)
        return _ops.score_mask_raw(S, q, self.rowptr, self.col, self.exclude_self, col0=self.lo)

    def _select(self, S, q, k, t=None, ts=None):
        if self.cand is not None:
            return _ops.topk_rows_raw(self._masked(S, q), k, target=t, target_score=ts, cand=self.cand)
        return _ops.topk_rows_raw(self._masked(S, q), k, target=t, target_score=ts, col0=self.lo)

    def topk(self, q, rows, k):
        """-> (ids int64 [Qc, k] global, scores [Qc, k]): the shard's k best candidates per query"""
        if self.scorer.width == 0:
            return _no_candidates(q.numel(), k, q.device)
        ids, sc, _, _ = self._select(self.scorer.chunk(q, rows), q, k)
        return ids, sc

    def target_scores(self, q, rows, t):
        """-> (S [Qc, width] or None, fp32 [Qc]): the unmasked score chunk and the score of every target this shard
        owns (0 for the others: summed over the shards, every target gets its score)"""
        if self.hi == self.lo:
            return None, torch.zeros(q.numel(), dtype=torch.float32, device=q.device)
        S = self.scorer.chunk(q, rows) if self.scorer.width else None
        own = (t >= self.lo) & (t < self.hi)
        ts = self.scorer.target_scores(S, q, t, rows)
        return S, torch.where(own, ts, torch.zeros_like(ts))

    def counts(self, S, q, t, ts):
        """-> int32 [2, Qc]: the shard's gt / ge counts against the target scores ``ts`` (summed over shards)"""
        if S is None:
            return torch.zeros(2, q.numel(), dtype=torch.int32, device=q.device)
        _, _, gt, ge = self._select(S, q, 0, t, ts)
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


def _edge_ids(edges, n):
    e = _node_ids(edges, n, "edges")
    if e.dim() != 2 or e.size(1) != 2:
        raise ValueError("edges must have shape [P, 2]")
    return e


def candidate_set(candidates, n, device):
    """``candidates`` as a strictly ascending int64 tensor on the device (``torch.unique``: order and duplicates do
    not matter), or None.  Raises ValueError for another dtype, a rank other than 1 or ids outside [0, n)."""
    if candidates is None:
        return None
    c = _node_ids(candidates, n, "candidates")
    if c.dim() != 1:
        raise ValueError("candidates must be a 1-D tensor of node ids")
    return torch.unique(c.to(device))


def candidate_slices(cand, bounds):
    """[(a, b)] per block [lo, hi) of ``bounds``: cand[a:b] are the candidates in that block (cand sorted).  The
    slices of a partition cover cand exactly once."""
    edges = torch.tensor([x for lo, hi in bounds for x in (lo, hi)], dtype=torch.int64, device=cand.device)
    at = torch.searchsorted(cand, edges).tolist()
    return [(at[2 * r], at[2 * r + 1]) for r in range(len(bounds))]


def exclude_csr(adj, exclude, n, device):
    """the known links to filter, as (rowptr int64 [n + 1], col int32) on the device, or (None, None):
    ``None``; ``'adj'``: the stored rows of the adjacency ``adj``; an int64 [E, 2] edge tensor: row q lists the dst
    of every edge whose src is q (built with CSRGraph.from_edge_index)"""
    if exclude is None:
        return None, None
    if isinstance(exclude, str):
        if exclude != "adj":
            raise ValueError(f"exclude: expected None, 'adj' or an int64 [E, 2] edge tensor, got {exclude!r}")
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
                         f"pass the same arguments (per rank [call, Q, k, batch_size, exclude_self, exclude kind, E, "
                         f"|candidates| or -1]: "
                         f"{every.tolist()})")


def _local_shard(model, data, sadj, exclude, exclude_self, cand=None):
    """this rank's ``Shard``: its row block encoded without an all-gather, its known links, its slice ``cand`` of
    the candidate set"""
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
    return Shard(model, h, lo, hi, n, rowptr, col, exclude_self, cand)


def _fetch(shard, q, group):
    """the ``table`` rows of the query nodes q from their owners"""
    from . import parallel
    uq, inv = torch.unique(q, return_inverse=True)
    return _ops.gather_rows_idx_raw(parallel.fetch_rows(shard.table, uq, group), inv)


def _rank_candidates(sadj, cand):
    """(this rank's slice of the candidate set or None, the width every rank's chunk budget is sized for): the
    padded block, or the largest slice of any rank -- computed alike on every rank, with no collective"""
    if cand is None:
        return None, sadj.blk
    from . import parallel
    R = sadj.world_size
    sl = candidate_slices(cand, [parallel.row_block(sadj.n_global, r, R) for r in range(R)])
    a, b = sl[sadj.rank]
    return cand[a:b], max(y - x for x, y in sl)


def _sharded_batch_size(width, shard, batch_size):
    """queries per chunk: from ``width`` (``_rank_candidates``), the same on every rank"""
    s = shard.scorer
    return int(batch_size) if batch_size else default_batch_size(width, s.path, s.n_partials)


def _n_candidates(candidates):
    return -1 if candidates is None else int(torch.as_tensor(candidates).numel())


@torch.no_grad()
def _recommend_sharded(model, data, sadj, nodes, k, exclude, exclude_self, batch_size, candidates):
    import torch.distributed as dist
    group, dev = sadj.group, model.device
    nodes = torch.as_tensor(nodes)
    _agree(group, dev, [1, nodes.numel(), int(k), int(batch_size or 0), int(bool(exclude_self)),
                        *_exclude_kind(exclude), _n_candidates(candidates)])
    k = _check_k(k)
    nodes = _node_ids(nodes, sadj.n_global, "nodes").reshape(-1).to(dev)
    cand = candidate_set(candidates, sadj.n_global, dev)
    if cand is not None and cand.numel() == 0:
        return _no_candidates(nodes.numel(), k, dev)
    mine, width = _rank_candidates(sadj, cand)
    shard = _local_shard(model, data, sadj, exclude, exclude_self, mine)
    bs = _sharded_batch_size(width, shard, batch_size)
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
def _rank_sharded(model, data, sadj, edges, exclude, exclude_self, batch_size, candidates):
    import torch.distributed as dist
    group, dev = sadj.group, model.device
    edges = torch.as_tensor(edges)
    _agree(group, dev, [2, edges.numel(), 0, int(batch_size or 0), int(bool(exclude_self)), *_exclude_kind(exclude),
                        _n_candidates(candidates)])
    edges = _edge_ids(edges, sadj.n_global).to(dev)
    cand = candidate_set(candidates, sadj.n_global, dev)
    if cand is not None and cand.numel() == 0:
        return torch.ones(edges.size(0), dtype=torch.float32, device=dev)
    mine, width = _rank_candidates(sadj, cand)
    shard = _local_shard(model, data, sadj, exclude, exclude_self, mine)
    bs = _sharded_batch_size(width, shard, batch_size)
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
def recommend(model, data, nodes, k, exclude=None, exclude_self=True, batch_size=None, candidates=None):
    """-> (ids int64 [Q, k], scores fp32 [Q, k]) on the device: row q holds the k candidates j in [0, N) with the
    largest score of the pair (nodes[q], j), by score descending then id ascending; excluded candidates (and
    nodes[q] itself when ``exclude_self``) and NaN scores never appear; a row with fewer than k candidates ends
    in (-1, -inf).  ``batch_size``: queries per chunk (default: a chunk of about 1 GiB).  ``candidates``: an int64
    tensor of node ids (a set: order and duplicates do not matter); only those nodes are candidates, exactly as if
    every other node were an excluded link of every query.  Row-partitioned model: a collective call, see the module
    docstring."""
    sadj = _sharded_adj(model, data)
    if sadj is not None:
        return _recommend_sharded(model, data, sadj, nodes, k, exclude, exclude_self, batch_size, candidates)
    k = _check_k(k)
    cand = None
    if candidates is not None:
        n = data.adj_t.size(0)
        cand = candidate_set(candidates, n, model.device)
        if cand.numel() == 0:                       # nothing to score: no encode, no kernel
            return _no_candidates(_node_ids(nodes, n, "nodes").numel(), k, model.device)
    h = _encode(model, data)
    n, dev = h.size(0) - 1, h.device
    nodes = _node_ids(nodes, n, "nodes").reshape(-1).to(dev)
    rowptr, col = exclude_csr(data.adj_t, exclude, n, dev)
    scorer = _Scorer(model, h, cand=cand)
    bs = int(batch_size) if batch_size else scorer.default_batch_size()
    Q = nodes.numel()
    ids = torch.empty(Q, k, dtype=torch.int64, device=dev)
    scores = torch.empty(Q, k, dtype=torch.float32, device=dev)
    for i in range(0, Q, bs):
        q = nodes[i:i + bs]
        S = scorer.chunk(q)
        _ops.score_mask_raw(S, q, rowptr, col, exclude_self, cand=cand)
        ids[i:i + bs], scores[i:i + bs], _, _ = _ops.topk_rows_raw(S, k, cand=cand)
    return ids, scores


@torch.no_grad()
def rank_against_all(model, data, edges, exclude=None, exclude_self=True, batch_size=None, candidates=None):
    """-> fp32 [P]: the rank of each target among all nodes for its source, 1 + (gt + ge) / 2, where gt (ge) counts
    the candidates j != target that are not excluded and score > (>=) the target (the tie rule of utils.mrr_list).
    The target itself is never excluded, even when it is a known link (the filtered setting).  ``candidates``: rank
    each target among that set of nodes plus the target itself (the target is never excluded, in the set or not).
    Row-partitioned model: a collective call, see the module docstring."""
    sadj = _sharded_adj(model, data)
    if sadj is not None:
        return _rank_sharded(model, data, sadj, edges, exclude, exclude_self, batch_size, candidates)
    cand = None
    if candidates is not None:
        n = data.adj_t.size(0)
        cand = candidate_set(candidates, n, model.device)
        if cand.numel() == 0:                       # nothing beats a target: rank 1, no encode, no kernel
            return torch.ones(_edge_ids(edges, n).size(0), dtype=torch.float32, device=model.device)
    h = _encode(model, data)
    n, dev = h.size(0) - 1, h.device
    edges = _edge_ids(edges, n).to(dev)
    rowptr, col = exclude_csr(data.adj_t, exclude, n, dev)
    scorer = _Scorer(model, h, cand=cand)
    bs = int(batch_size) if batch_size else scorer.default_batch_size()
    src, tgt = edges[:, 0].contiguous(), edges[:, 1].contiguous()
    ranks = torch.empty(edges.size(0), dtype=torch.float32, device=dev)
    for i in range(0, edges.size(0), bs):
        q, t = src[i:i + bs], tgt[i:i + bs]
        S = scorer.chunk(q)
        # read before the mask: the target is never excluded
        ts = S.gather(1, t.reshape(-1, 1)).reshape(-1) if cand is None else scorer.target_scores(S, q, t)
        _ops.score_mask_raw(S, q, rowptr, col, exclude_self, cand=cand)
        _, _, gt, ge = _ops.topk_rows_raw(S, 0, target=t, target_score=ts, cand=cand)
        ranks[i:i + bs] = 0.5 * (gt.to(torch.float32) + ge.to(torch.float32)) + 1.0
    return ranks


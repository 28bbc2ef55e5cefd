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
"""
from __future__ import annotations

import torch

from . import _ops, graph
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
    """score chunks S [Qc, N] for one encoded graph ``h`` ([N + 1, H], the mean row last)"""

    def __init__(self, model, h):
        pred = model.predictor
        self.n = h.size(0) - 1
        self.h = h
        self.path = "pairs"
        self.n_partials = 0
        if isinstance(pred, DotPredictor):
            self.path, self.src, self.dst = "gemm", h, h[:self.n]
        elif isinstance(pred, BilinearPredictor):
            self.path, self.src, self.dst = "gemm", pred.bilin(h), h[:self.n]
        elif isinstance(pred, (MLPDotPredictor, MLPBilPredictor)) and pred._node_level():
            z = pred._mlp(h)
            src = pred.bilin(z) if isinstance(pred, MLPBilPredictor) else z
            self.path, self.src, self.dst = "gemm", src, z[:self.n]
        elif (isinstance(pred, MLPPredictor) and pred.lins[-1].out_features == 1
              and _ops.fused_edge_mlp_ok(h, pred.flat_params())):
            self.path, self.params = "fused_mlp", pred.flat_params()
            self.n_partials = 2 * ((self.params[0].size(0) + 255) // 256)
        self.pred = pred
        if self.path == "gemm":
            self.backend = gemm_backend(self.n, self.dst.size(1))

    def default_batch_size(self):
        return default_batch_size(self.n, self.path, self.n_partials)

    def _pairs(self, q, j0, j1):
        """int64 [len(q) * (j1 - j0), 2]: (q[a], j) for j in [j0, j1), query-major"""
        cand = torch.arange(j0, j1, dtype=torch.int64, device=q.device)
        return torch.stack([q.repeat_interleave(j1 - j0), cand.repeat(q.numel())], 1)

    def chunk(self, q):
        """S [len(q), N] for the query nodes q (int64, on the device)"""
        Qc, N = q.numel(), self.n
        if self.path == "gemm":
            A = _ops.gather_rows_idx_raw(self.src, q)
            return _ops.gemm_raw(A, self.dst, transb=True, split_k=1, backend=self.backend)
        if self.path == "fused_mlp":
            W1, b1, w2, b2 = self.params
            score, _ = _ops.edge_mlp_fwd_raw(self.h, self._pairs(q, 0, N), W1, b1, w2, b2, 0.0, 0, need_a1=False)
            return score.reshape(Qc, N)
        # generic path: every score_edges call sees exactly PAIR_PIECE pairs (the tail is padded with pair (0, 0))
        S = torch.empty(Qc * N, dtype=torch.float32, device=q.device)
        flat_q = q.repeat_interleave(N)
        cand = torch.arange(N, dtype=torch.int64, device=q.device).repeat(Qc)
        for p0 in range(0, Qc * N, PAIR_PIECE):
            p1 = min(p0 + PAIR_PIECE, Qc * N)
            pairs = torch.zeros(PAIR_PIECE, 2, dtype=torch.int64, device=q.device)
            pairs[:p1 - p0, 0] = flat_q[p0:p1]
            pairs[:p1 - p0, 1] = cand[p0:p1]
            S[p0:p1] = self.pred.score_edges(self.h, pairs).reshape(-1)[:p1 - p0]
        return S.reshape(Qc, N)


def _check_model(model):
    if model.partitioned:
        raise NotImplementedError("recommend / rank_against_all on a row-partitioned model: shard the queries instead")


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


def _encode(model, data):
    _check_model(model)
    model.encoder.eval()
    model.predictor.eval()
    return model.encode_for_test(data)


@torch.no_grad()
def recommend(model, data, nodes, k, exclude=None, exclude_self=True, batch_size=None):
    """-> (ids int64 [Q, k], scores fp32 [Q, k]) on the device: row q holds the k candidates j in [0, N) with the
    largest score of the pair (nodes[q], j), by score descending then id ascending; excluded candidates (and
    nodes[q] itself when ``exclude_self``) and NaN scores never appear; a row with fewer than k candidates ends
    in (-1, -inf).  ``batch_size``: queries per chunk (default: a chunk of about 1 GiB)."""
    k = int(k)
    if not 1 <= k <= MAX_K:
        raise ValueError(f"k must lie in [1, {MAX_K}]")
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
    The target itself is never excluded, even when it is a known link (the filtered setting)."""
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

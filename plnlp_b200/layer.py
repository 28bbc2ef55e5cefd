"""Encoders and link predictors with the reference's module surface
(/root/reference/plnlp/layer.py), running on the plnlp_b200 kernels.

Differences a user can see: none for the in-scope classes (same constructor arguments, same
``.convs`` / ``.lins`` containers, same parameter names, same ``forward`` signatures and output
shapes).  Internally relu + dropout are fused into the producing kernel's epilogue and the conv
modules additionally accept a tuple of input blocks so ``[emb | x]`` is never concatenated.
"""
from __future__ import annotations

import math
import os

import torch

from . import _ops


# GCNConv: aggregate before the linear map when that side is narrower (see GCNConv.forward)
REASSOCIATE = os.environ.get("PLNLP_GCN_REASSOCIATE", "1") != "0"
# relu backward of the layer before a row-restricted last conv fused into that conv's backward SpMM (BaseGNN.forward)
FUSE_RELU_BWD = os.environ.get("PLNLP_FUSE_RELU_BWD", "1") != "0"


def mark_constant(x):
    """declare that ``x`` (node features) does not change between steps: the convs may keep its aggregate."""
    x._plnlp_const = True
    return x


def _is_const(x):
    return getattr(x, "_plnlp_const", False) and not x.requires_grad


def _const_aggregate(adj_t, x, reduce):
    """A @ x for a block marked constant (``mark_constant``: data.x), cached on the adjacency object; the key
    carries the tensor's storage, shape and version counter so an in-place update or another tensor
    invalidates it."""
    cache = adj_t.__dict__.setdefault("_plnlp_const_agg", {})
    key = (reduce, x.data_ptr(), tuple(x.shape), x.stride(0), x._version)
    hit = cache.get(key)
    if hit is None:
        cache.clear()                       # one constant block per adjacency: never hold stale copies
        with torch.no_grad():
            hit = cache[key] = _ops.spmm(adj_t, x, reduce=reduce)
    return hit


def _agg_buffer_ok(adj_t, parts):
    """sparse adjacency (single device or row-partitioned), fp32 blocks: the aggregates can live side by side
    in one buffer"""
    from . import parallel
    local = adj_t.local if isinstance(adj_t, parallel.ShardedAdj) else adj_t
    if _ops.structure_of(local).dense_ok:
        return False
    return all(p.dim() == 2 and p.dtype == torch.float32 for p in parts)


def _agg_buffer(adj_t, parts):
    """-> (buf [N, sum widths], holder, offsets of the live blocks, live blocks).  ``buf`` persists on the
    adjacency object; the column blocks of constant parts are filled here, once per (tensor, version)."""
    key = tuple((p.size(1),) + ((p.data_ptr(), p.stride(0), p._version) if _is_const(p) else ())
                for p in parts)
    holder = adj_t.__dict__.setdefault("_plnlp_agg_buffer", {})
    if holder.get("key") != key:
        holder.clear()
        # rows on a 16-byte pitch (the TMA-fed GEMM, csrc/gemm_tma.cu, reads this matrix as its A operand) with one
        # spare column that holds 1.0: the weight-gradient GEMM  dY^T [A x | 1]  then delivers the bias gradient
        # (the column sums of dY) in its last column for free -- no separate pass over dY (_ops.AggLinear.backward)
        width = sum(p.size(1) for p in parts)
        full = torch.empty(adj_t.size(0), (width + 1 + 3) // 4 * 4, dtype=torch.float32, device=parts[0].device)
        full[:, width:] = 0.0
        full[:, width] = 1.0
        buf = full[:, :width]
        off = 0
        with torch.no_grad():
            for p in parts:
                if _is_const(p):
                    _ops.aggregate_into(adj_t, p, buf[:, off:off + p.size(1)])
                off += p.size(1)
        holder.update(key=key, buf=buf, ext=full[:, :width + 1], stamp=0)
    offs, xs, off = [], [], 0
    for p in parts:
        if not _is_const(p):
            offs.append(off)
            xs.append(p)
        off += p.size(1)
    return holder["buf"], holder, offs, xs


def _as_parts(x):
    return list(x) if isinstance(x, (tuple, list)) else [x]


def _split_cols(weight, parts):
    """column blocks of ``weight`` matching the widths of ``parts`` (views, no copy)."""
    if len(parts) == 1:
        return [weight]
    out, c = [], 0
    for p in parts:
        out.append(weight[:, c:c + p.size(1)])
        c += p.size(1)
    if c != weight.size(1):
        raise RuntimeError(f"input blocks have {c} columns, the layer expects {weight.size(1)}")
    return out


def _kaiming_linear_(weight, bias):
    """torch.nn.Linear's default init (what PyG 2.0.1's SAGEConv lins use)."""
    torch.nn.init.kaiming_uniform_(weight, a=math.sqrt(5))
    if bias is not None:
        bound = 1.0 / math.sqrt(weight.size(1)) if weight.size(1) > 0 else 0.0
        torch.nn.init.uniform_(bias, -bound, bound)


class _Lin(torch.nn.Module):
    """parameter holder named like torch.nn.Linear (``weight`` [out, in], optional ``bias``)."""

    def __init__(self, in_channels, out_channels, bias=True):
        super().__init__()
        self.in_features, self.out_features = in_channels, out_channels
        self.weight = torch.nn.Parameter(torch.empty(out_channels, in_channels))
        self.bias = torch.nn.Parameter(torch.empty(out_channels)) if bias else None
        self.reset_parameters()

    def reset_parameters(self):
        _kaiming_linear_(self.weight, self.bias)

    def forward(self, x, act=_ops.ACT_NONE, drop_p=0.0):
        lead = x.shape[:-1]
        y = _ops.fused_linear([x.reshape(-1, x.size(-1))], [self.weight], self.bias, act, drop_p,
                              _ops.new_seed() if drop_p > 0 else 0)
        return y.reshape(*lead, self.out_features)


class SAGEConv(torch.nn.Module):
    """mean-aggregating GraphSAGE conv: lin_l(mean_{j in N(i)} x_j) + lin_r(x_i), adjacency values
    ignored (what ``SAGEConv(in, out)`` of PyG 2.0.1 computes at layer.py:36).  Parameters:
    lin_l.weight, lin_l.bias, lin_r.weight."""

    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.lin_l = _Lin(in_channels, out_channels, bias=True)
        self.lin_r = _Lin(in_channels, out_channels, bias=False)

    def reset_parameters(self):
        self.lin_l.reset_parameters()
        self.lin_r.reset_parameters()

    def forward(self, x, adj_t, act=_ops.ACT_NONE, drop_p=0.0, sparse_grad=False):
        parts = _as_parts(x)
        aggs = [_const_aggregate(adj_t, p, "mean") if _is_const(p)
                else _ops.spmm(adj_t, p, reduce="mean", sparse_grad=sparse_grad) for p in parts]
        wl, wr = _split_cols(self.lin_l.weight, parts), _split_cols(self.lin_r.weight, parts)
        return _ops.fused_linear(aggs + parts, wl + wr, self.lin_l.bias, act, drop_p,
                                 _ops.new_seed() if drop_p > 0 else 0)


class GraphConv(torch.nn.Module):
    """PyG 2.0.1 ``GraphConv(in, out)`` (aggr='add'), the conv of the reference's WSAGE (layer.py:48-54):
    lin_rel(sum_{j in N(i)} w_ij x_j) + lin_root(x_i) -- SAGEConv's shape with a WEIGHTED SUM in place of the
    mean: the stored adjacency values are the edge weights (a value-less adjacency counts every edge once).
    Parameters: lin_rel.weight, lin_rel.bias, lin_root.weight."""

    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.lin_rel = _Lin(in_channels, out_channels, bias=True)
        self.lin_root = _Lin(in_channels, out_channels, bias=False)

    def reset_parameters(self):
        self.lin_rel.reset_parameters()
        self.lin_root.reset_parameters()

    def forward(self, x, adj_t, act=_ops.ACT_NONE, drop_p=0.0, sparse_grad=False):
        parts = _as_parts(x)
        aggs = [_const_aggregate(adj_t, p, "sum") if _is_const(p)
                else _ops.spmm(adj_t, p, reduce="sum", sparse_grad=sparse_grad) for p in parts]
        wl, wr = _split_cols(self.lin_rel.weight, parts), _split_cols(self.lin_root.weight, parts)
        return _ops.fused_linear(aggs + parts, wl + wr, self.lin_rel.bias, act, drop_p,
                                 _ops.new_seed() if drop_p > 0 else 0)


class GCNConv(torch.nn.Module):
    """``GCNConv(in, out, normalize=False)`` (layer.py:45): A_hat @ (x W^T) + bias with the
    pre-normalised adjacency.  Parameters: lin.weight (glorot), bias (zeros)."""

    def __init__(self, in_channels, out_channels, normalize=False):
        super().__init__()
        if normalize:
            raise NotImplementedError("the reference pre-normalises the adjacency (main.py:177-179)")
        self.in_channels, self.out_channels = in_channels, out_channels
        self.lin = _Lin(in_channels, out_channels, bias=False)
        self.bias = torch.nn.Parameter(torch.zeros(out_channels))
        self.reset_parameters()

    def reset_parameters(self):
        a = math.sqrt(6.0 / (self.in_channels + self.out_channels))
        torch.nn.init.uniform_(self.lin.weight, -a, a)
        torch.nn.init.zeros_(self.bias)

    def can_restrict(self, x, adj_t):
        """whether ``forward(..., out_rows=)`` can compute just those output rows: a sparse adjacency (the dense
        tensor-core path computes every row).  On a row-partitioned adjacency ``out_rows`` are GLOBAL row ids, the
        same list on every rank, and every rank returns all of those rows (``parallel.pspmm_rows``)."""
        from . import parallel
        if isinstance(adj_t, parallel.ShardedAdj):
            return parallel.RESTRICT_LAST and not _ops.structure_of(adj_t.local).dense_ok
        return not _ops.structure_of(adj_t).dense_ok

    def uses_agg_buffer(self, x, adj_t):
        """will ``forward(x, adj_t)`` (all rows) take the aggregate-buffer path (``_ops.AggLinear``)?"""
        parts = _as_parts(x)
        live = sum(p.size(1) for p in parts if not _is_const(p))
        return REASSOCIATE and live < self.out_channels and _agg_buffer_ok(adj_t, parts)

    def forward(self, x, adj_t, act=_ops.ACT_NONE, drop_p=0.0, out_rows=None, sparse_grad=False, grad_premasked=False,
                premask_input=None):
        """``grad_premasked``: the only consumer of this layer's relu(-dropout) output applies the relu mask to the
        gradient itself (see ``premask_input``), so this layer's backward must not.  ``premask_input`` (the dropout
        scale of the layer that produced x): x is such an output and this conv is its only consumer -- the backward of
        the row-subset SpMM writes the gradient w.r.t. the producer's PRE-activation (mask in the SpMM epilogue; saves
        the separate relu-backward pass over [N, F]).  Both are set together by ``BaseGNN.forward``."""
        parts = _as_parts(x)
        ws = _split_cols(self.lin.weight, parts)
        seed = _ops.new_seed() if drop_p > 0 else 0
        if grad_premasked and not (out_rows is None and self.uses_agg_buffer(x, adj_t)):
            raise RuntimeError("grad_premasked is only implemented for the aggregate-buffer path")
        if premask_input is not None and (out_rows is None or len(parts) != 1):
            raise RuntimeError("premask_input needs the row-restricted path and a single input block")
        if out_rows is not None:
            # only these rows of the layer output, as a compact [T, out] matrix: (A_hat[rows, :] x) W^T + b.
            # Aggregating first keeps the linear map and both of its backward GEMMs at T rows instead of N.
            if not self.can_restrict(x, adj_t):
                raise RuntimeError("out_rows: this layer / adjacency cannot restrict its output rows")
            from . import parallel
            if isinstance(adj_t, parallel.ShardedAdj):
                if parallel.RESTRICT_COMBINE == "rs":
                    # every rank maps its 1 / R of the requested rows and the results are all-gathered
                    aggs = [parallel.pspmm_rows(adj_t, p, out_rows, reduce="sum", sharded=True, premask=premask_input)
                            for p in parts]
                    y = _ops.fused_linear(aggs, ws, self.bias, act, drop_p, seed)
                    return parallel.gather_rows(y, adj_t.group, tag="restricted rows")[: out_rows.numel()]
                aggs = [parallel.pspmm_rows(adj_t, p, out_rows, reduce="sum", premask=premask_input) for p in parts]
            else:
                aggs = [_ops.spmm_rows(adj_t, p, out_rows, reduce="sum", premask=premask_input) for p in parts]
            return _ops.fused_linear(aggs, ws, self.bias, act, drop_p, seed)
        live = sum(p.size(1) for p in parts if not _is_const(p))
        if REASSOCIATE and live < self.out_channels:
            # A_hat (x W^T) = (A_hat x) W^T.  The aggregation is the HBM-bound half of the layer, so run it on
            # whichever side is narrower: only the blocks that change between steps (the trainable embedding,
            # 50 of citation2-shape's 178 input columns) are aggregated per step; the aggregate of a constant
            # block (data.x) is computed once per (adjacency, tensor) and kept.  Rounding differs from the
            # reference's order by a few ulp (inside the 1e-5 bar, tests/test_gpu_model.py).
            if _agg_buffer_ok(adj_t, parts):
                buf, holder, offs, xs = _agg_buffer(adj_t, parts)
                return _ops.agg_linear(adj_t, buf, holder, offs, xs, self.lin.weight, self.bias, act, drop_p, seed,
                                       sparse_grad=sparse_grad, grad_premasked=grad_premasked)
            aggs = [_const_aggregate(adj_t, p, "sum") if _is_const(p)
                    else _ops.spmm(adj_t, p, reduce="sum", sparse_grad=sparse_grad) for p in parts]
            return _ops.fused_linear(aggs, ws, self.bias, act, drop_p, seed)
        z = _ops.fused_linear(parts, ws)
        return _ops.spmm(adj_t, z, reduce="sum", bias=self.bias, relu=(act == _ops.ACT_RELU),
                         drop_p=drop_p, seed=seed, sparse_grad=sparse_grad)


class TransformerConv(torch.nn.Module):
    """PyG 2.0.1 ``TransformerConv(in, out)`` with its defaults (heads = 1, concat, no beta gate, no edge
    features, attention dropout 0, root weight, bias) -- the conv of the reference's Transformer encoder
    (layer.py:57-63), which main.py feeds a value-less adjacency (main.py:181-184):

        out_i = lin_skip(x_i) + sum_{j in N(i)} softmax_j( <lin_query(x_i), lin_key(x_j)> / sqrt(out) ) lin_value(x_j)

    Kernels: four tcgen05 GEMMs, the edge-dot kernel over the stored entries for the scores, a per-row softmax
    (csrc/attn.cu), the SpMM kernel with the attention weights as values, and the skip connection accumulated in
    a GEMM epilogue.  Parameters: lin_key / lin_query / lin_value / lin_skip (.weight, .bias).

    On a row-partitioned adjacency (``parallel.ShardedAdj``) rank r holds rows [lo, hi) of x and the row block
    A[lo:hi, :].  Every input block is all-gathered (``parallel.gather_rows``; backward: the reduce-scatter of its
    gradient), key and value of ALL rows come from one GEMM with the two weights stacked, queries and the skip term
    from the local rows only, and the block's attention runs in ``forward_block`` (DESIGN.md section 6)."""

    def __init__(self, in_channels, out_channels, heads=1):
        super().__init__()
        if heads != 1:
            raise NotImplementedError("the reference uses the default heads = 1 (layer.py:63)")
        self.in_channels, self.out_channels = in_channels, out_channels
        self.lin_key = _Lin(in_channels, out_channels)
        self.lin_query = _Lin(in_channels, out_channels)
        self.lin_value = _Lin(in_channels, out_channels)
        self.lin_skip = _Lin(in_channels, out_channels)

    def reset_parameters(self):
        for lin in (self.lin_key, self.lin_query, self.lin_value, self.lin_skip):
            lin.reset_parameters()

    def forward(self, x, adj_t, act=_ops.ACT_NONE, drop_p=0.0, sparse_grad=False, attention=None):
        """``attention`` (row-partitioned adjacency only): the per-block attention ``attention(q, kv, adj, scale)``,
        by default ``_ops.block_attention``; a test can put a reference restatement in its place."""
        from . import parallel
        if isinstance(adj_t, parallel.ShardedAdj):
            parts = _as_parts(x)
            fulls = [_gather_input(p, adj_t) for p in parts]
            return self.forward_block(parts, fulls, adj_t.local, act, drop_p, attention)
        parts = _as_parts(x)
        x = parts[0] if len(parts) == 1 else torch.cat(parts, -1)
        st = _ops.structure_of(adj_t)
        q, k, v = self.lin_query(x), self.lin_key(x), self.lin_value(x)
        score = _ops.EdgeDot.apply(torch.cat([q, k], 0), st.entry_pairs())          # <q_i, k_j> per stored entry
        alpha = _ops.SegmentSoftmax.apply(score, st.rowptr, 1.0 / math.sqrt(self.out_channels))
        agg = _ops.SpMMValues.apply(alpha, v, adj_t)
        return _ops.AddLinear.apply(x, self.lin_skip.weight, self.lin_skip.bias, agg, int(act), float(drop_p),
                                    _ops.new_seed() if drop_p > 0 else 0)

    def forward_block(self, parts, fulls, adj, act=_ops.ACT_NONE, drop_p=0.0, attention=None):
        """the conv on one row block, no collective: ``parts`` are the block's own rows of every input block,
        ``fulls`` the same blocks over every column of ``adj`` (the block's rows of the adjacency).  The linears run
        on column slices of the weights, one GEMM per input block, so [emb | x] is never concatenated."""
        q = _ops.fused_linear(parts, _split_cols(self.lin_query.weight, parts), self.lin_query.bias)
        w_kv = torch.cat([self.lin_key.weight, self.lin_value.weight], 0)      # one GEMM -> [n_cols, 2F] = [k | v]
        b_kv = torch.cat([self.lin_key.bias, self.lin_value.bias], 0)
        kv = _ops.fused_linear(fulls, _split_cols(w_kv, fulls), b_kv)
        agg = (attention or _ops.block_attention)(q, kv, adj, 1.0 / math.sqrt(self.out_channels))
        return _ops.fused_linear(parts, _split_cols(self.lin_skip.weight, parts), self.lin_skip.bias, act, drop_p,
                                 _ops.new_seed() if drop_p > 0 else 0, addend=agg)


def _gather_input(x_local, sadj):
    """all rows [R*blk, w] of a row-partitioned input block.  A block marked constant (``mark_constant``: data.x) is
    gathered once and kept on the adjacency object, keyed on its storage, shape and version counter like
    ``_const_aggregate``; any other block goes through ``parallel.gather_rows`` (backward: reduce-scatter)."""
    from . import parallel
    if not _is_const(x_local):
        return parallel.gather_rows(parallel.pad_rows(x_local, sadj.blk), sadj.group, tag="attention input")
    cache = sadj.__dict__.setdefault("_plnlp_const_gather", {})
    key = (x_local.data_ptr(), tuple(x_local.shape), x_local.stride(0), x_local._version)
    hit = cache.get(key)
    if hit is None:
        cache.clear()                       # one constant block per adjacency: never hold stale copies
        with torch.no_grad():
            hit = cache[key] = parallel.all_gather_rows(parallel.pad_rows(x_local, sadj.blk), sadj.group,
                                                        name="nccl all_gather (constant attention input)")
    return hit


class BaseGNN(torch.nn.Module):
    """layer stacking of layer.py:7-27: relu + dropout after every conv but the last; a 1-layer
    net also applies them to its only conv."""

    def __init__(self, dropout, num_layers):
        super().__init__()
        self.convs = torch.nn.ModuleList()
        self.dropout = dropout
        self.num_layers = num_layers

    def reset_parameters(self):
        for conv in self.convs:
            conv.reset_parameters()

    def forward(self, x, adj_t, out_rows=None, sparse_grad=False):
        """``out_rows`` (extension; sorted distinct node ids): the caller only reads these rows of the output.
        Returns ``(h, restricted)``: when the last conv can restrict itself, h is the compact [len(out_rows), H]
        matrix of just those rows (restricted = True), otherwise the full output (restricted = False) -- and
        the last conv is then told (``sparse_grad``) that its output gradient will be zero outside a few rows,
        so its backward measures and skips them."""
        p = self.dropout if self.training else 0.0
        last = len(self.convs) - 1
        restricted = False
        will_restrict = (out_rows is not None and getattr(self.convs[last], "can_restrict", None)
                         and self.convs[last].can_restrict(None, adj_t))
        premask = False
        for i, conv in enumerate(self.convs):
            fused = i < last or self.num_layers == 1
            kw = {}
            if i == last and will_restrict:
                kw["out_rows"], restricted = out_rows, True
                if premask:
                    kw["premask_input"] = 1.0 / (1.0 - p)
            elif i == last and (sparse_grad or out_rows is not None):
                kw["sparse_grad"] = True
            elif (i == last - 1 and will_restrict and FUSE_RELU_BWD and isinstance(conv, GCNConv)
                  and isinstance(self.convs[last], GCNConv) and torch.is_grad_enabled() and conv.uses_agg_buffer(x, adj_t)):
                # this layer's relu(-dropout) output feeds ONLY the row-subset SpMM of the last conv: that SpMM's
                # backward applies the relu mask in its epilogue and this layer skips its relu-backward pass
                kw["grad_premasked"] = premask = True
            x = conv(x, adj_t, act=_ops.ACT_RELU if fused else _ops.ACT_NONE, drop_p=p if fused else 0.0, **kw)
        return x if out_rows is None else (x, restricted)


def _stack(conv_cls, in_channels, hidden_channels, out_channels, num_layers):
    dims = [in_channels] + [hidden_channels] * (num_layers - 1) + [out_channels]
    return [conv_cls(dims[i], dims[i + 1]) for i in range(num_layers)]


class SAGE(BaseGNN):
    def __init__(self, in_channels, hidden_channels, out_channels, num_layers, dropout):
        super().__init__(dropout, num_layers)
        self.convs.extend(_stack(SAGEConv, in_channels, hidden_channels, out_channels, num_layers))


class GCN(BaseGNN):
    def __init__(self, in_channels, hidden_channels, out_channels, num_layers, dropout):
        super().__init__(dropout, num_layers)
        self.convs.extend(_stack(GCNConv, in_channels, hidden_channels, out_channels, num_layers))


class WSAGE(BaseGNN):
    """layer.py:48-54: the weighted-sum variant of SAGE (PyG GraphConv)"""

    def __init__(self, in_channels, hidden_channels, out_channels, num_layers, dropout):
        super().__init__(dropout, num_layers)
        self.convs.extend(_stack(GraphConv, in_channels, hidden_channels, out_channels, num_layers))


class Transformer(BaseGNN):
    """layer.py:57-63"""

    def __init__(self, in_channels, hidden_channels, out_channels, num_layers, dropout):
        super().__init__(dropout, num_layers)
        self.convs.extend(_stack(TransformerConv, in_channels, hidden_channels, out_channels, num_layers))


class MLPPredictor(torch.nn.Module):
    """layer.py:66-87: Hadamard of the two endpoint embeddings -> (Linear, relu, dropout) x (L-1)
    -> Linear(-> out_channels).  ``forward(x_i, x_j)`` -> [B, out_channels]."""

    def __init__(self, in_channels, hidden_channels, out_channels, num_layers, dropout):
        super().__init__()
        dims = [in_channels] + [hidden_channels] * (num_layers - 1) + [out_channels]
        self.lins = torch.nn.ModuleList(_Lin(dims[i], dims[i + 1]) for i in range(num_layers))
        self.dropout = dropout

    def reset_parameters(self):
        for lin in self.lins:
            lin.reset_parameters()

    def _tail(self, x):
        p = self.dropout if self.training else 0.0
        for lin in self.lins[:-1]:
            x = lin(x, act=_ops.ACT_RELU, drop_p=p)
        last = self.lins[-1]
        if last.out_features == 1:
            return _ops.MLPOut.apply(x, last.weight, last.bias)
        return last(x)

    def forward(self, x_i, x_j):
        return self._tail(x_i * x_j)

    def score_edges(self, h, edges):
        """predictor(h[edges[:,0]], h[edges[:,1]]) with the gather and Hadamard fused.  Without autograd
        (scoring in ``BaseModel.test``: up to 86.6 M pairs per split on citation2-shape) the whole head runs
        as ONE kernel that neither materialises the Hadamard product nor stores the hidden activation."""
        params = self.flat_params()
        if not torch.is_grad_enabled() and self.lins[-1].out_features == 1 and _ops.fused_edge_mlp_ok(h, params):
            p = self.dropout if self.training else 0.0
            score, _ = _ops.edge_mlp_fwd_raw(h, edges, params[0], params[1], params[2], params[3], p,
                                             _ops.new_seed() if p > 0 else 0, need_a1=False)
            return score.reshape(-1, 1)
        return self._tail(_ops.GatherHadamard.apply(h, edges))

    def flat_params(self):
        out = []
        for lin in self.lins:
            out += [lin.weight, lin.bias]
        return out


class NCNPredictor(torch.nn.Module):
    """Neural Common Neighbour (Wang, Yang and Zhang, ICLR 2024; an extension, the reference has no such head): the
    MLP of ``MLPPredictor`` over [h_u * h_v | c_uv], c_uv the sum of h_w over the common neighbours w of u and v
    (``heuristics.common_neighbour_lists``).  ``lins[0]`` is one Linear(2 H, hidden) whose weight reads as the MLP on
    the concatenation; the concatenation itself is never built (one GEMM per block into the same output).  Relu +
    dropout follow every Linear but the last."""

    def __init__(self, in_channels, hidden_channels, out_channels, num_layers, dropout):
        super().__init__()
        dims = [2 * in_channels] + [hidden_channels] * (num_layers - 1) + [out_channels]
        self.lins = torch.nn.ModuleList(_Lin(dims[i], dims[i + 1]) for i in range(num_layers))
        self.in_channels = in_channels
        self.dropout = dropout

    def reset_parameters(self):
        for lin in self.lins:
            lin.reset_parameters()

    def forward(self, x_i, x_j):
        raise TypeError("NCNPredictor scores a pair from the graph as well as its two embeddings: call "
                        "score_edges(h, edges, cn) with cn = heuristics.common_neighbour_lists(adj_t, edges)")

    def score_edges(self, h, edges, cn):
        """-> [P, out_channels]: the head on h [N, H] for the pairs ``edges`` (rows of h) with ``cn = (rowptr int64
        [P + 1], col)`` their common-neighbour lists in the row numbering of h"""
        had = _ops.GatherHadamard.apply(h, edges)
        c = _ops.common_neighbour_sum(h, cn)
        H = self.in_channels
        p = self.dropout if self.training else 0.0
        first = self.lins[0]
        W = first.weight
        if len(self.lins) == 1:
            if first.out_features == 1:
                return _ops.MLPOut.apply(had, W[:, :H], first.bias) + _ops.MLPOut.apply(c, W[:, H:], None)
            return _ops.fused_linear([had, c], [W[:, :H], W[:, H:]], first.bias)
        x = _ops.fused_linear([had, c], [W[:, :H], W[:, H:]], first.bias, _ops.ACT_RELU, p,
                              _ops.new_seed() if p > 0 else 0)
        for lin in self.lins[1:-1]:
            x = lin(x, act=_ops.ACT_RELU, drop_p=p)
        last = self.lins[-1]
        if last.out_features == 1:
            return _ops.MLPOut.apply(x, last.weight, last.bias)
        return last(x)

    def flat_params(self):
        out = []
        for lin in self.lins:
            out += [lin.weight, lin.bias]
        return out


class DotPredictor(torch.nn.Module):
    """layer.py:167-176: sum(x_i * x_j, -1) -> [B]."""

    def reset_parameters(self):
        return

    def forward(self, x_i, x_j):
        return _ops.row_dot(x_i, x_j)

    def score_edges(self, h, edges):
        return _ops.EdgeDot.apply(h, edges)

    def flat_params(self):
        return []


def _endpoints(h, edges):
    """x_i = h[edge[0]], x_j = h[edge[1]] (model.py:155-156) as two [P, H] matrices"""
    return _ops.GatherRows.apply(h, edges, 0), _ops.GatherRows.apply(h, edges, 1)


def _stacked_dot(u, v, edges):
    """score[p] = <u[src_p], v[dst_p]> for node-level matrices u, v [N, H]: the edge-dot kernels on the stacked
    matrix [u; v] with the destination index shifted by N"""
    n = u.size(0)
    e = torch.where(edges < 0, edges + n, edges)
    shift = torch.tensor([0, n], dtype=edges.dtype, device=edges.device)
    return _ops.EdgeDot.apply(torch.cat([u, v], 0), e + shift)


class _NodeMLP(torch.nn.Module):
    """the shared head of MLPDotPredictor / MLPBilPredictor (layer.py:119-164): every Linear is followed by relu +
    dropout, applied to x_i and x_j separately.  While no dropout is active (eval, or p = 0) the transform of an
    endpoint depends on the node only, so ``score_edges`` applies it to the N rows of h once instead of to 2P
    gathered rows; with dropout active the two sides of every pair get their own masks, as in the reference."""

    def __init__(self, in_channels, hidden_channels, num_layers, dropout):
        super().__init__()
        dims = [in_channels] + [hidden_channels] * num_layers
        self.lins = torch.nn.ModuleList(_Lin(dims[i], dims[i + 1]) for i in range(num_layers))
        self.dropout = dropout

    def _mlp(self, x):
        p = self.dropout if self.training else 0.0
        for lin in self.lins:
            x = lin(x, act=_ops.ACT_RELU, drop_p=p)
        return x

    def _node_level(self):
        return not (self.training and self.dropout > 0)


class MLPDotPredictor(_NodeMLP):
    """layer.py:119-139: sum(mlp(x_i) * mlp(x_j), -1) -> [B]"""

    def reset_parameters(self):
        for lin in self.lins:
            lin.reset_parameters()

    def forward(self, x_i, x_j):
        return _ops.row_dot(self._mlp(x_i), self._mlp(x_j))

    def score_edges(self, h, edges):
        if self._node_level():
            return _ops.EdgeDot.apply(self._mlp(h), edges)
        return self.forward(*_endpoints(h, edges))


class MLPBilPredictor(_NodeMLP):
    """layer.py:142-164: sum(bilin(mlp(x_i)) * mlp(x_j), -1) -> [B]"""

    def __init__(self, in_channels, hidden_channels, num_layers, dropout):
        super().__init__(in_channels, hidden_channels, num_layers, dropout)
        self.bilin = _Lin(hidden_channels, hidden_channels, bias=False)

    def reset_parameters(self):
        for lin in self.lins:
            lin.reset_parameters()
        self.bilin.reset_parameters()

    def forward(self, x_i, x_j):
        return _ops.row_dot(self.bilin(self._mlp(x_i)), self._mlp(x_j))

    def score_edges(self, h, edges):
        if self._node_level():
            z = self._mlp(h)
            return _stacked_dot(self.bilin(z), z, edges)
        return self.forward(*_endpoints(h, edges))


class BilinearPredictor(torch.nn.Module):
    """layer.py:179-189: sum(bilin(x_i) * x_j, -1) -> [B]; ``score_edges`` maps the N rows of h once."""

    def __init__(self, hidden_channels):
        super().__init__()
        self.bilin = _Lin(hidden_channels, hidden_channels, bias=False)

    def reset_parameters(self):
        self.bilin.reset_parameters()

    def forward(self, x_i, x_j):
        return _ops.row_dot(self.bilin(x_i), x_j)

    def score_edges(self, h, edges):
        return _stacked_dot(self.bilin(h), h, edges)


class MLPCatPredictor(torch.nn.Module):
    """layer.py:90-116: the MLP on [x_i | x_j] and on [x_j | x_i], averaged -> [B, out_channels].  Both orders run
    as ONE batch of 2B rows through the tensor-core GEMMs (the same weights serve both)."""

    def __init__(self, in_channels, hidden_channels, out_channels, num_layers, dropout):
        super().__init__()
        dims = [2 * in_channels] + [hidden_channels] * (num_layers - 1) + [out_channels]
        self.lins = torch.nn.ModuleList(_Lin(dims[i], dims[i + 1]) for i in range(num_layers))
        self.dropout = dropout

    def reset_parameters(self):
        for lin in self.lins:
            lin.reset_parameters()

    def forward(self, x_i, x_j):
        p = self.dropout if self.training else 0.0
        x = torch.cat([torch.cat([x_i, x_j], -1), torch.cat([x_j, x_i], -1)], 0)      # [2B, 2H]
        for lin in self.lins[:-1]:
            x = lin(x, act=_ops.ACT_RELU, drop_p=p)
        last = self.lins[-1]
        if last.out_features == 1:
            s = _ops.MLPOut.apply(x, last.weight, last.bias).reshape(-1)
            return _ops.PairMean.apply(s).reshape(-1, 1)
        y = last(x)
        B = x_i.size(0)
        return (y[:B] + y[B:]) / 2

    def score_edges(self, h, edges):
        return self.forward(*_endpoints(h, edges))



"""``BaseModel`` with the reference's constructor / train / test surface
(/root/reference/plnlp/model.py), re-plumbed on the plnlp_b200 kernels.

What changes underneath (results are the reference's):
  * negatives are sampled on the GPU, the epoch permutation is drawn on the GPU;
  * ``[emb | x]`` is never concatenated, the first conv consumes the two blocks;
  * endpoint gather + Hadamard + predictor + pairwise loss + d loss/d score run as one fused
    autograd node (``_ops.EdgeScoreLoss``);
  * the running loss is accumulated on the device: ONE host sync per epoch instead of one per
    batch (model.py:170);
  * ``test`` encodes once (the reference recomputes an identical ``h``, model.py:190,204) and
    ranks on the GPU.
"""
from __future__ import annotations

import os

import torch

from . import _ops, profiling
from .layer import *  # noqa: F401,F403
from .layer import (GCN, SAGE, WSAGE, BilinearPredictor, DotPredictor, MLPBilPredictor, MLPCatPredictor,
                    MLPDotPredictor, MLPPredictor, NCNPredictor, mark_constant)
from .loss import *  # noqa: F401,F403
from .utils import *  # noqa: F401,F403
from .utils import evaluate_hits, evaluate_mrr, get_pos_neg_edges

_IN_SCOPE_LOSSES = ('AUC', 'HingeAUC', 'WeightedHingeAUC')

# skip all-zero gradient rows in the backward of the last conv (see train_batch)
ROW_SPARSE_GRAD = os.environ.get("PLNLP_ROW_SPARSE_GRAD", "1") != "0"
# do the index work of the next batch on a side stream while the current one runs (BaseModel.prepare_batch)
PREPARE_AHEAD = os.environ.get("PLNLP_PREPARE_AHEAD", "1") != "0"


class PreparedBatch:
    __slots__ = ("ids", "pos_edge", "neg_edge", "event", "cn")

    def __init__(self, ids, pos_edge, neg_edge, event, cn=None):
        self.ids, self.pos_edge, self.neg_edge, self.event, self.cn = ids, pos_edge, neg_edge, event, cn


def ncn_restrict(edges, cn):
    """the rows a restricted last conv must compute for the NCN predictor, which reads h at the endpoints AND at
    their common neighbours: (ids = the sorted union of the ids in ``edges`` [P, 2] and in the lists ``cn =
    (rowptr, col)``, ``edges`` renumbered into ids, ``(rowptr, col renumbered into ids)``).  ids[edges'] == edges
    and ids[col'] == col."""
    rowptr, col = cn
    ids = torch.unique(torch.cat([edges.reshape(-1), col]))
    return ids, torch.searchsorted(ids, edges), (rowptr, torch.searchsorted(ids, col))


class BaseModel(object):
    """Same keyword arguments as model.py:45-48."""

    def __init__(self, lr, dropout, grad_clip_norm, gnn_num_layers, mlp_num_layers, emb_hidden_channels,
                 gnn_hidden_channels, mlp_hidden_channels, num_nodes, num_node_feats, gnn_encoder_name,
                 predictor_name, loss_func, optimizer_name, device, use_node_feats, train_node_emb,
                 pretrain_emb=None):
        device = torch.device(device)
        if device.type != 'cuda':
            raise RuntimeError("plnlp_b200.BaseModel runs on a CUDA (sm_100) device only; there is no CPU path")
        self.loss_func_name = loss_func
        self.num_nodes = num_nodes
        self.num_node_feats = num_node_feats
        self.use_node_feats = use_node_feats
        self.train_node_emb = train_node_emb
        self.clip_norm = grad_clip_norm
        self.device = device

        self.input_channels, self.emb = create_input_layer(
            num_nodes=num_nodes, num_node_feats=num_node_feats, hidden_channels=emb_hidden_channels,
            use_node_feats=use_node_feats, train_node_emb=train_node_emb, pretrain_emb=pretrain_emb)
        if self.emb is not None:
            self.emb = self.emb.to(device)

        self.encoder = create_gnn_layer(input_channels=self.input_channels, hidden_channels=gnn_hidden_channels,
                                        num_layers=gnn_num_layers, dropout=dropout,
                                        encoder_name=gnn_encoder_name).to(device)
        self.predictor = create_predictor_layer(hidden_channels=mlp_hidden_channels, num_layers=mlp_num_layers,
                                                dropout=dropout, predictor_name=predictor_name)
        if self.predictor is None:
            raise NotImplementedError(f"predictor {predictor_name!r}")
        self.predictor = self.predictor.to(device)

        # same parameter order as model.py:81-83: encoder, predictor, embedding
        self.para_list = list(self.encoder.parameters()) + list(self.predictor.parameters())
        if self.emb is not None:
            self.para_list += list(self.emb.parameters())

        trainable = [p for p in self.para_list if p.requires_grad]
        if optimizer_name == 'AdamW':
            self.optimizer = torch.optim.AdamW(trainable, lr=lr, fused=True)
        elif optimizer_name == 'SGD':
            self.optimizer = torch.optim.SGD(trainable, lr=lr, momentum=0.9, weight_decay=1e-5, nesterov=True)
        else:
            self.optimizer = torch.optim.Adam(trainable, lr=lr, fused=True)
        self.last_epoch_stats = {}
        # multi-GPU state, set by the launcher (bench.py / tests): see plnlp_b200/parallel.py
        self.world_size, self.rank, self.partitioned = 1, 0, False

    # ------------------------------------------------------------------
    def param_init(self):
        self.encoder.reset_parameters()
        self.predictor.reset_parameters()
        if self.emb is not None:
            torch.nn.init.xavier_uniform_(self.emb.weight)

    def input_parts(self, data):
        """the blocks of the encoder input, in the column order of model.py:98-105."""
        if self.use_node_feats:
            x = self._features(data)
            if self.train_node_emb:
                return (self.emb.weight, x)
            return (x,)
        return (self.emb.weight,)

    def _features(self, data):
        """data.x on the device in fp32, converted once per tensor and marked constant so the first conv can
        keep its aggregate (layer.mark_constant)"""
        x = data.x
        key = (id(x), x.data_ptr(), x._version)
        if getattr(self, "_x_key", None) != key:
            xd = x.to(self.device).to(torch.float32)
            if xd is x:
                xd = x.view(x.shape)          # do not tag the caller's tensor object
            self._x_key, self._x_dev = key, mark_constant(xd.detach())
        return self._x_dev

    def create_input_feat(self, data):
        """model.py:98-105 (materialised; the training loop uses ``input_parts`` instead)."""
        parts = self.input_parts(data)
        return parts[0] if len(parts) == 1 else torch.cat(parts, dim=-1)

    def _loss_name(self, has_margin):
        """the dispatch of model.py:107-126: margin / weight losses need split_edge['train']['weight'] and
        fall back to AUC without it; unknown names are AUC"""
        name = self.loss_func_name
        if name in ('CE', 'InfoNCE', 'LogRank', 'HingeAUC'):
            return name
        if name in ('AdaAUC', 'WeightedAUC', 'AdaHingeAUC', 'WeightedHingeAUC') and has_margin:
            return name
        return 'AUC'

    def calculate_loss(self, pos_out, neg_out, num_neg, margin=None):
        return _ops.pair_loss(self._loss_name(margin is not None), pos_out, neg_out, num_neg, margin)

    # ------------------------------------------------------------------
    def _sparse_rows(self, pos_edge, neg_edge):
        """does this batch touch a small part of the node set?  (then the last conv computes only the endpoint rows)"""
        n_touch = 2 * (pos_edge.size(0) + neg_edge.size(0)) * (self.world_size if self.partitioned else 1)
        return ROW_SPARSE_GRAD and n_touch < 0.5 * self.num_nodes

    def _ncn(self):
        """is the predictor NCN?  (raises on a row-partitioned model, where it is not implemented)"""
        if not isinstance(self.predictor, NCNPredictor):
            return False
        if self.partitioned:
            raise NotImplementedError("the NCN predictor is not implemented on a row-partitioned model")
        return True

    def _side(self):
        if getattr(self, "_side_stream", None) is None:
            self._side_stream = torch.cuda.Stream(device=self.device)
        return self._side_stream

    def prepare_batch(self, data, pos_edge, neg_edge, wait_main=True):
        """The index work of one step that does not depend on any parameter: the sorted distinct endpoint rows of the
        batch (on a row-partitioned run: the union over ranks), the edges renumbered into that compact table, the
        row-subset SpMM plan of the last conv and the index vector of its backward.  It runs on a SIDE stream, so
        ``run_batches`` can issue it for batch i + 1 while the GPU is still busy with batch i: the host reads it needs
        (``torch.unique``, the plan's item counts) then cost nothing on the main stream.  ``wait_main=False``: the
        edge tensors were themselves produced on the side stream (``run_batches``), so the side stream must NOT wait
        for the main one -- that would queue this work behind the whole step in flight.  Returns None when the batch
        is not row-sparse or the last conv cannot restrict itself (``train_batch`` then does everything itself)."""
        ncn = self._ncn()
        if not self._sparse_rows(pos_edge, neg_edge):
            return None
        last = self.encoder.convs[-1]
        parts = self.input_parts(data) if len(self.encoder.convs) == 1 else None
        if not (getattr(last, "can_restrict", None) and last.can_restrict(parts, data.adj_t)):
            return None
        from . import graph, heuristics
        main = torch.cuda.current_stream()
        side = self._side()
        # NCN: the neighbour table is built once per adjacency, on the main stream, and the side stream reads it below,
        # so the side stream must wait for that build.  Only a build made here is waited for: a prepared batch never
        # waits for the step in flight.
        fresh_table = ncn and heuristics.cached_table(data.adj_t) is None
        if fresh_table:
            heuristics.neighbour_table(data.adj_t)
        if wait_main:                                            # the edge tensors were produced on the main stream
            side.wait_stream(main)
        elif fresh_table:
            built = torch.cuda.Event()
            built.record(main)
            side.wait_event(built)
        with torch.cuda.stream(side):
            mine = torch.cat([pos_edge, neg_edge], 0)
            cn = None
            if ncn:                                              # the list total is read on the side stream too
                ids, inv, cn = ncn_restrict(mine, heuristics.common_neighbour_lists(data.adj_t, mine))
                st = graph.structure_of(data.adj_t)
            elif self.partitioned:
                from . import parallel
                if not parallel.RESTRICT_LAST:
                    return None
                ids = parallel.union_ids(mine.reshape(-1), data.adj_t.group)
                inv = torch.searchsorted(ids, mine)
                st = graph.structure_of(data.adj_t.cols())
            else:
                ids, inv = torch.unique(mine, return_inverse=True)
                st = graph.structure_of(data.adj_t)
            plan = graph.build_subset_plan(st.fwd, st.rowptr, ids)
            x_index = torch.full((st.n_rows,), -1, dtype=torch.int32, device=ids.device)
            x_index[ids] = torch.arange(ids.numel(), dtype=torch.int32, device=ids.device)
            ids._plnlp_prepared = {id(st): (plan, x_index)}      # picked up by _ops.SpMMRows
            n_pos = pos_edge.size(0)
            prep = PreparedBatch(ids, inv[:n_pos], inv[n_pos:], torch.cuda.Event(), cn)
            for t in [ids, inv, x_index] + list(cn or ()) + graph.plan_tensors(plan):
                t.record_stream(main)                            # allocated on the side stream, consumed on the main one
            prep.event.record(side)
        return prep

    def train_batch(self, data, pos_edge, neg_edge, num_neg, weight_margin=None, prepared=None):
        """one optimisation step (model.py:148-167).  pos_edge [B,2], neg_edge [B*num_neg,2].
        Returns the batch loss as a 0-d device tensor (no host sync).  ``prepared``: the result of
        ``prepare_batch`` for these edges (else the same index work is done here, on the main stream)."""
        self.optimizer.zero_grad(set_to_none=True)
        # Scoring reads h only at the endpoint rows of the batch, and d loss / d h is non-zero only there.  When
        # those are a small part of the node set (citation2-shape: ~10 %) the last conv computes just those
        # rows (compact h, edges renumbered) and its backward gathers just their gradient rows; a conv that cannot
        # restrict itself is told that its output gradient is row-sparse (``sparse_grad``) and skips the zero rows
        # in its backward.
        sparse_rows = self._sparse_rows(pos_edge, neg_edge)
        restricted = False
        ncn = self._ncn()
        cn = None               # NCN: the common-neighbour lists of [pos_edge; neg_edge], in the row numbering of h
        if self.partitioned:
            from . import parallel
        if prepared is not None:
            torch.cuda.current_stream().wait_event(prepared.event)
            h, restricted = self.encoder(self.input_parts(data), data.adj_t, out_rows=prepared.ids)
            assert restricted
            pos_edge, neg_edge, cn = prepared.pos_edge, prepared.neg_edge, prepared.cn
        elif sparse_rows and not self.partitioned:
            mine = torch.cat([pos_edge, neg_edge], 0)
            if ncn:
                # h is then read at the endpoints and at their common neighbours: the last conv computes the union
                from .heuristics import common_neighbour_lists
                cn = common_neighbour_lists(data.adj_t, mine)
                with profiling.span("torch: union of endpoint and common-neighbour ids + renumber"):
                    ids, inv, cn_local = ncn_restrict(mine, cn)
            else:
                with profiling.span("torch: unique endpoint ids + renumber"):
                    ids, inv = torch.unique(mine, return_inverse=True)
            h, restricted = self.encoder(self.input_parts(data), data.adj_t, out_rows=ids)
            if restricted:
                pos_edge, neg_edge = inv[:pos_edge.size(0)], inv[pos_edge.size(0):]
                if ncn:
                    cn = cn_local
        elif sparse_rows and parallel.RESTRICT_LAST:
            # row-partitioned run: the union of every rank's endpoint rows (the same sorted list everywhere) is
            # what the last conv computes -- as partial products over each rank's column block, summed by one
            # all-reduce (parallel.pspmm_rows) -- so every rank holds the compact h of ALL batches and scores its own
            mine = torch.cat([pos_edge, neg_edge], 0)
            with profiling.span("torch + nccl: union of endpoint ids (all_gather + unique)"):
                ids = parallel.union_ids(mine.reshape(-1), data.adj_t.group)
            h, restricted = self.encoder(self.input_parts(data), data.adj_t, out_rows=ids)
            if restricted:
                inv = torch.searchsorted(ids, mine)
                pos_edge, neg_edge = inv[:pos_edge.size(0)], inv[pos_edge.size(0):]
        else:
            h = self.encoder(self.input_parts(data), data.adj_t, sparse_grad=sparse_rows)
        if self.partitioned and not restricted:
            # row-partitioned encoder (SURVEY 8e): h is this rank's row block and scoring needs arbitrary
            # endpoints.  Fetch just the distinct endpoint rows of this rank's batch from their owners
            # (parallel.FetchRows; gradients return the same way) and score on that compact table.
            if parallel.EXCHANGE == "rows":
                ids, inv = torch.unique(torch.cat([pos_edge, neg_edge], 0), return_inverse=True)
                h = parallel.fetch_rows(h, ids)
                pos_edge, neg_edge = inv[:pos_edge.size(0)], inv[pos_edge.size(0):]
            else:       # all-gather the whole matrix (backward: reduce-scatter of grad_h)
                h = parallel.gather_rows(h)
        loss_name = self._loss_name(weight_margin is not None)
        if isinstance(self.predictor, (DotPredictor, MLPPredictor)):
            head = 'DOT' if isinstance(self.predictor, DotPredictor) else 'MLP'
            p = self.predictor.dropout if (head == 'MLP' and self.predictor.training) else 0.0
            loss = _ops.edge_score_loss(h, pos_edge, neg_edge, num_neg, loss_name, weight=weight_margin,
                                        head=head, params=self.predictor.flat_params(), drop_p=p,
                                        seed=_ops.new_seed() if p > 0 else 0)
        else:
            # the other --predictor choices (layer.py:90-189) and NCN: positives and negatives scored in one pass
            edges = torch.cat([pos_edge, neg_edge], 0)
            if ncn and cn is None:                   # full h: the lists on the batch's global ids
                from .heuristics import common_neighbour_lists
                cn = common_neighbour_lists(data.adj_t, edges)
            score = (self.predictor.score_edges(h, edges, cn) if ncn
                     else self.predictor.score_edges(h, edges)).reshape(-1)
            B = pos_edge.size(0)
            loss = _ops.pair_loss(loss_name, score[:B], score[B:], num_neg, weight_margin)
        loss.backward()
        if getattr(self, 'world_size', 1) > 1:
            self._allreduce_grads()
        with profiling.span("torch: clip_grad_norm + fused Adam step"):
            if self.clip_norm >= 0:
                torch.nn.utils.clip_grad_norm_(self.encoder.parameters(), self.clip_norm)
                pp = list(self.predictor.parameters())
                if pp:
                    torch.nn.utils.clip_grad_norm_(pp, self.clip_norm)
            self.optimizer.step()
        return loss.detach()

    def _allreduce_grads(self):
        """data-parallel edge batches (no counterpart in the reference, SURVEY.md 8e): every rank
        scored its own batch against a replicated encoder; the loss is a SUM over pairs, so summing
        the gradients over ranks gives the gradient of the global batch.  One flat NCCL all-reduce."""
        from . import parallel
        params = self.para_list
        if self.partitioned and self.emb is not None:
            # embedding rows are owned by exactly one rank; their gradient arrived complete through
            # the reduce-scatter of the gathers (owner computes) -> no all-reduce
            own = {id(p) for p in self.emb.parameters()}
            params = [p for p in params if id(p) not in own]
        # AUC-family losses are SUMS over pairs (loss.py:8,14,21,28,35,42): the summed gradient is the gradient of
        # the global batch.  CE / LogRank / InfoNCE are MEANS (loss.py:48,52-53,62): average over ranks, so the
        # step (and what the clip sees) does not depend on the number of GPUs.
        parallel.allreduce_grads(params, average=self._loss_is_mean())
        if self._loss_is_mean() and self.partitioned and self.emb is not None:
            for p in self.emb.parameters():
                if p.grad is not None:
                    p.grad.div_(self.world_size)

    def _loss_is_mean(self):
        return self.loss_func_name in ('CE', 'InfoNCE', 'LogRank')

    def train(self, data, split_edge, batch_size, neg_sampler_name, num_neg, perms=None, neg_edges=None,
              max_batches=None):
        """model.py:128-173.  Extensions (all optional): ``perms`` (iterable of index tensors) and
        ``neg_edges`` ([E,num_neg,2]) replace the shuffle / sampler so a run can be replayed;
        ``max_batches`` stops early (bench time-boxing)."""
        self.encoder.train()
        self.predictor.train()
        if self.world_size > 1 and neg_edges is None:
            # data-parallel edge batches: rank r trains on the r-th contiguous block of the epoch's edges (equal
            # counts on every rank so the per-step collectives line up).  A contiguous block is a VIEW of the
            # caller's (pinned host) tensor, so only this rank's share is copied to the device; a strided pick
            # r, r+R, ... would first gather on the host, inside the epoch.
            tr = split_edge['train']
            n_each = next(iter(tr.values())).size(0) // self.world_size
            tr = {k: v[self.rank * n_each:(self.rank + 1) * n_each] for k, v in tr.items()}
            split_edge = dict(split_edge, train=tr)
        if neg_edges is None:
            pos_train_edge, neg_train_edge = get_pos_neg_edges(
                'train', split_edge, edge_index=data.edge_index, num_nodes=self.num_nodes,
                neg_sampler_name=neg_sampler_name, num_neg=num_neg, device=self.device)
        else:
            pos_train_edge = self._train_pos(split_edge)
            neg_train_edge = neg_edges.to(self.device)
        pos_train_edge = pos_train_edge.to(self.device)
        margin = split_edge['train']['weight'].to(self.device).to(torch.float32) \
            if 'weight' in split_edge['train'] else None

        E = pos_train_edge.size(0)
        if perms is None:
            order = torch.randperm(E, device=self.device)
            perms = [order[i:i + batch_size] for i in range(0, E, batch_size)]
        def batches():
            for it, perm in enumerate(perms):
                if max_batches is not None and it >= max_batches:
                    break
                perm = perm.to(self.device)
                yield (pos_train_edge[perm], neg_train_edge[perm].reshape(-1, 2),
                       margin[perm] if margin is not None else None)

        total_loss, total_examples, n_batches = self.run_batches(data, batches(), num_neg)
        self.last_epoch_stats = {'batches': n_batches, 'examples': total_examples}
        value = total_loss / max(total_examples, 1)
        if self.world_size > 1:
            # every rank scored 1/R of each batch: the global-batch value of model.py:169-173 is the SUM of the
            # ranks' values for the sum-type losses and their average for the mean-type ones
            import torch.distributed as dist
            dist.all_reduce(value)
            if self._loss_is_mean():
                value = value / self.world_size
        return value.item()   # the one host sync of the epoch

    def run_batches(self, data, batches, num_neg):
        """the batch loop of model.py:147-171 over an iterable of (pos_edge [B,2], neg_edge [B*num_neg,2], weight or
        None) device tensors, with the parameter-independent index work of batch i + 1 (``prepare_batch``) issued on
        a side stream right after the kernels of batch i were enqueued.  -> (sum of loss * B as a 0-d fp64 device
        tensor, examples, batches); no host read of the loss."""
        total_loss = torch.zeros((), dtype=torch.float64, device=self.device)
        total_examples = n_batches = 0
        it = iter(batches)
        if not PREPARE_AHEAD:
            for pos_edge, neg_edge, w in it:
                loss = self.train_batch(data, pos_edge, neg_edge, num_neg, w)
                total_loss += loss.double() * pos_edge.size(0)
                total_examples += pos_edge.size(0)
                n_batches += 1
            return total_loss, total_examples, n_batches
        main, side = torch.cuda.current_stream(), self._side()
        side.wait_stream(main)                  # once: the epoch's edge / negative tensors exist from here on

        def fetch():
            """slice out the next batch AND prepare it, all on the side stream (nothing here waits for the step that
            the main stream is busy with)"""
            with torch.cuda.stream(side):
                b = next(it, None)
                if b is None:
                    return None, None, None
                for t in b:
                    if t is not None:
                        t.record_stream(main)
                ready = torch.cuda.Event()
            prep = self.prepare_batch(data, b[0], b[1], wait_main=False)
            ready.record(side)
            return b, prep, ready

        cur, prep, ready = fetch()
        while cur is not None:
            pos_edge, neg_edge, w = cur
            main.wait_event(ready)
            loss = self.train_batch(data, pos_edge, neg_edge, num_neg, w, prepared=prep)
            nxt, nprep, nready = fetch()        # enqueued while the GPU works on the step above
            total_loss += loss.double() * pos_edge.size(0)
            total_examples += pos_edge.size(0)
            n_batches += 1
            cur, prep, ready = nxt, nprep, nready
        return total_loss, total_examples, n_batches

    def _train_pos(self, split_edge):
        tr = split_edge['train']
        if 'edge' in tr:
            return tr['edge']
        return torch.stack([tr['source_node'], tr['target_node']], dim=1)

    # ------------------------------------------------------------------
    @torch.no_grad()
    def batch_predict(self, h, edges, batch_size, adj_t=None):
        """model.py:175-182; scores stay on the device.  ``adj_t``: the adjacency whose common neighbours the NCN
        predictor reads (required for it, unused by the others)."""
        edges = edges.to(self.device)
        if isinstance(self.predictor, NCNPredictor):
            if adj_t is None:
                raise ValueError("batch_predict with the NCN predictor needs adj_t (the graph of the common "
                                 "neighbours)")
            from .heuristics import common_neighbour_lists
            preds = [self.predictor.score_edges(h, e, common_neighbour_lists(adj_t, e)).reshape(-1)
                     for e in (edges[i:i + batch_size] for i in range(0, edges.size(0), batch_size))]
            return torch.cat(preds, dim=0) if preds else torch.empty(0, device=self.device)
        preds = [self.predictor.score_edges(h, edges[i:i + batch_size]).reshape(-1)
                 for i in range(0, edges.size(0), batch_size)]
        return torch.cat(preds, dim=0) if preds else torch.empty(0, device=self.device)

    @torch.no_grad()
    def encode_for_test(self, data):
        """model.py:189-194: eval-mode encoding plus the mean row that index -1 resolves to."""
        h = self.encoder(self.input_parts(data), data.adj_t)
        if self.partitioned:
            # row-partitioned encoder: every rank evaluates against the whole matrix (all-gather of the blocks,
            # padding rows dropped) -- scoring and ranking are then the single-GPU code
            from . import parallel
            h = parallel.all_gather_rows(h.contiguous(), data.adj_t.group)[: data.adj_t.n_global]
        mean_h = _ops.colsum_raw(h, 1.0 / h.size(0)).reshape(1, -1)
        return torch.cat([h, mean_h], dim=0)

    @torch.no_grad()
    def test(self, data, split_edge, batch_size, evaluator, eval_metric):
        """model.py:184-226 -> {'Hits@20'|'Hits@50'|'Hits@100'|'MRR': (valid, test)}"""
        self._ncn()
        self.encoder.eval()
        self.predictor.eval()
        h = self.encode_for_test(data)
        pos_valid_edge, neg_valid_edge = get_pos_neg_edges('valid', split_edge, device=self.device)
        pos_test_edge, neg_test_edge = get_pos_neg_edges('test', split_edge, device=self.device)
        adj = data.adj_t
        pos_valid_pred = self.batch_predict(h, pos_valid_edge, batch_size, adj_t=adj)
        neg_valid_pred = self.batch_predict(h, neg_valid_edge, batch_size, adj_t=adj)
        pos_test_pred = self.batch_predict(h, pos_test_edge, batch_size, adj_t=adj)
        neg_test_pred = self.batch_predict(h, neg_test_edge, batch_size, adj_t=adj)
        if eval_metric == 'hits':
            return evaluate_hits(evaluator, pos_valid_pred, neg_valid_pred, pos_test_pred, neg_test_pred)
        return evaluate_mrr(evaluator, pos_valid_pred, neg_valid_pred, pos_test_pred, neg_test_pred)

    def recommend(self, data, nodes, k, exclude=None, exclude_self=True, batch_size=None, candidates=None):
        """extension: the k most likely links of every query node among all nodes -> (ids int64 [Q, k], scores fp32
        [Q, k]) on the device.  ``exclude``: None, 'adj' (the stored rows of data.adj_t) or an int64 [E, 2] edge
        tensor of known links.  ``candidates``: an int64 tensor of node ids; only those are recommended.  On a
        row-partitioned model a collective call (every rank, same arguments, full result everywhere).  See
        plnlp_b200/recommend.py."""
        from . import recommend
        return recommend.recommend(self, data, nodes, k, exclude, exclude_self, batch_size, candidates)

    def rank_against_all(self, data, edges, exclude=None, exclude_self=True, batch_size=None, candidates=None):
        """extension: filtered full-ranking evaluation -> fp32 [P], the rank of every target among all nodes for
        its source (1 + (gt + ge) / 2; known links other than the target itself filtered out).  ``candidates``: rank
        among those node ids and the target instead.  Feed it to utils.full_rank_metrics.  On a row-partitioned model
        a collective call.  See plnlp_b200/recommend.py."""
        from . import recommend
        return recommend.rank_against_all(self, data, edges, exclude, exclude_self, batch_size, candidates)


def create_input_layer(num_nodes, num_node_feats, hidden_channels, use_node_feats=True,
                       train_node_emb=False, pretrain_emb=None):
    """model.py:229-249 -> (input width, embedding module or None)."""
    emb, width = None, 0
    pretrained = pretrain_emb is not None and pretrain_emb != ''
    if use_node_feats:
        width = num_node_feats
        if train_node_emb:
            emb = torch.nn.Embedding(num_nodes, hidden_channels)
        elif pretrained:
            emb = torch.nn.Embedding.from_pretrained(torch.load(pretrain_emb))
    else:
        emb = torch.nn.Embedding.from_pretrained(torch.load(pretrain_emb)) if pretrained \
            else torch.nn.Embedding(num_nodes, hidden_channels)
    if emb is not None:
        width += emb.weight.size(1)
    return width, emb


def create_gnn_layer(input_channels, hidden_channels, num_layers, dropout=0, encoder_name='SAGE'):
    """model.py:252-260"""
    name = encoder_name.upper()
    if name == 'GCN':
        return GCN(input_channels, hidden_channels, hidden_channels, num_layers, dropout)
    if name == 'WSAGE':
        return WSAGE(input_channels, hidden_channels, hidden_channels, num_layers, dropout)
    if name == 'TRANSFORMER':
        return Transformer(input_channels, hidden_channels, hidden_channels, num_layers, dropout)  # noqa: F405
    return SAGE(input_channels, hidden_channels, hidden_channels, num_layers, dropout)


def create_predictor_layer(hidden_channels, num_layers, dropout=0, predictor_name='MLP'):
    """model.py:263-276 (unknown names -> None, as in the reference), plus 'NCN'."""
    name = predictor_name.upper()
    if name == 'DOT':
        return DotPredictor()
    if name == 'MLP':
        return MLPPredictor(hidden_channels, hidden_channels, 1, num_layers, dropout)
    if name == 'BIL':
        return BilinearPredictor(hidden_channels)
    if name == 'MLPDOT':          # the reference passes hidden_channels = 1 here (model.py:271): kept as is
        return MLPDotPredictor(hidden_channels, 1, num_layers, dropout)
    if name == 'MLPBIL':
        return MLPBilPredictor(hidden_channels, 1, num_layers, dropout)
    if name == 'MLPCAT':
        return MLPCatPredictor(hidden_channels, hidden_channels, 1, num_layers, dropout)
    if name == 'NCN':             # extension: Neural Common Neighbour (layer.NCNPredictor)
        return NCNPredictor(hidden_channels, hidden_channels, 1, num_layers, dropout)
    return None


def adjust_lr(optimizer, decay_ratio, lr):
    """model.py:279-286: linear decay floored at 1e-4 * lr."""
    lr_ = max(lr * (1 - decay_ratio), lr * 0.0001)
    for group in optimizer.param_groups:
        group['lr'] = lr_
    return lr_

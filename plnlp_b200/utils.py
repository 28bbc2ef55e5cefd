"""Edge assembly, evaluation glue and graph normalisation with the reference's signatures
(/root/reference/plnlp/utils.py).  Ranking runs on the GPU (csrc/rank.cu)."""
from __future__ import annotations

import torch

from . import _ops
from .negative_sample import global_neg_sample, global_perm_neg_sample, local_neg_sample  # noqa: F401


def _on(t, device):
    return t if device is None or t.device == device else t.to(device, non_blocking=True)


def get_pos_neg_edges(split, split_edge, edge_index=None, num_nodes=None, neg_sampler_name=None,
                      num_neg=None, device=None):
    """utils.py:7-41.  ``device`` (extension): where the returned tensors live; training negatives
    are always generated on the GPU (the device of ``edge_index`` when ``device`` is None)."""
    if device is None and edge_index is not None and edge_index.is_cuda:
        device = edge_index.device
    train = split_edge['train']
    if 'edge' in train:
        pos_edge = _on(split_edge[split]['edge'], device)
    elif 'source_node' in train:
        source = _on(split_edge[split]['source_node'], device)
        target = _on(split_edge[split]['target_node'], device)
        pos_edge = torch.stack([source, target], dim=1)
    else:
        raise KeyError("split_edge['train'] has neither 'edge' nor 'source_node'")

    if split == 'train':
        if neg_sampler_name == 'local':
            neg_edge = local_neg_sample(pos_edge, num_nodes=num_nodes, num_neg=num_neg)
        elif neg_sampler_name == 'global':
            neg_edge = global_neg_sample(_on(edge_index, device), num_nodes=num_nodes,
                                         num_samples=pos_edge.size(0), num_neg=num_neg)
        else:  # the reference falls back to the perm-copy sampler here (utils.py:27-32)
            neg_edge = global_perm_neg_sample(edge_index, num_nodes=num_nodes,
                                              num_samples=pos_edge.size(0), num_neg=num_neg)
    else:
        if 'edge' in train:
            neg_edge = _on(split_edge[split]['edge_neg'], device)
        else:
            target_neg = _on(split_edge[split]['target_node_neg'], device)
            k = target_neg.size(1)
            neg_edge = torch.stack([source.repeat_interleave(k), target_neg.reshape(-1)], dim=1)
    return pos_edge, neg_edge


def hits_at_k(pos_pred, neg_pred, K):
    """ogb Evaluator._eval_hits: fraction of positives strictly above the K-th largest negative
    (1.0 when there are fewer than K negatives).  Returns a python float."""
    if neg_pred.numel() < K:
        return 1.0
    kth = _ops.kth_largest_raw(neg_pred, K)
    cnt = _ops.count_greater_raw(pos_pred, kth)
    return float(cnt.item()) / pos_pred.numel()


def mrr_list(pos_pred, neg_pred):
    """per-row reciprocal rank.  Without ties rank = 1 + #{neg > pos}, which is what ogb 1.3.2's argsort gives.
    Under exact ties (a collapsed model, relu outputs that are all zero) that argsort is implementation defined;
    the rank used here is the mean of the optimistic and the pessimistic one, 1 + (#{neg > pos} + #{neg >= pos}) / 2
    -- the rule of current ogb -- so a constant-score model reports MRR ~ 2/K, not 1."""
    gt, ge = _ops.mrr_counts_raw(pos_pred, neg_pred)
    return 1.0 / (0.5 * (gt.to(torch.float32) + ge.to(torch.float32)) + 1.0)


def _cuda_f32(t):
    if not t.is_cuda:
        t = t.cuda()
    return t.to(torch.float32)


def evaluate_hits(evaluator, pos_val_pred, neg_val_pred, pos_test_pred, neg_test_pred):
    """utils.py:44-60.  ``evaluator`` is accepted for signature compatibility; its K is still set so
    code inspecting it afterwards sees the reference's side effect."""
    pv, nv, pt, nt = map(_cuda_f32, (pos_val_pred, neg_val_pred, pos_test_pred, neg_test_pred))
    results = {}
    for K in [20, 50, 100]:
        if evaluator is not None:
            evaluator.K = K
        results[f'Hits@{K}'] = (hits_at_k(pv, nv, K), hits_at_k(pt, nt, K))
    return results


def evaluate_mrr(evaluator, pos_val_pred, neg_val_pred, pos_test_pred, neg_test_pred):
    """utils.py:63-80."""
    pv, nv, pt, nt = map(_cuda_f32, (pos_val_pred, neg_val_pred, pos_test_pred, neg_test_pred))
    nv = nv.reshape(pv.shape[0], -1)
    nt = nt.reshape(pt.shape[0], -1)
    return {'MRR': (mrr_list(pv, nv).mean().item(), mrr_list(pt, nt).mean().item())}


def full_rank_metrics(ranks, ks=(1, 3, 10, 20, 50, 100)):
    """MRR and Hits@K of full-ranking ranks (``BaseModel.rank_against_all``): mean of 1 / rank and the fraction of
    ranks <= K, computed on the GPU with one host read -> {'MRR': float, 'Hits@K': float, ...}"""
    r = _cuda_f32(ranks).reshape(-1)
    vals = torch.stack([r.reciprocal().mean()] + [(r <= K).to(torch.float32).mean() for K in ks]).tolist()
    out = {'MRR': vals[0]}
    out.update({f'Hits@{K}': v for K, v in zip(ks, vals[1:])})
    return out


def gcn_normalization(adj_t):
    """utils.py:83-89: D^-1/2 (A + I) D^-1/2 with inf -> 0, on whatever adjacency type is given
    (CSRGraph or torch_sparse.SparseTensor: only set_diag / sum / broadcast-mul are used)."""
    adj_t = adj_t.set_diag()
    from .graph import CSRGraph, sym_normalize
    if isinstance(adj_t, CSRGraph) and adj_t.device.type == "cuda" and adj_t.size(0) == adj_t.size(1):
        return sym_normalize(adj_t)                      # csrc/graph_build.cu: degree + scaling in one kernel pair
    deg = adj_t.sum(dim=1).to(torch.float)
    dis = deg.pow(-0.5)
    dis[dis == float('inf')] = 0
    return dis.view(-1, 1) * adj_t * dis.view(1, -1)


def adj_normalization(adj_t):
    """utils.py:92-97: row-normalise the adjacency, D^-1 A (main.py applies it for the WSAGE encoder, :179-180)."""
    deg = adj_t.sum(dim=1).to(torch.float)
    inv = deg.pow(-1)
    inv[inv == float('inf')] = 0
    return inv.view(-1, 1) * adj_t

"""CPU restatement of the cross-shard top-k merge (csrc/topk.cu, plnlp_topk_merge_f32), in the rules of
oracle/ranking.py: the k best of R per-shard (id, score) lists by score descending, then id ascending; -0 ties with
+0 (reported as +0); an entry with id < 0 or a non-finite score is dead; a row with fewer than k live entries ends in
(-1, -inf).  The ids are global, so merging the per-block top-k lists of a row gives the top-k of the whole row."""
import numpy as np
import torch


def merge_topk(ids, scores, k):
    """ids int64 / scores [R, Q, k_in] (per-shard lists, rank-major) -> (ids int64 [Q, k], scores [Q, k])"""
    ids = torch.as_tensor(ids).cpu().numpy()
    sc = torch.as_tensor(scores).cpu().numpy()
    _, Q, _ = ids.shape
    out_i = np.full((Q, k), -1, dtype=np.int64)
    out_s = np.full((Q, k), -np.inf, dtype=sc.dtype)
    for q in range(Q):
        i, v = ids[:, q].reshape(-1), sc[:, q].reshape(-1)
        live = (i >= 0) & np.isfinite(v)
        i, v = i[live], v[live]
        v = np.where(v == 0, np.zeros_like(v), v)
        order = np.lexsort((i, -v))[:k]
        out_i[q, :order.size] = i[order]
        out_s[q, :order.size] = v[order]
    return torch.from_numpy(out_i), torch.from_numpy(out_s)

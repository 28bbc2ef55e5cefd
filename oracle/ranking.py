"""CPU restatement of link recommendation over all nodes (plnlp_b200/recommend.py, csrc/topk.cu).

Rules restated here:
  * known-link mask: s[q, j] = -inf for every j in row nodes[q] of the exclude CSR (columns outside [0, N)
    ignored) and, with exclude_self, for j = nodes[q];
  * top-k: the k largest FINITE entries of a row (NaN and +-inf are never candidates) by score descending, then
    column ascending; -0 ties with +0 (reported as +0); a row with fewer than k candidates ends in (-1, -inf);
  * filtered rank counts: gt / ge = #{j != target, s_j finite, s_j > / >= target_score}.
Works on float32 or float64 scores (the comparison happens in the given dtype).
"""
import numpy as np
import torch


def mask_scores(s, nodes, rowptr=None, col=None, exclude_self=True):
    """copy of s [Q, N] with the known links of nodes[q] (and nodes[q] itself) set to -inf"""
    s = s.clone()
    N = s.size(1)
    for q, n in enumerate(torch.as_tensor(nodes).tolist()):
        if rowptr is not None:
            c = torch.as_tensor(col[int(rowptr[n]):int(rowptr[n + 1])]).to(torch.int64)
            c = c[(c >= 0) & (c < N)]
            s[q, c] = float("-inf")
        if exclude_self and 0 <= n < N:
            s[q, n] = float("-inf")
    return s


def topk_rows(s, k):
    """-> (ids int64 [Q, k], scores [Q, k] in s's dtype)"""
    a = s.detach().cpu().numpy()
    Q = a.shape[0]
    ids = np.full((Q, k), -1, dtype=np.int64)
    sc = np.full((Q, k), -np.inf, dtype=a.dtype)
    for q in range(Q):
        row = a[q]
        col = np.flatnonzero(np.isfinite(row))
        v = row[col]
        v = np.where(v == 0, np.zeros_like(v), v)          # -0 -> +0
        if col.size > k:                                    # keep the k largest values and everything tied with them
            thresh = np.partition(v, col.size - k)[col.size - k]
            keep = v >= thresh
            col, v = col[keep], v[keep]
        order = np.lexsort((col, -v))[:k]                   # primary: score descending; then column ascending
        ids[q, :order.size] = col[order]
        sc[q, :order.size] = v[order]
    return torch.from_numpy(ids), torch.from_numpy(sc)


def rank_counts(s, target, target_score):
    """-> (gt int32 [Q], ge int32 [Q])"""
    a = s.detach().cpu().numpy()
    t = torch.as_tensor(target).cpu().numpy()
    ts = torch.as_tensor(target_score).cpu().numpy().astype(a.dtype)
    Q, N = a.shape
    fin = np.isfinite(a) & (np.arange(N)[None, :] != t[:, None])
    gt = ((a > ts[:, None]) & fin).sum(1)
    ge = ((a >= ts[:, None]) & fin).sum(1)
    return torch.from_numpy(gt.astype(np.int32)), torch.from_numpy(ge.astype(np.int32))


def filtered_ranks(S, targets, nodes, rowptr=None, col=None, exclude_self=True):
    """1 + (gt + ge) / 2 of each target on full score rows S [P, N] (row p = source nodes[p]): the target score is
    read before masking, so the target is never excluded"""
    t = torch.as_tensor(targets)
    ts = S[torch.arange(S.size(0)), t]
    gt, ge = rank_counts(mask_scores(S, nodes, rowptr, col, exclude_self), t, ts)
    return 1.0 + 0.5 * (gt.double() + ge.double())

"""CPU restatement of the path-based link scores (plnlp_b200/paths.py, csrc/propagate.cu), in two forms.

Rules restated here:
  * N(u) and d(w) = |N(w)| as in oracle/heuristics.py (distinct columns of stored row u without u; values ignored);
    R(j) = {w : j in N(w)};
  * one hop of the state column x of a source u: y[j] = fp32(c * s_j + b * [j == u]), s_j = sum over w in R(j) of
    wt(w) * x[w];
  * Katz(beta, L): wt = 1, c = beta, L hops from x = e_u with b = 1 on hops 1 .. L-1 and b = 0 on hop L;
  * PPR(alpha, T): wt(w) = 1 / d(w) (0 when d(w) = 0), c = 1 - alpha, b = alpha, T hops from x = e_u;
  * the score of (u, v) is x[v] of u's column.

``*_fp64``: the truncated series in fp64 with scipy (no rounding to fp32).  ``propagate_exact``: the hop rule as the
kernel computes it, bit for bit -- fp64 products and sums, R(j) in ascending w cut into items of PROP_CHUNK entries,
each item summed in order from +0, the item partials added in order, one rounding to fp32 per hop.
"""
import numpy as np
import scipy.sparse as sp

from oracle.heuristics import neighbour_sets

PROP_CHUNK = 256


def reach_lists(sets):
    """[sorted list of w] per node j: R(j) = {w : j in N(w)}"""
    R = [[] for _ in sets]
    for w, s in enumerate(sets):
        for j in s:
            R[j].append(w)
    return [sorted(r) for r in R]


def walk_matrix(sets):
    """scipy CSR fp64 A [n, n]: A[w, j] = 1 for j in N(w)"""
    n = len(sets)
    rows = [w for w, s in enumerate(sets) for _ in s]
    cols = [j for s in sets for j in sorted(s)]
    return sp.csr_matrix((np.ones(len(rows)), (rows, cols)), shape=(n, n))


def inv_degree(sets):
    """fp64 [n]: 1 / d(w), 0 when d(w) = 0"""
    d = np.array([len(s) for s in sets], dtype=np.float64)
    return np.where(d > 0, 1.0 / np.maximum(d, 1.0), 0.0)


def hops(method, beta=0.005, L=3, alpha=0.15, T=30):
    """[(c, b, weighted)] per hop"""
    if method == "Katz":
        return [(beta, 1.0 if h < L else 0.0, False) for h in range(1, L + 1)]
    return [(1.0 - alpha, alpha, True)] * T


def katz_fp64(sets, sources, beta=0.005, L=3):
    """fp64 [len(sources), n]: row a = sum over l = 1 .. L of beta^l (A^l)[sources[a], :]"""
    A = walk_matrix(sets)
    n = len(sets)
    X = sp.csr_matrix((np.ones(len(sources)), (np.arange(len(sources)), sources)), shape=(len(sources), n))
    out = np.zeros((len(sources), n))
    for l in range(1, L + 1):
        X = X @ A
        out += beta ** l * X.toarray()
    return out


def ppr_fp64(sets, sources, alpha=0.15, T=30):
    """fp64 [len(sources), n]: T iterations r <- (1 - alpha) r P + alpha e_u from r = e_u, P = D^-1 A"""
    P = sp.diags(inv_degree(sets)) @ walk_matrix(sets)
    E = np.zeros((len(sources), len(sets)))
    E[np.arange(len(sources)), sources] = 1.0
    X = E.copy()
    for _ in range(T):
        X = (1.0 - alpha) * (P.T @ X.T).T + alpha * E
    return X


def dense_power(sets, sources, method, beta=0.005, L=3, alpha=0.15, T=30):
    """the same series from dense matrix powers (tiny graphs)"""
    A = walk_matrix(sets).toarray()
    if method == "Katz":
        S = sum(beta ** l * np.linalg.matrix_power(A, l) for l in range(1, L + 1))
    else:
        M = (1.0 - alpha) * (np.diag(inv_degree(sets)) @ A)
        S = sum(alpha * np.linalg.matrix_power(M, t) for t in range(T)) + np.linalg.matrix_power(M, T)
    return S[np.asarray(sources)]


def hop_exact(R, weight, x, src, c, b, lo=0, hi=None):
    """fp32 [hi - lo, B]: one hop of the rows [lo, hi) from the fp32 state x [n, B] (R: ``reach_lists``; weight fp64
    [n] or None; src int64 [B], -1 padding), in the kernel's order"""
    hi = len(R) if hi is None else hi
    x = np.asarray(x, dtype=np.float32)
    src = np.asarray(src)
    B = x.shape[1]
    y = np.empty((hi - lo, B), dtype=np.float32)
    for j in range(lo, hi):
        r = R[j]
        s = np.zeros(B)
        for a in range(0, len(r), PROP_CHUNK):
            acc = np.zeros(B)
            for w in r[a:a + PROP_CHUNK]:
                t = x[w].astype(np.float64)
                acc = acc + (t if weight is None else weight[w] * t)
            s = s + acc
        y[j - lo] = (c * s + np.where(src == j, b, 0.0)).astype(np.float32)
    return y


def propagate_exact(sets, sources, method, **params):
    """fp32 [n, B]: the final state of the sources (int64 [B], -1 padding), bit for bit as the kernel computes it"""
    n = len(sets)
    R = reach_lists(sets)
    src = np.asarray(sources)
    x = np.zeros((n, src.size), dtype=np.float32)
    a = np.flatnonzero(src >= 0)
    x[src[a], a] = 1.0
    inv = inv_degree(sets)
    for c, b, weighted in hops(method, **params):
        x = hop_exact(R, inv if weighted else None, x, src, c, b)
    return x


def sets_of(adj):
    """``neighbour_sets`` of a CSRGraph / SparseTensor"""
    rowptr, col, _ = adj.csr()
    return neighbour_sets(rowptr.cpu(), col.cpu(), adj.size(0))

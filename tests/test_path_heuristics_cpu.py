"""CPU tests (-m "not gpu") of the path-based link scores Katz and PPR (plnlp_b200/paths.py): the exact restatement of
the hop rule (tests/path_oracle.py) against the fp64 series and the series against dense matrix powers, argument
validation, the grouping of sources into blocks and the readout positions, per-rank hop steps that add up to the
whole for R = 1, 2, 3, the one-GPU calls with the kernel swapped for the restatement, and a 2-rank gloo run of the
collective calls."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import ranking
from tests import path_oracle as po
from tests.ranking_merge import merge_topk
from tests.test_heuristics_cpu import _csr, _graph, ref_clean
from tests.test_heuristics_recommend_cpu import ref_mask, ref_topk

PARAMS = {"Katz": dict(beta=0.05, L=3), "PPR": dict(alpha=0.2, T=12)}


def method_obj(m):
    from plnlp_b200 import heuristics
    p = PARAMS[m]
    return heuristics.Katz(p["beta"], p["L"]) if m == "Katz" else heuristics.PPR(p["alpha"], p["T"])


def ref_hop(shard, x, live, src, c, b, weight):
    """CPU restatement of _ops.propagate_raw for a ``paths.PathShard`` (its own reach rows, as the kernel walks them)"""
    rowptr, col = shard.rowptr.tolist(), shard.col.tolist()
    rows = shard.hi - shard.lo
    R = [None] * shard.lo + [col[rowptr[i]:rowptr[i + 1]] for i in range(rows)]
    xn = x.numpy()
    if live is not None:                                     # the promise the live map makes
        assert not xn[:shard.n][live.numpy()[:shard.n] == 0].any()
    y = po.hop_exact(R, None if weight is None else weight.numpy(), xn, src.numpy(), c, b, shard.lo, shard.hi)
    return torch.from_numpy(y), torch.from_numpy((y != 0).any(1).astype(np.uint8))


@pytest.fixture
def ref_ops(monkeypatch):
    from plnlp_b200 import _ops, heuristics, paths
    monkeypatch.setattr(paths, "_hop_gpu", ref_hop)
    monkeypatch.setattr(heuristics, "clean_csr", ref_clean)
    for name, fn in (("score_mask_raw", ref_mask), ("topk_rows_raw", ref_topk), ("topk_merge_raw", merge_topk)):
        monkeypatch.setattr(_ops, name, fn)


@pytest.mark.parametrize("symmetric", [True, False])
@pytest.mark.parametrize("method", ["Katz", "PPR"])
def test_exact_form_matches_fp64_series(method, symmetric):
    n = 600
    src, dst = _graph(n, 1500, 5, symmetric=symmetric)
    src, dst = torch.cat([src, torch.arange(1, n, 2)]), torch.cat([dst, torch.full((n // 2,), 3)])   # R(3): a hub
    adj = _csr(src, dst, n)
    sets = po.sets_of(adj)
    assert max(len(r) for r in po.reach_lists(sets)) > po.PROP_CHUNK          # a hub row split into items
    srcs = np.array([0, 1, 7, 150, 599, 42, 3])
    p = PARAMS[method]
    ref = po.katz_fp64(sets, srcs, p["beta"], p["L"]) if method == "Katz" else po.ppr_fp64(sets, srcs, p["alpha"],
                                                                                           p["T"])
    got = po.propagate_exact(sets, srcs, method, **p).T.astype(np.float64)
    assert np.all(np.abs(got - ref) <= 1e-6 * np.abs(ref) + 1e-12)
    assert np.array_equal(got > 0, ref > 0)


@pytest.mark.parametrize("method", ["Katz", "PPR"])
def test_fp64_series_matches_dense_powers(method):
    for n, seed, sym in ((12, 1, True), (15, 2, False), (9, 3, False)):
        sets = po.sets_of(_csr(*_graph(n, 3 * n, seed, symmetric=sym), n))
        srcs = np.arange(n)
        for kw in ({}, PARAMS[method], dict(beta=0.3, L=1) if method == "Katz" else dict(alpha=0.5, T=1)):
            full = {**(dict(beta=0.005, L=3) if method == "Katz" else dict(alpha=0.15, T=30)), **kw}
            ser = po.katz_fp64(sets, srcs, full["beta"], full["L"]) if method == "Katz" else \
                po.ppr_fp64(sets, srcs, full["alpha"], full["T"])
            assert np.allclose(ser, po.dense_power(sets, srcs, method, **full), rtol=1e-12, atol=1e-15)


def test_parameters_and_method_parsing():
    from plnlp_b200 import heuristics, paths
    assert heuristics.path_method("Katz") == heuristics.Katz(0.005, 3)
    assert heuristics.path_method("PPR") == heuristics.PPR(0.15, 30)
    k = heuristics.Katz(beta=0.01, hops=2)
    assert heuristics.path_method(k) is k
    for m in ("CN", "AA", "RA", "Jaccard", "katz", None):
        assert heuristics.path_method(m) is None
    assert heuristics.METHODS == ("CN", "AA", "RA") and heuristics.PATH_METHODS == ("Katz", "PPR")
    for bad in (dict(beta=0.0), dict(beta=-1.0), dict(beta=float("inf")), dict(beta=float("nan")), dict(beta="1"),
                dict(beta=True), dict(hops=0), dict(hops=heuristics.MAX_KATZ_HOPS + 1), dict(hops=2.0),
                dict(hops=True)):
        with pytest.raises(ValueError):
            heuristics.Katz(**bad)
    for bad in (dict(alpha=0.0), dict(alpha=1.0), dict(alpha=-0.1), dict(alpha=float("nan")), dict(iters=0),
                dict(iters=heuristics.MAX_PPR_ITERS + 1), dict(iters=1.5)):
        with pytest.raises(ValueError):
            heuristics.PPR(**bad)
    assert heuristics.Katz(hops=heuristics.MAX_KATZ_HOPS).hops == heuristics.MAX_KATZ_HOPS
    assert heuristics.PPR(iters=np.int64(3)).iters == 3 and type(heuristics.PPR(iters=np.int64(3)).iters) is int
    with pytest.raises(Exception):
        k.beta = 1.0                                                      # frozen
    # hop schedules
    assert paths.hops(heuristics.Katz(0.1, 3)) == [(0.1, 1.0, False), (0.1, 1.0, False), (0.1, 0.0, False)]
    assert paths.hops(heuristics.Katz(0.1, 1)) == [(0.1, 0.0, False)]
    assert paths.hops(heuristics.PPR(0.25, 2)) == [(0.75, 0.25, True)] * 2
    # the words the ranks compare change with every parameter
    words = [paths.agree_params(m) for m in (heuristics.Katz(), heuristics.Katz(0.006), heuristics.Katz(hops=4),
                                             heuristics.PPR(), heuristics.PPR(0.2), heuristics.PPR(iters=31))]
    assert len({tuple(w) for w in words}) == len(words)
    assert paths.agree_params(heuristics.Katz()) == paths.agree_params(heuristics.path_method("Katz"))


def test_invalid_methods_still_raise():
    from plnlp_b200 import heuristics
    n = 20
    adj = _csr(*_graph(n, 50, 1), n)
    e = torch.zeros(3, 2, dtype=torch.int64)
    for m in ("Jaccard", "jaccard", "katz", "ppr", 3):
        with pytest.raises(ValueError):
            heuristics.score_edges(adj, e, m)
        with pytest.raises(ValueError):
            heuristics.recommend(adj, torch.tensor([0]), 2, m)
        with pytest.raises(ValueError):
            heuristics.rank_against_all(adj, e, m)


def test_block_width():
    from plnlp_b200 import paths
    assert [paths.block_width(b, 0) for b in (1, 31, 32, 33, 64, 100, 256, 257, 10 ** 6)] == \
        [32, 32, 32, 64, 64, 128, 256, 256, 256]
    assert [paths.block_width(b, 0) for b in (65, 129, 200, 224)] == [128, 256, 256, 256]   # kernel widths only
    for bad in (-1, -32):
        with pytest.raises(ValueError):
            paths.block_width(bad, 0)
    n = 2927963                                              # citation2 shape: the budget holds B = 256 ...
    assert paths.block_width(None, paths.column_bytes(n, 0)) == 256
    assert paths.block_width(None, paths.column_bytes(n, n)) == 128          # 224 would fit: the next width down
    assert paths.block_width(None, 1 << 40) == 32            # ... and never drops below one warp of columns
    assert 2 * 4 * n * 256 < 6.1e9                           # two fp32 [N, 256] states


@pytest.mark.parametrize("B", [32, 64])
def test_source_blocks_and_readout_positions(B):
    from plnlp_b200 import paths
    g = torch.Generator().manual_seed(3)
    u = torch.randint(0, 500, (700,), generator=g)
    blocks = paths.source_blocks(u, B)
    us = torch.unique(u)
    assert torch.equal(torch.cat([s for s, _, _ in blocks]), us)          # distinct, ascending
    assert all(s.numel() == B for s, _, _ in blocks[:-1]) and 0 < blocks[-1][0].numel() <= B
    seen = torch.cat([sel for _, sel, _ in blocks])
    assert torch.equal(torch.sort(seen).values, torch.arange(u.numel()))  # every pair exactly once
    for s, sel, col in blocks:
        assert torch.equal(s[col], u[sel])                                # the column that holds the pair's source
    assert paths.source_blocks(torch.zeros(0, dtype=torch.int64), B) == []
    p = paths.padded(torch.tensor([5, 2]), 32)
    assert p.numel() == 32 and p[:2].tolist() == [5, 2] and (p[2:] == -1).all()


def _shards(adj, n, R, inv=None):
    from plnlp_b200 import parallel, paths
    from plnlp_b200.graph import CSRGraph
    out = []
    for r in range(R):
        lo, hi = parallel.row_block(n, r, R)
        sadj = parallel.shard_graph(adj, r, R, CSRGraph)
        rowptr, col, deg = paths.reach_rows(sadj.local, sadj.local_t, lo, hi, n, clean=ref_clean)
        out.append((paths.PathShard(rowptr, col, lo, hi, n, sadj.blk, inv, op=ref_hop), deg))
    return out


@pytest.mark.parametrize("method", ["Katz", "PPR"])
@pytest.mark.parametrize("n,symmetric", [(31, True), (29, False), (4, True)])   # n = 4, R = 3: an empty last block
def test_rank_hops_add_up_to_the_whole(method, n, symmetric):
    from plnlp_b200 import paths
    from plnlp_b200.heuristics import weight_table
    adj = _csr(*_graph(n, 4 * n, 9, symmetric=symmetric), n)
    sets = po.sets_of(adj)
    src = paths.padded(torch.tensor([0, n - 1, 1, 0]), 32)
    want = po.propagate_exact(sets, src.numpy(), method, **PARAMS[method])
    for R in (1, 2, 3):
        shards = _shards(adj, n, R)
        deg = torch.cat([torch.cat([d, d.new_zeros(sh.blk - d.numel())]) for sh, d in shards])
        assert deg[:n].tolist() == [len(s) for s in sets]                     # d(j) from the rank's own rows
        inv = weight_table(deg, "RA")[:n]
        for sh, _ in shards:
            assert [sh.col[sh.rowptr[i]:sh.rowptr[i + 1]].tolist() for i in range(sh.hi - sh.lo)] == \
                po.reach_lists(sets)[sh.lo:sh.hi]
            sh.inv_deg = inv
        blocks = [sh.start(src) for sh, _ in shards]
        for c, b, weighted in paths.hops(method_obj(method)):
            xf = torch.cat([x for x, _ in blocks])
            lf = torch.cat([lv for _, lv in blocks])
            blocks = [sh.hop(xf, lf, src, c, b, weighted) for sh, _ in shards]
        got = torch.cat([x for x, _ in blocks])[:n].numpy()
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), R
        live = torch.cat([lv for _, lv in blocks])[:n].numpy()
        assert np.array_equal(live.astype(bool), (want != 0).any(1))


def _oracle_scores(adj, n, method, sources):
    return po.propagate_exact(po.sets_of(adj), np.asarray(sources), method, **PARAMS[method])


def _oracle_calls(adj, n, method, nodes, edges, k, exclude, cand):
    """(ids, scores, ranks) of recommend / rank_against_all from the restatement's score rows (oracle/ranking.py)"""
    keep = torch.ones(n, dtype=torch.bool)
    if cand is not None:
        keep[:] = False
        keep[cand] = True
    er = ec = None
    if exclude is not None:
        er = torch.zeros(n + 1, dtype=torch.int64)
        er[1:] = torch.cumsum(torch.bincount(exclude[:, 0], minlength=n), 0)
        ec = exclude[torch.argsort(exclude[:, 0], stable=True), 1]
    S = torch.from_numpy(_oracle_scores(adj, n, method, nodes).T.copy())
    Sm = ranking.mask_scores(S, nodes, er, ec, True)
    Sm[:, ~keep] = float("-inf")
    ids, sc = ranking.topk_rows(Sm, k)
    St = torch.from_numpy(_oracle_scores(adj, n, method, edges[:, 0]).T.copy())
    t = edges[:, 1]
    ts = St[torch.arange(t.numel()), t]
    Sr = ranking.mask_scores(St, edges[:, 0], er, ec, True)
    drop = ~keep[None, :].expand_as(Sr).clone()
    drop[torch.arange(t.numel()), t] = False
    Sr[drop] = float("-inf")
    gt, ge = ranking.rank_counts(Sr, t, ts)
    return ids, sc, (1.0 + 0.5 * (gt.double() + ge.double())).float()


N_CALLS = 37


def _call_args():
    src, dst = _graph(N_CALLS, 120, 11, symmetric=False)
    g = torch.Generator().manual_seed(13)
    nodes = torch.randint(0, N_CALLS, (40,), generator=g)
    edges = torch.stack([nodes, torch.randint(0, N_CALLS, (40,), generator=g)], 1)
    exclude = torch.randint(0, N_CALLS, (40, 2), generator=g)
    cand = torch.tensor([3, 30, 1, 17, 17, 22, 36, 8])
    return _csr(src, dst, N_CALLS), nodes, edges, exclude, cand


@pytest.mark.parametrize("method", ["Katz", "PPR"])
def test_one_gpu_calls_with_reference_hop(ref_ops, method):
    from plnlp_b200 import heuristics
    adj, nodes, edges, exclude, cand = _call_args()
    m = method_obj(method)
    S = _oracle_scores(adj, N_CALLS, method, edges[:, 0])
    want = torch.from_numpy(S[edges[:, 1].numpy(), np.arange(edges.size(0))])
    for bs in (None, 1, 33):
        assert torch.equal(heuristics.score_edges(adj, edges, m, bs), want), bs
    for ex in (None, exclude):
        for c in (None, cand):
            ids, sc, ranks = _oracle_calls(adj, N_CALLS, method, nodes, edges, 6, ex, c)
            gi, gs = heuristics.recommend(adj, nodes, 6, m, ex, True, 33, c)
            assert torch.equal(gi, ids) and torch.equal(gs, sc), (ex is None, c is None)
            assert torch.equal(heuristics.rank_against_all(adj, edges, m, ex, True, 33, c), ranks)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, ws, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=ws)
    try:
        from plnlp_b200 import _ops, heuristics, parallel, paths
        from plnlp_b200.graph import CSRGraph
        heuristics.clean_csr = ref_clean                  # this process only
        paths._hop_gpu = ref_hop
        _ops.score_mask_raw, _ops.topk_rows_raw, _ops.topk_merge_raw = ref_mask, ref_topk, merge_topk
        real_gather = dist.all_gather_into_tensor

        def flat_gather(out, inp, group=None, async_op=False):   # gloo wants the outputs flat
            return real_gather(out.view(-1), inp.reshape(-1), group=group, async_op=async_op)
        dist.all_gather_into_tensor = flat_gather
        adj, nodes, edges, exclude, cand = _call_args()
        sadj = parallel.shard_graph(adj, rank, ws, CSRGraph)
        out = {}
        for m in ("Katz", "PPR"):
            mo = method_obj(m)
            out[(m, "score")] = heuristics.score_edges(sadj, edges, mo, 33)
            for ex in (None, exclude):
                for c in (None, cand):
                    out[(m, ex is not None, c is not None)] = (heuristics.recommend(sadj, nodes, 6, mo, ex, True, 33, c),
                                                               heuristics.rank_against_all(sadj, edges, mo, ex, True,
                                                                                           33, c))
        errors = []
        for bad in (heuristics.Katz(0.05 if rank == 0 else 0.06, 3), heuristics.PPR(0.2, 12 + rank),
                    "Katz" if rank == 0 else "CN"):
            try:
                heuristics.recommend(sadj, nodes, 5, bad)
                errors.append(None)
            except ValueError as e:
                errors.append(str(e))
            try:
                heuristics.score_edges(sadj, edges, bad)
                errors.append(None)
            except ValueError as e:
                errors.append(str(e))
        out["errors"] = errors
        ret[rank] = out
    finally:
        dist.destroy_process_group()


def test_collective_calls_gloo():
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(2, _free_port(), ret), nprocs=2, join=True)
    adj, nodes, edges, exclude, cand = _call_args()
    for m in ("Katz", "PPR"):
        S = _oracle_scores(adj, N_CALLS, m, edges[:, 0])
        want = torch.from_numpy(S[edges[:, 1].numpy(), np.arange(edges.size(0))])
        for r in range(2):
            assert torch.equal(ret[r][(m, "score")], want), (m, r)
        for ex in (False, True):
            for c in (False, True):
                ids, sc, ranks = _oracle_calls(adj, N_CALLS, m, nodes, edges, 6, exclude if ex else None,
                                               cand if c else None)
                for r in range(2):
                    (gi, gs), gr = ret[r][(m, ex, c)]
                    assert torch.equal(gi, ids) and torch.equal(gs, sc), (m, ex, c, r)
                    assert torch.equal(gr, ranks), (m, ex, c, r)
    for r in range(2):
        assert all(e is not None and "collective" in e for e in ret[r]["errors"]), ret[r]["errors"]

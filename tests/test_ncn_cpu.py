"""CPU tests (-m "not gpu") of the NCN predictor's host side: the list rules of tests/ncn_oracle.py against their
dense restatement and the fp64 head against its concatenation, the union / renumber helper of the restricted last
conv (model.ncn_restrict), the argument checks of heuristics.common_neighbour_lists and the predictor factory."""
import pytest
import torch

from tests import ncn_oracle as no


def _sets(n, m, seed):
    g = torch.Generator().manual_seed(seed)
    src, dst = torch.randint(0, n - 3, (m,), generator=g), torch.randint(0, n - 3, (m,), generator=g)
    sets = [set() for _ in range(n)]                 # the last 3 nodes isolated
    for a, b in zip(src.tolist(), dst.tolist()):
        if a != b:
            sets[a].add(b)
            if seed % 2 == 0:                        # even seeds symmetric, odd seeds not
                sets[b].add(a)
    return sets


def _pairs(n, P, seed):
    g = torch.Generator().manual_seed(seed)
    e = torch.randint(0, n, (P, 2), generator=g)
    e[:5, 1] = e[:5, 0]                              # (u, u)
    e[5:8, 0] = -1                                   # the mean row
    e[8:10, 1] = n - 1                               # isolated
    return e


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_oracle_lists_match_dense_restatement(seed):
    n = 40
    sets = _sets(n, 200, seed)
    e = _pairs(n, 300, seed)
    rowptr, col = no.lists(sets, e)
    drowptr, dcol = no.dense_lists(sets, e)
    assert torch.equal(rowptr, drowptr) and torch.equal(col, dcol)
    for p, (u, v) in enumerate(e.tolist()):
        got = col[rowptr[p]:rowptr[p + 1]].tolist()
        assert got == sorted(got)
        assert u not in got or u < 0                 # u is never its own common neighbour
        if u < 0 or v < 0:
            assert got == []
        if u == v and u >= 0:
            assert got == sorted(sets[u])
    assert int(rowptr[-1]) > 0


@pytest.mark.parametrize("L", [1, 2, 3])
def test_oracle_head_is_the_mlp_on_the_concatenation(L):
    torch.manual_seed(L)
    n, H, hid = 30, 6, 5
    sets = _sets(n, 150, 4)
    e = _pairs(n, 50, 5)
    cn = no.lists(sets, e)
    h = torch.randn(n + 1, H, dtype=torch.float64, requires_grad=True)
    dims = [2 * H] + [hid] * (L - 1) + [1]
    lins = [(torch.randn(dims[i + 1], dims[i], dtype=torch.float64, requires_grad=True),
             torch.randn(dims[i + 1], dtype=torch.float64, requires_grad=True)) for i in range(L)]
    s = no.score(h, e, cn, lins)
    # restatement: the dense 0/1 matrix of the lists times h, concatenated explicitly
    C = torch.zeros(e.size(0), n + 1, dtype=torch.float64)
    rowptr, col = cn
    for p in range(e.size(0)):
        C[p, col[rowptr[p]:rowptr[p + 1]]] = 1.0
    x = torch.cat([h[e[:, 0]] * h[e[:, 1]], C @ h], 1)
    for W, b in lins[:-1]:
        x = torch.relu(x @ W.t() + b)
    ref = (x @ lins[-1][0].t() + lins[-1][1]).reshape(-1)
    assert torch.allclose(s, ref, rtol=1e-12, atol=1e-12)
    gs = torch.autograd.grad(s.square().sum(), [h] + [t for wb in lins for t in wb])
    gr = torch.autograd.grad(ref.square().sum(), [h] + [t for wb in lins for t in wb])
    for a, b in zip(gs, gr):
        assert torch.allclose(a, b, rtol=1e-10, atol=1e-10)


def test_ncn_restrict_renumbers_to_the_same_nodes():
    from plnlp_b200.model import ncn_restrict
    edges = torch.tensor([[7, 3], [3, 7], [100, 2], [5, 5]])
    rowptr = torch.tensor([0, 2, 4, 4, 6])
    col = torch.tensor([1, 9, 1, 9, 40, 6])
    ids, e2, (r2, c2) = ncn_restrict(edges, (rowptr, col))
    assert ids.tolist() == [1, 2, 3, 5, 6, 7, 9, 40, 100]
    assert torch.equal(ids[e2], edges) and torch.equal(ids[c2], col) and r2 is rowptr
    # no common neighbours at all: the union is the endpoint set
    ids, e2, (_, c2) = ncn_restrict(edges, (torch.zeros(5, dtype=torch.int64), torch.empty(0, dtype=torch.int64)))
    assert ids.tolist() == [2, 3, 5, 7, 100] and torch.equal(ids[e2], edges) and c2.numel() == 0
    # random batches
    g = torch.Generator().manual_seed(0)
    for _ in range(5):
        edges = torch.randint(0, 1000, (64, 2), generator=g)
        col = torch.randint(0, 1000, (300,), generator=g)
        ids, e2, (_, c2) = ncn_restrict(edges, (None, col))
        assert torch.equal(ids, torch.unique(torch.cat([edges.reshape(-1), col])))
        assert torch.equal(ids[e2], edges) and torch.equal(ids[c2], col)


def test_common_neighbour_lists_argument_checks():
    from plnlp_b200 import heuristics, parallel
    from plnlp_b200.graph import CSRGraph
    adj = CSRGraph(torch.tensor([0, 1, 2, 2]), torch.tensor([1, 0]), None, (3, 3))
    bad = [torch.tensor([[0, 1]], dtype=torch.int32),                     # dtype
           torch.tensor([0, 1]),                                          # shape
           torch.tensor([[0, 1, 2]]),
           torch.tensor([[0, 3]]),                                        # out of range
           torch.tensor([[-2, 0]])]
    for e in bad:
        with pytest.raises(ValueError):
            heuristics.common_neighbour_lists(adj, e)
    with pytest.raises(ValueError):                                       # not square
        heuristics.common_neighbour_lists(CSRGraph(torch.tensor([0, 1, 2]), torch.tensor([1, 2]), None, (2, 3)),
                                          torch.tensor([[0, 1]]))
    with pytest.raises(NotImplementedError):
        heuristics.common_neighbour_lists(object.__new__(parallel.ShardedAdj), torch.tensor([[0, 1]]))


@pytest.mark.parametrize("L", [1, 2, 3])
def test_create_predictor_layer_ncn(L):
    from plnlp_b200.layer import NCNPredictor
    from plnlp_b200.model import create_predictor_layer
    H = 16
    m = create_predictor_layer(H, L, 0.3, "NCN")
    assert isinstance(m, NCNPredictor) and m.dropout == 0.3
    dims = [2 * H] + [H] * (L - 1) + [1]
    shapes = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    want = {}
    for i in range(L):
        want[f"lins.{i}.weight"] = (dims[i + 1], dims[i])
        want[f"lins.{i}.bias"] = (dims[i + 1],)
    assert shapes == want
    assert [tuple(p.shape) for p in m.flat_params()] == [want[f"lins.{i}.{k}"] for i in range(L)
                                                          for k in ("weight", "bias")]
    assert create_predictor_layer(H, L, 0.0, "ncn").__class__ is NCNPredictor
    with pytest.raises(TypeError, match="score_edges"):
        m(torch.zeros(2, H), torch.zeros(2, H))


def test_unknown_predictor_names_still_none():
    from plnlp_b200.layer import MLPPredictor
    from plnlp_b200.model import create_predictor_layer
    for name in ("NCNC", "XYZ", "", "N C N"):
        assert create_predictor_layer(8, 2, 0.0, name) is None
    assert isinstance(create_predictor_layer(8, 2, 0.0, "MLP"), MLPPredictor)

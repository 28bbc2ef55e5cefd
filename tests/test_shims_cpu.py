"""CPU tests (-m "not gpu") of plnlp_b200/shims.py (SURVEY.md 8f rank 4): the stand-ins for the third-party calls
of the reference's main.py against the oracle's restatement of the same calls."""
import pytest
import torch

from oracle import sparse
from plnlp_b200 import shims


def test_to_sparse_tensor_and_constructor_match_oracle():
    g = torch.Generator().manual_seed(1)
    N, E = 50, 400
    ei = torch.randint(0, N, (2, E), generator=g)             # duplicates and self loops included
    w = torch.rand(E, generator=g)
    data = shims.ToSparseTensor()(shims.Data(edge_index=ei.clone(), edge_weight=w.clone(), num_nodes=N, x=None))
    assert not hasattr(data, "edge_index") and not hasattr(data, "edge_weight")
    want = sparse.to_sparse_tensor(ei, w, N)
    for a, b in zip(data.adj_t.csr(), want.csr()):
        assert torch.equal(a, b)
    # SparseTensor(row=, col=, value=) as main.py:124-126 builds it
    adj = shims.SparseTensor(row=ei[0], col=ei[1], value=w, sparse_sizes=(N, N))
    want = sparse.SparseTensor(row=ei[0], col=ei[1], value=w, sparse_sizes=(N, N))
    for a, b in zip(adj.csr(), want.csr()):
        assert torch.equal(a, b)
    assert data.num_features == 0 and shims.Data(x=torch.zeros(3, 7)).num_features == 7


def test_to_undirected_and_coalesce_brute_force():
    g = torch.Generator().manual_seed(2)
    N, E = 30, 200
    ei = torch.randint(0, N, (2, E), generator=g)
    w = torch.randint(1, 5, (E,), generator=g).float()
    idx, val = shims.to_undirected(ei, w, reduce="add")
    ref = {}
    for (s, d), x in zip(ei.t().tolist(), w.tolist()):
        for a, b in ((s, d), (d, s)):
            ref[(a, b)] = ref.get((a, b), 0.0) + x
    keys = sorted(ref)
    assert idx.t().tolist() == [list(k) for k in keys]
    assert torch.allclose(val, torch.tensor([ref[k] for k in keys]))
    assert torch.equal(shims.to_undirected(ei), idx)                      # without an attribute: the index only
    cidx, cval = shims.coalesce(ei, w, N, N)
    one = {}
    for (s, d), x in zip(ei.t().tolist(), w.tolist()):
        one[(s, d)] = one.get((s, d), 0.0) + x
    assert cidx.t().tolist() == [list(k) for k in sorted(one)]
    assert torch.allclose(cval, torch.tensor([one[k] for k in sorted(one)]))


@pytest.mark.parametrize("name", ["ogbl-ddi", "ogbl-collab", "ogbl-citation2"])
def test_synthetic_dataset_has_the_ogb_layout(name, monkeypatch):
    monkeypatch.setenv("PLNLP_SYNTH_SCALE", "0.002")
    ds = shims.SyntheticLinkPropPredDataset(name)
    data, split = ds[0], ds.get_edge_split()
    assert set(split) == {"train", "valid", "test"} and data.edge_index.size(0) == 2
    if name == "ogbl-citation2":
        assert set(split["valid"]) == {"source_node", "target_node", "target_node_neg"}
        assert split["valid"]["target_node_neg"].size(0) == split["valid"]["source_node"].numel()
    else:
        assert split["train"]["edge"].size(1) == 2 and "edge_neg" in split["valid"]
        assert data.edge_index.size(1) == 2 * split["train"]["edge"].size(0)     # both directions, like OGB
    assert (name == "ogbl-collab") == hasattr(data, "edge_weight")
    assert int(data.edge_index.max()) < data.num_nodes

"""GPU test (-m gpu): the call sequence of the reference's main.py (main.py:70-266) through plnlp_b200.shims on tiny
synthetic OGB-shape datasets -- dataset, ToSparseTensor, graph preparation, data.to(device), BaseModel, train, test."""
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name,encoder,predictor,metric,sampler,loss", [
    ("ogbl-ddi", "SAGE", "MLP", "hits", "global", "AUC"),
    ("ogbl-collab", "WSAGE", "DOT", "hits", "global_perm", "WeightedHingeAUC"),
    ("ogbl-citation2", "GCN", "MLP", "mrr", "local", "AUC"),
])
def test_main_py_call_sequence_through_the_shims(name, encoder, predictor, metric, sampler, loss, monkeypatch):
    from plnlp_b200 import shims
    from plnlp_b200.logger import Logger
    from plnlp_b200.model import BaseModel, adjust_lr
    from plnlp_b200.utils import adj_normalization, gcn_normalization
    monkeypatch.setenv("PLNLP_SYNTH_SCALE", "0.004")
    torch.manual_seed(0)
    device = torch.device("cuda")
    dataset = shims.SyntheticLinkPropPredDataset(name=name, root="dataset")
    data = dataset[0]
    if getattr(data, "edge_weight", None) is not None:
        data.edge_weight = data.edge_weight.view(-1).to(torch.float)
    data = shims.ToSparseTensor()(data)
    row, col, _ = data.adj_t.coo()
    data.edge_index = torch.stack([col, row], dim=0)
    num_node_feats, num_nodes = data.num_features, data.num_nodes
    split_edge = dataset.get_edge_split()
    if data.x is not None:
        data.x = data.x.to(torch.float)
    if name == "ogbl-citation2":
        data.adj_t = data.adj_t.to_symmetric()
    data = data.to(device)
    if encoder == "GCN":
        data.adj_t = gcn_normalization(data.adj_t)
    if encoder == "WSAGE":
        data.adj_t = adj_normalization(data.adj_t)
    use_feats = name == "ogbl-citation2"
    model = BaseModel(lr=0.005, dropout=0.1, grad_clip_norm=2.0, gnn_num_layers=2, mlp_num_layers=2,
                      emb_hidden_channels=32, gnn_hidden_channels=32, mlp_hidden_channels=32, num_nodes=num_nodes,
                      num_node_feats=num_node_feats, gnn_encoder_name=encoder, predictor_name=predictor,
                      loss_func=loss, optimizer_name="Adam", device=device, use_node_feats=use_feats,
                      train_node_emb=True, pretrain_emb="")
    assert sum(p.numel() for param in model.para_list for p in param) > 0          # main.py:209
    evaluator = shims.Evaluator(name=name)
    keys = ["MRR"] if metric == "mrr" else ["Hits@20", "Hits@50", "Hits@100"]
    loggers = {k: Logger(1) for k in keys}
    model.param_init()
    losses = []
    for epoch in range(1, 4):
        losses.append(model.train(data, split_edge, batch_size=512, neg_sampler_name=sampler, num_neg=2))
        results = model.test(data, split_edge, batch_size=512, evaluator=evaluator, eval_metric=metric)
        assert set(results) == set(keys)
        for key, result in results.items():
            loggers[key].add_result(0, result)
            assert all(0.0 <= v <= 1.0 for v in result)
        adjust_lr(model.optimizer, epoch / 3, 0.005)
    assert all(l == l and abs(l) < float("inf") for l in losses)                 # finite

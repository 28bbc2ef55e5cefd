"""bench.py -- the driver's measurement contract for the PLNLP hot path on B200.

  python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload citation2|ddi|collab]
                  [--dump-outputs DIR]

A "step" is one optimisation step of ``BaseModel.train`` over one batch of 65 536 positive edges and
their negatives: full-graph encode (fwd + bwd), fused edge scoring + pairwise loss, clip, Adam.
Metric (BASELINE.json): pos+neg pairs/s.

Default workload = the configuration the metric is quoted on: the citation2-shape graph (2.93 M nodes, 30.6 M
edges, GCN 2 x 200 + MLP head, local sampler).  N = 1: single GPU.  N = 2 / 4 / 8: the encoder is ROW
PARTITIONED and the run is STRONG scaling -- the global batch stays 65 536 positives (main.py:36), every rank
scores 1/N of it -- preceded by an untimed partitioned-vs-single parity check on a small graph
(``parity_check``).  The ddi- and collab-shape configs (single-GPU by north_star) ride along in ``configs`` of
the N = 1 line.

  value : K steps with the training edges resident in HBM (negatives for those K batches are sampled
          on the GPU inside the timed region, as the per-epoch sampler of the reference would).
  e2e   : the public call ``BaseModel.train(data, split_edge, ...)`` with split_edge in (pinned) HOST
          memory: H2D of the positive edges + sampler + K steps + D2H of the epoch loss.
  roofline / kernels : per-kernel CUDA-event durations from an instrumented pass of the same K steps.
  cpu_baseline : the oracle restatement of the reference step (torch CPU, all host threads) on a
          bounded sample of the same workload.

--dump-outputs DIR writes, after the timed steps, what the last of them left for its caller (``dump_outputs``) as
DIR/<name>.npy, so that two builds can be compared output for output on the same seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from

import torch  # noqa: E402

WORKLOADS = {
    # BASELINE.json configs[1] / SURVEY.md 8d config 1-2
    "ddi": dict(name="ddi-shape", N=4267, E=1067911, feats=0, emb=512, hid=512, gnn_layers=2, mlp_layers=2,
                encoder="SAGE", predictor="MLP", loss="AUC", sampler="global", num_neg=3, batch=65536,
                dropout=0.3, clip=2.0, use_feats=False, directed=False),
    # BASELINE.json configs[2] / SURVEY.md 8d config 3: the training pairs of every epoch come from the
    # random-walk augmentation (main.py:228-253, README.md:35), walk_length 10 from both endpoints
    "collab": dict(name="collab-shape", N=235868, E=1285465, feats=0, emb=256, hid=256, gnn_layers=1, mlp_layers=2,
                   encoder="SAGE", predictor="DOT", loss="WeightedHingeAUC", sampler="global", num_neg=1,
                   batch=65536, dropout=0.3, clip=1.0, use_feats=False, directed=False, powerlaw=True,
                   weighted=True, walk_length=10),
    # BASELINE.json configs[3] / SURVEY.md 8d config 4
    "citation2": dict(name="citation2-shape", N=2927963, E=30561187, feats=128, emb=50, hid=200, gnn_layers=2,
                      mlp_layers=2, encoder="GCN", predictor="MLP", loss="AUC", sampler="local", num_neg=3,
                      batch=65536, dropout=0.0, clip=1.0, use_feats=True, directed=True),
}


def workload_label(cfg):
    """the ``config.workload`` string, identical for our arm and the reference arm"""
    return (f"{cfg['name']} N={cfg['N']} E~{cfg['E']} {cfg['gnn_layers']}x{cfg['encoder']}{cfg['hid']} + "
            f"{cfg['predictor']} head, num_neg={cfg['num_neg']}, {cfg['loss']} loss, "
            f"global batch={cfg['batch']} positives/step")


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return dict(hbm=p["hbm_gbs"], tensor=p["bf16_tflops_sustained"], tensor_burst=p["bf16_tflops"], src="measured")
    except Exception:
        return dict(hbm=6650.0, tensor=1400.0, tensor_burst=1590.0, src="fallback")


class Data:
    pass


# ----------------------------------------------------------------------------- synthetic graphs
def make_edges(cfg, device, seed=0):
    """synthetic OGB-shape edge list [2, E] (SURVEY.md 8d): ddi-shape = uniform undirected simple graph;
    citation2-shape = directed, power-law in-degree."""
    g = torch.Generator(device=device).manual_seed(seed)
    N, E = cfg["N"], cfg["E"]
    if not cfg["directed"]:
        lo = torch.randint(0, N, (int(E * 1.3),), generator=g, device=device)
        if cfg.get("powerlaw"):      # collab-shape: power-law degrees (alpha ~ 2.1)
            perm = torch.randperm(N, generator=g, device=device)
            hi = perm[(N * torch.rand(int(E * 1.3), generator=g, device=device).pow(2.1)).long().clamp(max=N - 1)]
        else:
            hi = torch.randint(0, N, (int(E * 1.3),), generator=g, device=device)
        key = torch.unique(torch.minimum(lo, hi) * N + torch.maximum(lo, hi))
        key = key[torch.div(key, N, rounding_mode="floor") != key % N]
        key = key[torch.randperm(key.numel(), generator=g, device=device)[:E]]
        return torch.stack([torch.div(key, N, rounding_mode="floor"), key % N])
    u = torch.rand(E, generator=g, device=device)
    rank = (N * u.pow(2.1)).long().clamp(max=N - 1)
    perm = torch.randperm(N, generator=g, device=device)
    dst = perm[rank]
    src = torch.randint(0, N, (E,), generator=g, device=device)
    keep = src != dst
    return torch.stack([src[keep], dst[keep]])


def build_workload(cfg, device, graph_cls, normalize):
    ei = make_edges(cfg, device)
    N = cfg["N"]
    data = Data()
    if cfg["directed"]:
        adj = graph_cls.from_edge_index(ei, None, N)
        row, col, _ = adj.coo()
        data.edge_index = torch.stack([col, row], 0)         # main.py:82-83 (before symmetrisation)
        adj = adj.to_symmetric()                              # main.py:109-110
        split = {"train": {"source_node": ei[0].contiguous(), "target_node": ei[1].contiguous()}}
    else:
        und = torch.cat([ei, ei.flip(0)], 1)
        w = None
        if cfg.get("weighted"):      # collab-shape: integer collaboration counts 1..5 (ignored by SAGE's mean)
            gw = torch.Generator(device=device).manual_seed(2)
            w1 = torch.randint(1, 6, (ei.size(1),), generator=gw, device=device).float()
            w = torch.cat([w1, w1])
        adj = graph_cls.from_edge_index(und, w, N)
        row, col, _ = adj.coo()
        data.edge_index = torch.stack([col, row], 0)
        split = {"train": {"edge": ei.t().contiguous()}}
    if cfg["encoder"] == "GCN":
        adj = normalize(adj)                                  # main.py:177-179
    data.adj_t = adj
    g = torch.Generator(device=device).manual_seed(1)
    data.x = torch.randn(N, cfg["feats"], generator=g, device=device) if cfg["feats"] else None
    return data, split


def make_model(cfg, device):
    from plnlp_b200.model import BaseModel
    m = BaseModel(lr=0.001, dropout=cfg["dropout"], grad_clip_norm=cfg["clip"], gnn_num_layers=cfg["gnn_layers"],
                  mlp_num_layers=cfg["mlp_layers"], emb_hidden_channels=cfg["emb"], gnn_hidden_channels=cfg["hid"],
                  mlp_hidden_channels=cfg["hid"], num_nodes=cfg["N"], num_node_feats=cfg["feats"],
                  gnn_encoder_name=cfg["encoder"], predictor_name=cfg["predictor"], loss_func=cfg["loss"],
                  optimizer_name="Adam", device=device, use_node_feats=cfg["use_feats"], train_node_emb=True)
    m.param_init()
    return m


DUMP_TENSOR_BYTES = 8 << 20      # a larger [rows, cols] tensor is dumped as a fixed sample of its rows
DUMP_TOTAL_BYTES = 64 << 20


def dump_outputs(out_dir, model, loss_sum):
    """--dump-outputs: what the last timed step left for the caller of the batch loop, as <out_dir>/<name>.npy --
    ``loss_sum`` (float64: the batch loop's return value, sum of loss x batch size over the timed steps) and, in
    float32, every parameter after that step's Adam update (``param.<name>``) and the gradient the update used
    (``grad.<name>``; post-clip for the encoder and predictor).  A tensor over DUMP_TENSOR_BYTES (the node
    embedding) keeps the rows ``sorted(torch.randperm(rows, generator seeded 0)[:n])``, the same rows for the
    parameter and its gradient.  Multi-GPU: rank 0's tensors (its row block of the embedding)."""
    import numpy as np
    tensors = {"loss_sum": loss_sum.detach().double().reshape(1)}
    named = [(prefix + n, p) for prefix, mod in (("emb.", model.emb), ("encoder.", model.encoder),
                                                 ("predictor.", model.predictor)) if mod is not None
             for n, p in mod.named_parameters()]
    for name, p in named:
        for kind, t in (("param", p), ("grad", p.grad)):
            if t is None:
                continue
            t = t.detach().float()
            if t.dim() == 2 and t.numel() * 4 > DUMP_TENSOR_BYTES:
                n = DUMP_TENSOR_BYTES // (4 * t.size(1))
                rows = torch.randperm(t.size(0), generator=torch.Generator().manual_seed(0))[:n].sort().values
                t = t[rows.to(t.device)]
            tensors[f"{kind}.{name}"] = t
    arrays = {name: t.cpu().numpy() for name, t in tensors.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_TOTAL_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_TOTAL_BYTES}-byte budget")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    """one streaming `nvidia-smi -lms 20` process started before the warm-up; `mark()` brackets the
    timed region and only the samples that arrived inside it are summarised."""

    def __init__(self, index=0):
        self.index, self.rows, self.t0, self.t1 = index, [], None, None
        self._proc, self._t = None, None

    def _run(self):
        for line in self._proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.strip().split(",")]))

    def start(self):
        try:
            self._proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.QUERY}",
                                           "--format=csv,noheader,nounits", "-lms", "20"],
                                          stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()
        except Exception:
            self._proc = None
        return self

    def mark(self, begin):
        if begin:
            self.t0 = time.perf_counter()
        else:
            self.t1 = time.perf_counter()

    def stop(self):
        if self._proc is not None:
            self._proc.terminate()
            try:
                self._proc.wait(timeout=5)
            except Exception:
                self._proc.kill()

    def summary(self):
        inside = [r for t, r in self.rows if self.t0 is not None and self.t1 is not None and self.t0 <= t <= self.t1]
        note = "inside the timed region"
        if not inside:       # region shorter than the sampling period: fall back to the nearest samples
            inside = [r for t, r in self.rows if self.t0 is not None and t >= self.t0 - 0.5][:5]
            note = "nearest to the timed region"
        ok = [r for r in inside if len(r) >= 7]
        sm = sorted(float(r[0]) for r in ok if r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in ok if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in ok for n, v in zip(names, r[3:7]) if v.lower() == "active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(ok), "sampling": note}


# ----------------------------------------------------------------------------- our arm
NVLINK_PEER_GBS = 770.0        # measured peer-copy bandwidth per direction per GPU on this pool (B200_PROFILING.md)
EPOCH_BATCHES = {"citation2": 464, "ddi": 17, "collab": 390}     # SURVEY.md 8d: batches of one full epoch


def measure(args, workload, world, rank, device, full):
    """build the synthetic workload and time it.  ``full``: everything the JSON line needs (value, e2e, per-kernel
    pass, roofline); otherwise only the device-timed value (the secondary configs of the N = 1 line)."""
    import torch.distributed as dist

    from plnlp_b200 import _lib, profiling
    from plnlp_b200.graph import CSRGraph
    from plnlp_b200.utils import gcn_normalization, get_pos_neg_edges

    cfg = dict(WORKLOADS[workload])
    torch.manual_seed(0)
    data, split = build_workload(cfg, device, CSRGraph, gcn_normalization)
    # citation2-shape on N > 1 GPUs: ROW-PARTITIONED encoder, STRONG scaling -- the global batch stays
    # main.py:36's 65 536 positives, every rank scores 1/N of it.  The smaller graphs stay single-GPU
    # (north_star); if they are asked for with N > 1 they run as data-parallel replicas (weak scaling).
    partitioned = world > 1 and workload == "citation2"
    strong = partitioned
    if partitioned:
        from plnlp_b200 import parallel
        blk = parallel.block_size(cfg["N"], world)
        lo, hi = parallel.row_block(cfg["N"], rank, world)
        data.adj_t = parallel.shard_graph(data.adj_t, rank, world, CSRGraph, symmetric=True)
        if data.x is not None:
            data.x = parallel.pad_rows(data.x[lo:hi].contiguous(), blk)
        torch.cuda.empty_cache()
        model = make_model(dict(cfg, N=blk), device)
        model.num_nodes = cfg["N"]                     # samplers draw destinations over the global id space
    else:
        model = make_model(cfg, device)
    model.partitioned = partitioned
    model.world_size, model.rank = world, rank
    B, k = cfg["batch"], cfg["num_neg"]
    Bl = B // world if strong else B                   # positives per rank per step
    K, W = args.steps, max(args.warmup, 3)
    pos_all = split["train"]["edge"] if "edge" in split["train"] else \
        torch.stack([split["train"]["source_node"], split["train"]["target_node"]], 1)
    E = pos_all.size(0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    rw_len = cfg.get("walk_length", 0)

    def rw_epoch(edges, n_pairs):
        """random-walk augmentation (main.py:228-253): walks from both endpoints of `edges`, expanded to
        weighted (start, visited) pairs; exactly n_pairs of them are kept"""
        from plnlp_b200 import augment
        pairs, wgt = augment.random_walk_pairs(data.adj_t, edges.reshape(-1), rw_len)
        assert pairs.size(0) >= n_pairs, (pairs.size(0), n_pairs)
        return pairs[:n_pairs].contiguous(), wgt[:n_pairs].contiguous()

    def n_seed_edges(n_pairs):      # each seed edge yields 2 walks x rw_len pairs, a few are self pairs
        return int(n_pairs / (2 * rw_len) * 1.15) + 64

    def device_steps(n, seed_shift):
        """n steps on HBM-resident edges; the per-epoch producers of exactly these n batches (random-walk
        augmentation where the recipe has it, negative sampling) run on the GPU inside the call"""
        g = torch.Generator(device=device).manual_seed(1000 + seed_shift + rank)
        if rw_len:
            idx = torch.randint(0, E, (n_seed_edges(n * Bl),), generator=g, device=device)
            pos_e, wgt = rw_epoch(pos_all[idx], n * Bl)
            sub = {"train": {"edge": pos_e, "weight": wgt}}
        else:
            idx = torch.randint(0, E, (n * Bl,), generator=g, device=device)
            sub = {"train": {"edge": pos_all[idx]}}
            wgt = None
        pos, neg = get_pos_neg_edges("train", sub, edge_index=data.edge_index, num_nodes=cfg["N"],
                                     neg_sampler_name=cfg["sampler"], num_neg=k, device=device)
        model.encoder.train(); model.predictor.train()
        # the batch loop of BaseModel.train (index work of batch i + 1 prepared on a side stream while batch i runs)
        return model.run_batches(data, ((pos[i * Bl:(i + 1) * Bl], neg[i * Bl:(i + 1) * Bl].reshape(-1, 2),
                                         None if wgt is None else wgt[i * Bl:(i + 1) * Bl]) for i in range(n)), k)

    out = {"cfg": cfg, "E": E, "partitioned": partitioned, "strong": strong, "K": K, "W": W}

    # ---- multi-GPU parity, untimed: the partitioned step vs the single-GPU step on a small graph ---------
    if full and partitioned:
        from plnlp_b200 import selfcheck
        errs = selfcheck.summarize(selfcheck.partitioned_step(rank, world, device, force_sparse=True))
        out["parity_check"] = {
            "loss_rel": max_over_ranks(errs["loss_rel"]), "max_grad_rel": max_over_ranks(errs["max_grad_rel"]),
            "max_grad_rel_per_tensor": max_over_ranks(errs["max_grad_rel_per_tensor"]),
            "fp32_noise_floor": max_over_ranks(errs["fp32_noise_floor"]),
            "what": f"one optimisation step of the row-partitioned model on {world} ranks vs the single-GPU model on "
                    "the same parameters, graph (60 000 nodes, GCN 2x32 + MLP head, features + embedding) and global "
                    "batch; max over ranks; max_grad_rel = largest |d - d_single| over every gradient tensor / largest "
                    "gradient magnitude of the model (per_tensor: relative to each tensor's own magnitude, which for "
                    "the predictor biases is cancellation noise: d loss / d score sums to 0 under the AUC loss); "
                    "fp32_noise_floor = the same quantity between two SINGLE-GPU runs of that step that differ only in "
                    "the order of the pairs inside the batch -- what a change of summation order alone costs"}
        torch.cuda.empty_cache()

    # ---- value: device-resident ------------------------------------------------------------
    import gc
    clk = ClockSampler(device.index or 0).start()
    device_steps(W, 0)
    barrier()
    w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0.record()
    device_steps(K, 3)            # untimed for the record: lets the caching allocator see the K-step tensor sizes once
    w1.record()
    barrier()
    out["ms_per_step_rehearsal_pass"] = max_over_ranks(w0.elapsed_time(w1)) / K
    gc.collect()
    gc.disable()                  # no python garbage-collection pause inside a 0.1 - 0.5 s timed region
    barrier()
    l0 = _lib.launch_count()
    clk.mark(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    timed = device_steps(K, 1)
    e1.record()
    barrier()
    gc.enable()
    clk.mark(False)
    clk.stop()
    ms = max_over_ranks(e0.elapsed_time(e1))
    out["launches"] = _lib.launch_count() - l0
    if full and rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, model, timed[0])
    # host side of the same K steps: how long python + the launch calls take to ENQUEUE them (no device wait).  When
    # this approaches ms_per_step the run is launch-bound, not kernel-bound
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    device_steps(K, 4)
    out["host_enqueue_ms_per_step"] = max_over_ranks((time.perf_counter() - t0) * 1e3 / K)
    barrier()
    pairs = K * Bl * (1 + k) * world
    out.update(ms=ms, pairs=pairs, value=pairs / (ms / 1e3), clocks=clk.summary(), Bl=Bl)
    if not full:
        return out

    # ---- e2e: public API with HOST split_edge ----------------------------------------------
    # the "epoch" handed to train() holds exactly K (resp. W) full batches per rank, in pinned host memory;
    # BaseModel.train gives rank r the r-th contiguous block of it
    def host_epoch(n_steps, seed):
        g = torch.Generator().manual_seed(seed)
        n = n_seed_edges(n_steps * Bl) if rw_len else n_steps * Bl * world
        idx = torch.randint(0, E, (n,), generator=g)
        return {"train": {kk: v.cpu()[idx].contiguous().pin_memory() for kk, v in split["train"].items()}}

    def public_epoch(hs, n_steps):
        """what main.py does per epoch: [random-walk augmentation of the train edges ->] BaseModel.train"""
        if rw_len:
            assert world == 1, "the collab-shape workload is single-GPU (north_star: smaller graphs stay single-GPU)"
            pos_e, wgt = rw_epoch(hs["train"]["edge"].to(device, non_blocking=True), n_steps * Bl)
            hs = {"train": {"edge": pos_e, "weight": wgt}}
        return model.train(data, hs, batch_size=Bl, neg_sampler_name=cfg["sampler"], num_neg=k)

    warm_split, host_split = host_epoch(W, 11), host_epoch(K, 12)
    public_epoch(warm_split, W)
    public_epoch(host_split, K)                                   # allocator warm-up with the K-step sizes
    gc.collect()
    gc.disable()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    public_epoch(host_split, K)
    e1.record()
    barrier()
    gc.enable()
    assert model.last_epoch_stats == {"batches": K, "examples": K * Bl}, model.last_epoch_stats
    e2e_ms = max_over_ranks(e0.elapsed_time(e1))
    h2d = sum(v.numel() * v.element_size() for v in host_split["train"].values()) // world
    out["e2e"] = {"value": pairs / (e2e_ms / 1e3), "unit": "pairs/s", "h2d_bytes_per_step": h2d // K,
                  "d2h_bytes_per_step": 8, "ms_per_step": e2e_ms / K,
                  "note": "one BaseModel.train(data, split_edge) call whose split_edge (pinned HOST tensors) holds exactly "
                          "K batches: H2D of this rank's share of the positive edges, GPU negative sampling, K optimisation "
                          "steps, D2H of the epoch loss (one 8-byte read per call, not per step)"}

    # ---- instrumented pass: per-kernel durations (rank 0) ------------------------------------
    # every rank runs the pass instrumented (identical control flow on every rank: the instrumented form runs the
    # collectives synchronously); only rank 0 reports
    profiling.enable()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    device_steps(K, 2)
    p1.record()
    barrier()
    stats = profiling.disable()
    if rank == 0:
        pk = peaks()
        ours = sum(s["ms"] for s in stats.values())
        stats["(torch plumbing: adam, clip, unique / sort, sampler glue, launch gaps)"] = {
            "n": 1, "ms": max(p0.elapsed_time(p1) - ours, 0.0), "bytes": 0, "flops": 0}
        total = sum(s["ms"] for s in stats.values()) or 1.0
        kernels = []
        for name, s in sorted(stats.items(), key=lambda kv: -kv[1]["ms"]):
            rec = {"kernel": name, "launches": s["n"], "ms_total": round(s["ms"], 3),
                   "share": round(s["ms"] / total, 4), "avg_ms": round(s["ms"] / s["n"], 4)}
            if name.startswith(("nccl", "p2p")):
                if s["bytes"]:
                    rec["recv_gbs_per_rank"] = round(s["bytes"] / s["ms"] / 1e6, 1)
                    rec["frac_nvlink"] = round(s["bytes"] / s["ms"] / 1e6 / NVLINK_PEER_GBS, 4)
            else:
                if s["bytes"]:
                    rec["achieved_gbs"] = round(s["bytes"] / s["ms"] / 1e6, 1)
                    rec["frac_hbm"] = round(s["bytes"] / s["ms"] / 1e6 / pk["hbm"], 4)
                if s["flops"]:
                    rec["achieved_tflops"] = round(s["flops"] / s["ms"] / 1e9, 2)
                    rec["frac_tensor"] = round(s["flops"] / s["ms"] / 1e9 / pk["tensor"], 4)
            kernels.append(rec)
        out["kernels"] = kernels
        # dominant kernel of OURS (collectives and torch glue have their own lines)
        top = next(r for r in kernels if not r["kernel"].startswith(("(", "nccl", "p2p", "torch")))
        if "achieved_gbs" in top or "achieved_tflops" not in top:
            roof = {"kernel": top["kernel"], "bound": "hbm", "achieved": top.get("achieved_gbs"),
                    "peak": pk["hbm"], "unit": "GB/s", "frac": top.get("frac_hbm"), "traffic": None,
                    "peak_source": pk["src"] + " (copy bandwidth)"}
        else:
            roof = {"kernel": top["kernel"], "bound": "tensor", "achieved": top["achieved_tflops"],
                    "peak": pk["tensor"], "unit": "TFLOP/s", "frac": top["frac_tensor"], "traffic": None,
                    "peak_source": pk["src"] + " bf16 sustained; kernel computes in fp32 (3xTF32)",
                    "passes": 3, "ceiling_3xtf32": round(pk["tensor"] / 6.0, 1),
                    "frac_of_3xtf32_ceiling": round(top["achieved_tflops"] / (pk["tensor"] / 6.0), 4)}
        try:        # measured DRAM traffic per launch of that kernel, from the committed ncu --set full capture
            if world > 1:     # the captures are single-GPU launches over the whole graph: no per-rank figure
                raise KeyError("no ncu capture at the row-partitioned shape")
            tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))[workload][top["kernel"]]
            roof["traffic"], roof["traffic_source"] = tr["bytes"], "profiles/" + tr["source"]
        except Exception:
            pass
        spmm = [r for r in kernels if r["kernel"].startswith("spmm") and "achieved_gbs" in r]
        if spmm:
            src_bytes = cfg["N"] * cfg["hid"] * 4
            roof["spmm"] = [{"kernel": r["kernel"], "achieved_gbs": r["achieved_gbs"], "frac_hbm": r["frac_hbm"],
                             "share_of_step": r["share"]} for r in spmm]
            roof["spmm_note"] = ("source matrix exceeds L2" if src_bytes >= 126e6 else
                                 "source matrix is L2-resident: effective bandwidth of the gather model")
        out["roofline"] = roof
        nccl = [r for r in kernels if r["kernel"].startswith(("nccl", "p2p"))]
        if nccl:
            out["nvlink"] = {"peak_gbs_per_direction": NVLINK_PEER_GBS, "peak_source": "measured peer copy (B200_PROFILING.md)",
                             "collectives": nccl, "ms_per_step_run_alone": round(sum(r["ms_total"] for r in nccl) / K, 3),
                             "note": "durations from the instrumented pass, which runs every collective synchronously; in "
                                     "the timed passes the layer-1 reduce-scatter overlaps the weight-gradient GEMM"}
    # ---- the stated fast path (N = 1): plain single-pass TF32 dense layers, NOT the parity path ---------------
    if world == 1 and rank == 0 and not args.no_extra:
        from plnlp_b200 import _ops
        with torch.no_grad():
            model.encoder.eval()
            h_ref = model.encoder(model.input_parts(data), data.adj_t)
        was = _ops.GEMM_BACKEND
        _ops.GEMM_BACKEND = "tf32c2"
        try:
            with torch.no_grad():
                h_fast = model.encoder(model.input_parts(data), data.adj_t)
            err = float((h_fast - h_ref).abs().max() / h_ref.abs().max())
            del h_fast, h_ref
            device_steps(W, 20)
            torch.cuda.synchronize()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
            device_steps(K, 21)
            f1.record()
            torch.cuda.synchronize()
            fms = f0.elapsed_time(f1)
            out["fast_path"] = {"dtype": "tf32", "value": pairs / (fms / 1e3), "unit": "pairs/s", "ms_per_step": fms / K,
                                "max_rel_err_of_encoder_output_vs_fp32_path": err,
                                "note": "same workload with the dense layers in plain single-pass TF32 (PLNLP_GEMM=tf32c2; "
                                        "tcgen05 kind::tf32, one MMA per product instead of the error-compensated three). "
                                        "Stated separately: it does not meet the 1e-5 parity bar and is never used for the "
                                        "headline value, the parity tests or smoke()"}
        finally:
            _ops.GEMM_BACKEND = was
            model.encoder.train()
    return out


def run_ours(args):
    import torch.distributed as dist

    from plnlp_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    assert _lib.load().plnlp_check_device() == 0, "plnlp_b200 needs an sm_100 device"
    m = measure(args, args.workload, world, rank, device, full=True)
    cfg, K, W, B, k = m["cfg"], m["K"], m["W"], m["cfg"]["batch"], m["cfg"]["num_neg"]

    # ---- the other single-GPU configs of BASELINE.json (N = 1 line only): one epoch-sized run each ----------
    others = []
    if world == 1 and args.workload == "citation2" and not args.no_extra:
        import gc
        for wl in ("ddi", "collab"):
            gc.collect()
            torch.cuda.empty_cache()
            sub = argparse.Namespace(**vars(args))
            sub.steps, sub.warmup = 17, 3
            try:
                o = measure(sub, wl, 1, 0, device, full=False)
                c = o["cfg"]
                others.append({"workload": f"{c['name']} N={c['N']} {c['gnn_layers']}x{c['encoder']}{c['hid']} + "
                                           f"{c['predictor']} head, {c['loss']} loss, num_neg={c['num_neg']}"
                                           + (f", random-walk augmentation L={c['walk_length']}" if c.get("walk_length") else ""),
                               "value": o["value"], "unit": "pairs/s", "ms_per_step": o["ms"] / o["K"], "steps": o["K"],
                               "warmup": o["W"], "epoch_s": o["ms"] / o["K"] * EPOCH_BATCHES[wl] / 1e3,
                               "gpu_launches": int(o["launches"]), "clocks": o["clocks"]})
            except Exception as ex:      # a secondary config must never take the headline line with it
                others.append({"workload": wl, "error": repr(ex)[:300]})

    # ---- CPU baseline (rank 0, N=1 only) -------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_baseline_guarded(args.workload, args.cpu_steps)

    if rank == 0:
        ms = m["ms"]
        par = ("single GPU" if world == 1 else
               f"encoder row-partitioned over {world} ranks (all-gather / reduce-scatter of the 50-wide embedding block "
               f"per step, restricted last conv as column-block partial products + all-reduce of the compact rows), "
               f"global batch of {B} positives split {world} ways, flat all-reduce of the dense-weight gradients"
               if m["partitioned"] else f"dp{world} over edge batches, encoder replicated, flat grad all-reduce")
        line = {"metric": "pos+neg pairs/s (train step)", "value": m["value"], "unit": "pairs/s", "n_gpus": world,
                "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True,
                "scaling": "strong" if (m["strong"] or world == 1) else "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": workload_label(cfg), "edges": m["E"], "dropout": cfg["dropout"],
                           "pairs_per_step": m["Bl"] * (1 + k) * world,
                           "positives_per_step_per_gpu": m["Bl"],
                           "l2": "inputs larger than L2: every step streams the adjacency (> 0.7 GB) and [N, F] "
                                 "activations (> 0.5 GB each) through the 126 MB L2; no explicit flush",
                           "parallelism": par},
                "epoch": {"batches": EPOCH_BATCHES[args.workload],
                          "seconds": ms / K * EPOCH_BATCHES[args.workload] / 1e3,
                          "note": "ms_per_step x the batches of one full epoch (SURVEY.md 8d)"},
                "clocks": m["clocks"], "e2e": m["e2e"], "gpu_launches": int(m["launches"]),
                "host_enqueue_ms_per_step": round(m["host_enqueue_ms_per_step"], 3),
                "ms_per_step_rehearsal_pass": round(m["ms_per_step_rehearsal_pass"], 3),
                "roofline": m.get("roofline"), "kernels": m.get("kernels", [])[:14]}
        if "nvlink" in m:
            line["nvlink"] = m["nvlink"]
        if "parity_check" in m:
            line["parity_check"] = m["parity_check"]
        if "fast_path" in m:
            line["fast_path"] = m["fast_path"]
        if others:
            line["configs"] = others
        line["cpu_baseline"] = cpu
        emit(line)
    if world > 1:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------- CPU arm
def cpu_baseline_guarded(workload, steps, timeout_s=None):
    """``cpu_baseline`` in a CHILD interpreter with a time limit.  A fresh process keeps the host-thread pool of
    the CPU arm apart from the CUDA process (one such run stalled indefinitely inside the bench process on a
    GPU box), and a stall can then cost at most ``timeout_s``: the run is retried once with 8 threads and
    otherwise reported as unavailable instead of taking the whole bench line with it."""
    import subprocess
    if timeout_s is None:       # normal duration: ~15 s (ddi / collab shape), ~90 s (citation2 shape: graph build + steps)
        timeout_s = 420 if workload == "citation2" else 240
    code = ("import json, sys, bench; "
            "print('CPU_BASELINE ' + json.dumps(bench.cpu_baseline(dict(bench.WORKLOADS[sys.argv[1]]), "
            "steps=int(sys.argv[2]), threads=int(sys.argv[3]) or None)))")
    last = "no attempt"
    for threads in (0, 8):
        try:
            r = subprocess.run([sys.executable, "-B", "-c", code, workload, str(steps), str(threads)], cwd=ROOT,
                               capture_output=True, text=True, timeout=timeout_s)
            for ln in r.stdout.splitlines():
                if ln.startswith("CPU_BASELINE "):
                    return json.loads(ln[len("CPU_BASELINE "):])
            last = f"child exited {r.returncode}: {r.stderr.strip()[-300:]}"
        except subprocess.TimeoutExpired:
            last = f"timed out after {timeout_s} s with {'all' if not threads else threads} threads"
    return {"unavailable": last, "kind": "port"}


def cpu_baseline(cfg, steps=2, threads=None):
    """the oracle restatement of the reference's train step (torch CPU, all host threads) on a bounded
    sample: `steps` optimisation steps of the same workload (full-graph encode each)."""
    from oracle import plnlp_ref, sparse
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    cpu = torch.device("cpu")
    data, split = build_workload(cfg, cpu, _OracleGraph, sparse.gcn_normalization)
    m = plnlp_ref.OracleModel(num_nodes=cfg["N"], emb_hidden=cfg["emb"], gnn_hidden=cfg["hid"], mlp_hidden=cfg["hid"],
                              gnn_layers=cfg["gnn_layers"], mlp_layers=cfg["mlp_layers"], encoder=cfg["encoder"],
                              predictor=cfg["predictor"], loss=cfg["loss"], lr=0.001, clip_norm=cfg["clip"],
                              num_node_feats=cfg["feats"], use_node_feats=cfg["use_feats"])
    pos_all = plnlp_ref.train_pos_edges(split)
    B, k, N = cfg["batch"], cfg["num_neg"], cfg["N"]
    g = torch.Generator().manual_seed(3)

    def one():
        idx = torch.randint(0, pos_all.size(0), (B,), generator=g)
        pos = pos_all[idx]
        neg = torch.stack([pos[:, :1].expand(B, k), torch.randint(0, N, (B, k), generator=g)], -1)
        wgt = (1.0 / torch.randint(1, 11, (B,), generator=g).float()) if cfg["loss"] == "WeightedHingeAUC" else None
        m.step(data.x, data.adj_t, pos, neg, k, wgt)

    one()                                    # warm-up (allocator, MKL)
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    dt = time.perf_counter() - t0
    return {"value": steps * B * (1 + k) / dt, "unit": "pairs/s", "cores": threads, "kind": "port",
            "sample": f"{steps} train steps of {B * (1 + k)} pairs on the same {cfg['name']} workload after 1 warm-up "
                      f"step ({dt:.1f} s); oracle restatement of the reference step in torch CPU "
                      "(torch_geometric / torch_sparse are not installable here, so this is NOT the PyG path); "
                      "negatives pre-drawn uniformly (sampler cost excluded)", "seconds": dt}


class _OracleGraph:
    """adapter giving oracle.sparse.SparseTensor the constructor name build_workload uses"""

    @staticmethod
    def from_edge_index(ei, w, N):
        from oracle import sparse
        return sparse.to_sparse_tensor(ei, w, N)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = dict(WORKLOADS[args.workload])
    K, W = args.steps, args.warmup
    steps = max(1, min(K, args.cpu_steps))
    cpu = cpu_baseline_guarded(args.workload, steps)
    if "unavailable" in cpu:
        emit({"impl": "reference", "unavailable": cpu["unavailable"]})
        return
    B, k = cfg["batch"], cfg["num_neg"]
    line = {"impl": "reference", "metric": "pos+neg pairs/s (train step)", "value": cpu["value"], "unit": "pairs/s",
            "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": steps, "warmup": 1,
            "ms_per_step": cpu["seconds"] / steps * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_label(cfg), "requested_steps": K, "requested_warmup": W,
                       "pairs_per_step": B * (1 + k)},
            "cpu_baseline": cpu,
            "e2e": {"value": cpu["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


_OUT = None


def emit(line):
    out = _OUT if _OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    # default: the configuration BASELINE.json's metric is quoted on -- citation2-shape, single GPU at N = 1,
    # row-partitioned at N = 2 / 4 / 8 (the ddi / collab shapes ride along in "configs" of the N = 1 line)
    ap.add_argument("--workload", default="citation2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-extra", action="store_true", help="skip the ddi / collab one-epoch runs of the N = 1 line")
    ap.add_argument("--cpu-steps", type=int, default=None,
                    help="steps of the CPU arm's bounded sample (default: ~10-20 s of CPU work: one 17-batch epoch of "
                         "the ddi / collab shape, 2 steps of the citation2 shape)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.cpu_steps is None:
        args.cpu_steps = 2 if args.workload == "citation2" else 17
    # the contract is ONE JSON line on stdout: keep a private handle to the real stdout and point fd 1
    # at stderr so that library banners (e.g. "NCCL version ...") cannot pollute it
    global _OUT
    _OUT = os.fdopen(os.dup(1), "w")
    sys.stdout.flush()
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

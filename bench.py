#!/usr/bin/env python
"""Benchmark of the PC-GNN pick-and-choose hot path on B200 (contract: see DESIGN.md "Measurement").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload yelp|amazon|yelp100|amazon_gcn|big]
                  [--scaling weak|strong] [--impl reference] [--check-only] [--torch-adam] [--nccl-scores]
                  [--no-graph] [--no-cpu-baseline] [--dump-outputs DIR]

One "step" = one full training step of PCALayer(InterAgg3(IntraAgg x3)) on one label-balanced batch of target
nodes: score table + pool sort (next to the choose preparation), choose, aggregate, the fused dense / loss /
activation-gradient kernel, the weight-gradient kernel, gradient mean over the ranks + Adam (one kernel over NVLink
peer memory; --torch-adam: NCCL all-reduce + torch.optim.Adam). Under torchrun every rank runs its shard; rank 0
prints ONE JSON line.

  value      train target-nodes/s with the batches already resident in HBM (one CUDA-graph replay per step)
  e2e        host inputs, host<->device copies inside the timed region, through runtime.GraphedTrainStep.run(ids,
             labels) + loss.item() (pinned staging, H2D, one graph replay, D2H) -- the same call at every GPU count.
             e2e_reference_loop (1 GPU; the reference has no data parallelism): the REFERENCE's own loop, unchanged
             (model_handler.py:142-156: zero_grad; model.loss(list_of_ids, cuda LongTensor labels); backward;
             torch.optim.Adam.step; loss.item()), which the package serves from its CUDA-graph cache
  roofline   the slower of the two hot-path kernel groups (choose / aggregate): SURVEY 8(d) algorithmic bytes per
             launch / CUDA-event time against MEASURED_PEAKS.json, next to the bytes the kernels must actually move
             (`required_*`: without the reference's per-target pool scan, which the sorted pool makes unnecessary);
             traffic = ncu DRAM bytes per launch (profiles/)
  cpu_baseline  the oracle port (same per-target structure as the reference, CPU) on a bounded sample of a batch

Workloads (BASELINE.json configs): yelp = C2 (default, the config the metric is quoted on), amazon = C1,
yelp100 = C3 (BASELINE: global batch 4096 sharded over the GPUs = --scaling strong), amazon_gcn = C4, big = C5
(row-partitioned CSR, 1.25M nodes / 1.26e8 entries per GPU). --scaling weak (default): `batch` targets per GPU;
strong: `batch` targets in total. Shards are dealt by row length (largest first, round robin) so that every rank
gets the same number of targets AND about the same number of neighbour entries.
`--impl reference` times the oracle port alone on the host cores (the reference is pure Python and is not present
on the GPU box; oracle/port.py is its restatement, pinned by tests/golden).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (synthetic spec, batch per GPU, embed dim, description)
    "yelp": ("yelp", 1024, 64, "C2 YelpChi-shaped N=45954 F=32 R=3 ~4.0M edges, emb 64, batch 1024/GPU"),
    "amazon": ("amazon", 1024, 64, "C1 Amazon-shaped N=11944 F=25 R=3 ~4.8M edges, emb 64, batch 1024/GPU"),
    "yelp100": ("yelp100", 4096, 128, "C3 YelpChi-shaped F=100, emb 128, batch 4096/GPU"),
    "amazon_gcn": ("amazon", 1024, 64, "C4 GCN baseline on the Amazon-shaped union graph, emb 64, batch 1024/GPU"),
    "big": ("big", 1024, 64, "C5 power-law fraud graph, 1.25M nodes and ~1.25e8 CSR entries PER GPU (10M / 1e9 at 8 GPUs), "
                             "F=64, R=3, 10% positives, CSR row-partitioned by node range, emb 64, batch 1024/GPU"),
}
RHO, ALPHA, LR, WD = 0.5, 2.0, 0.01, 1e-3
SEED = 72


MY_KERNELS_PER_STEP = 9    # choose prep 1 (side branch) | score table + pool sort 2, choose 2 (wide, small), aggregate 1,
#                            fused dense/loss/activation-gradient 1, weight gradients 1, gradient exchange + Adam 1
#                            (+2 when P > 8192, +1 per extra row tier, +1 loss-word copy kernel in the host-batch
#                            recording; device batches: + one multi-tensor copy of ids / labels in front of the replay)


def config_dict(desc, global_batch, world, scaling="weak"):
    return {"workload": desc, "global_batch": global_batch, "rho": RHO, "thresholds": 0.5, "optimizer": "Adam",
            "l2": "flushed between timed steps (256 MiB write)",
            "parallelism": (f"dp{world} (targets dealt to the ranks by row length, grads averaged; {scaling} scaling)"
                            if world > 1 else "single")}


def deal(nodes, labels, weight, rank, world):
    """This rank's share of a global batch: targets sorted by `weight` (their total row length) descending and dealt
    round robin, so every rank gets len/world targets and about the same number of neighbour entries (contiguous
    shards differ by the hubs they happen to contain: the ranks then wait for the slowest in the exchange)."""
    order = np.argsort(-weight[nodes], kind="stable")
    mine = order[rank::world]
    return nodes[mine], labels[mine]


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def make_batches(data, n_batches, batch, seed):
    """Label-balanced batches: nodes drawn with pick_step's weights deg/LF (utils.py:274-278)."""
    from pcgnn_b200.utils import pick_weights

    w = pick_weights(data.idx_train, data.y_train, data.homo)
    rng = np.random.default_rng(seed)
    idx = np.asarray(data.idx_train)
    out = []
    for _ in range(n_batches):
        nodes = idx[rng.choice(len(idx), batch, p=w / w.sum())]
        out.append((nodes.astype(np.int64), data.labels[nodes].astype(np.int64)))
    return out


def init_params(feat_dim, embed, n_rel, seed):
    rng = np.random.default_rng(seed)

    def xavier(r, c):
        a = np.sqrt(6.0 / (r + c))
        return rng.uniform(-a, a, size=(r, c)).astype(np.float32)

    return dict(intra=[xavier(2 * feat_dim, embed) for _ in range(n_rel)], inter=xavier(feat_dim + n_rel * embed, embed),
                clf_w=xavier(2, feat_dim), clf_b=np.zeros(2, np.float32), head=xavier(2, embed),
                enc=xavier(embed, feat_dim))      # enc: GCNEncoder weight [E,F] (C4 only)


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.samples, self.reasons, self.stop_flag, self.max_mhz = [], set(), False, None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def sample(self):
        if self.nv is None:
            return
        nv = self.nv
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                     "hw_power_brake": 0x80, "sync_boost": 0x10}
            for k, bit in names.items():
                if r & bit:
                    self.reasons.add(k)
        except Exception:
            pass

    def run(self):
        while not self.stop_flag:
            self.sample()
            time.sleep(0.02)

    def result(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def cpu_port_rate(data, params, batches, sample, steps, warmup, gcn=False):
    """Oracle port (CPU restatement of the reference's structure): full train steps on `sample` targets."""
    import torch
    from oracle import port

    tp = sorted(data.train_pos)
    if gcn:
        pm = port.PortGCN(data.feat, data.homo, params["enc"], params["head"])
    else:
        pm = port.PortPCGNN(data.feat, data.graph, tp, params, rho=RHO, alpha=ALPHA)
    opt = torch.optim.Adam(pm.parameters(), lr=LR, weight_decay=WD)
    times = []
    for s in range(warmup + steps):
        nodes, labels = batches[s % len(batches)]
        t0 = time.perf_counter()
        opt.zero_grad()
        if gcn:
            loss = pm.loss(nodes[:sample].tolist(), labels[:sample])
        else:
            loss = pm.loss(nodes[:sample].tolist(), labels[:sample], True, shared_table=False)
        loss.backward()
        opt.step()
        dt = time.perf_counter() - t0
        if s >= warmup:
            times.append(dt)
    return sample / float(np.mean(times)), float(np.mean(times))


def c_port_rate(data, batches, reps=3):
    """C restatement (OpenMP, all host cores) of choose + aggregate only, full batch."""
    from oracle import c_oracle

    c_oracle.lib()
    rng = np.random.default_rng(1)
    score = (data.feat @ rng.normal(size=data.feat.shape[1]).astype(np.float32) * 0.3).astype(np.float32)
    tp = sorted(data.train_pos)
    best = 1e9
    for i in range(reps):
        nodes, labels = batches[i % len(batches)]
        t0 = time.perf_counter()
        sp, si = c_oracle.choose(data.graph, score, nodes, labels == 1, rho=RHO, pool=tp, train=True)
        c_oracle.aggregate(data.feat, sp, si)
        best = min(best, time.perf_counter() - t0)
    return len(batches[0][0]) / best


GCN_KERNELS_PER_STEP = 7   # select-all, aggregate, encoder fwd, head+CE fwd, head+CE bwd, encoder bwd, exchange + Adam


def build_cuda_pcgnn_device(feat_dev, graph, train_pos_dev, params, dev):
    """PCALayer(InterAgg3(IntraAgg x3)) over tables that already live on the device (workload big)."""
    import torch
    import torch.nn as nn

    from pcgnn_b200.layers import InterAgg3, IntraAgg
    from pcgnn_b200.model import PCALayer

    F_, E = feat_dev.shape[1], params["inter"].shape[1]
    features = nn.Embedding(1, 1)
    features.weight = nn.Parameter(feat_dev, requires_grad=False)          # no copy of the 2.56 GB table
    features.num_embeddings, features.embedding_dim = feat_dev.shape
    intras = [IntraAgg(features, F_, E, train_pos_dev, RHO, cuda=True) for _ in range(graph.n_rel)]
    inter = InterAgg3(features, F_, E, train_pos_dev, graph, intras, cuda=True)
    model = PCALayer(2, inter, ALPHA)
    with torch.no_grad():
        for ia, w in zip(intras, params["intra"]):
            ia.weight.copy_(torch.from_numpy(np.asarray(w)))
        inter.weight.copy_(torch.from_numpy(params["inter"]))
        inter.label_clf.weight.copy_(torch.from_numpy(params["clf_w"]))
        inter.label_clf.bias.copy_(torch.from_numpy(params["clf_b"]))
        model.weight.copy_(torch.from_numpy(params["head"]))
    return model.to(dev)


def build_cuda_gcn(data, params, dev):
    """GCN(GCNEncoder(GCNAggregator)) of the product on the union graph (model_handler.py:99-101, 119-120)."""
    import torch
    import torch.nn as nn
    from pcgnn_b200 import graphsage as gs

    F_ = data.feat.shape[1]
    E = params["enc"].shape[0]
    features = nn.Embedding(*data.feat.shape)
    features.weight = nn.Parameter(torch.from_numpy(np.ascontiguousarray(data.feat)), requires_grad=False)
    features = features.to(dev)
    enc = gs.GCNEncoder(features, F_, E, data.homo, gs.GCNAggregator(features, cuda=True), cuda=True)
    model = gs.GCN(2, enc)
    with torch.no_grad():
        enc.weight.copy_(torch.from_numpy(params["enc"]))
        model.weight.copy_(torch.from_numpy(params["head"]))
    return model.to(dev)


def _ncu_traffic(workload, group):
    """DRAM bytes per launch of a kernel group from the committed ncu capture (profiles/r02_traffic.json)."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            t = json.load(open(os.path.join(ROOT, "profiles", name)))
            return t[workload][group]["bytes"]
        except Exception:
            continue
    return None


def _roof(kern, dom, extra=None, workload=None):
    """roofline object for the dominant kernel group. `achieved` follows SURVEY 8(d) (algorithmic bytes); when that
    figure exceeds what the memory system can do (it counts a per-target scan of the whole pool that the sorted-pool
    kernels never perform) the bytes the kernels must move are used instead, and said so."""
    peak, peak_src = measured_peaks()
    k = kern[dom]
    r = {"bound": "hbm", "kernel": dom, "achieved": k["gbs"], "peak": peak, "unit": "GB/s", "frac": k["gbs"] / peak,
         "traffic": _ncu_traffic(workload, dom), "peak_source": peak_src, "algorithmic_bytes": k["alg_bytes"],
         "bytes": "algorithmic (SURVEY 8d)"}
    if "req_bytes" in k:
        r.update({"required_bytes": k["req_bytes"], "required_gbs": k["req_gbs"], "required_frac": k["req_gbs"] / peak})
        if r["frac"] > 1.2:
            r.update({"achieved": k["req_gbs"], "frac": k["req_gbs"] / peak, "algorithmic_gbs": k["gbs"],
                      "bytes": "required (the 8d figure counts a scan of the whole pool per positive target that the "
                               "sorted-pool kernels do not perform; it would exceed the peak)"})
    r.update(extra or {})
    return r


def hot_kernels_pcgnn(eng, inter, data, shards, dev_nodes, dev_labels, cap, W, K, flush, dev, batch, workload=None):
    """The hot-path kernel groups captured alone in CUDA graphs, CUDA-event time per replay, L2 flushed before each:
      front      what runs in front of the selection as in the step: pool scores -> (choose preparation || pool sort ||
                 score table)
      choose     the selection kernels (k_choose_small || k_choose_wide [|| huge / big tiers]): the dominant group
      aggregate  k_aggregate
    Bytes per SURVEY 8(d): filter = 8 per CSR entry of the batch's rows + 16 R B + 4 B + 4 P R B+ (pool scan)
    [+ 4 per kept id written]; aggregate = (4F + 4) per gathered row + 4 F R B."""
    import torch
    from pcgnn_b200 import _lib

    R, F_ = data.graph.n_rel, data.feat.shape[1]
    t_choose = t_agg = t_front = 0.0
    alg_choose = alg_agg = req_choose = 0.0
    P = eng.P
    st_nodes = dev_nodes[W].clone()
    st_labels = dev_labels[W].clone()
    exchange = eng.score_group is not None          # partitioned graph + NCCL scores: the all-gather stays outside the graphs
    w_, b_ = inter.label_clf.weight, inter.label_clf.bias
    rho = inter.intra_agg1.rho
    holder = {}

    def front():
        cur = torch.cuda.current_stream(dev)
        s0, s1 = eng.side_stream(0), eng.side_stream(1)
        if exchange:
            eng.score_local(w_, b_)
            return
        ps = eng.pool_scores(w_, b_)
        s0.wait_stream(cur)
        s1.wait_stream(cur)
        with torch.cuda.stream(s0):
            holder["sel"] = eng.choose(st_nodes, st_labels, True, inter.thresholds, rho, cap, phases=1)
        with torch.cuda.stream(s1):
            eng.sort_pool_from(ps)
        eng.score_table_only(w_, b_)
        cur.wait_stream(s0)
        cur.wait_stream(s1)

    def tiers():
        if exchange:
            holder["sel"] = eng.choose(st_nodes, st_labels, True, inter.thresholds, rho, cap)
        else:
            eng.choose(st_nodes, st_labels, True, inter.thresholds, rho, cap, phases=2, sel=holder["sel"])

    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for _ in range(2):
            front()
            if exchange:
                eng.score_exchange()
                eng.resort_pool()
            tiers()
            eng.aggregate(holder["sel"], copy_dups=False)
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize()
    g_front, g_choose, g_agg = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
    with _lib.capture(g_front):
        front()
    with _lib.capture(g_choose):
        tiers()
    sel = holder["sel"]
    with _lib.capture(g_agg):
        eng.aggregate(sel, copy_dups=False)       # as in the train step: the dense kernels read through it_rep
    for s in range(K):
        i = W + s
        st_nodes.copy_(dev_nodes[i])
        st_labels.copy_(dev_labels[i])
        flush.zero_()
        e0, e1, e2, e3 = (torch.cuda.Event(enable_timing=True) for _ in range(4))
        e0.record()
        g_front.replay()
        if exchange:
            eng.score_exchange()
            eng.resort_pool()
        e1.record()
        g_choose.replay()
        e2.record()
        g_agg.replay()
        e3.record()
        torch.cuda.synchronize()
        t_front += e0.elapsed_time(e1)
        t_choose += e1.elapsed_time(e2)
        t_agg += e2.elapsed_time(e3)
        nodes, labels = shards[i]
        n_pos = int((labels == 1).sum())
        sum_d = sum(int(data.graph.degrees(r)[nodes - data.graph.row_lo].sum()) for r in range(R))
        m_tot = int(sel.it_m[sel.it_rep.long()].sum().item())
        req = 8.0 * sum_d + R * batch * 16 + 4 * batch + 4.0 * m_tot
        req_choose += req
        alg_choose += req + 4.0 * P * n_pos * R
        alg_agg += (4.0 * F_ + 4.0) * m_tot + 4.0 * F_ * R * batch
        assert not sel.overflowed()
    kern = {
        "choose": {"ms": t_choose / K, "alg_bytes": alg_choose / K, "gbs": alg_choose / t_choose / 1e6,
                   "req_bytes": req_choose / K, "req_gbs": req_choose / t_choose / 1e6,
                   "launches_per_step": 2, "what": "the selection kernels k_choose_small || k_choose_wide (|| huge / big tiers)"},
        "aggregate": {"ms": t_agg / K, "alg_bytes": alg_agg / K, "gbs": alg_agg / t_agg / 1e6,
                      "req_bytes": alg_agg / K, "req_gbs": alg_agg / t_agg / 1e6, "launches_per_step": 1},
        "front": {"ms": t_front / K, "launches_per_step": 4,
                  "what": "k_pool_scores -> (k_choose_prep || pool sort || k_score_table) as in the step"},
    }
    dom = "choose" if t_choose >= t_agg else "aggregate"
    return kern, _roof(kern, dom, {"filter_plus_aggregate_gbs": (alg_choose + alg_agg) / (t_choose + t_agg) / 1e6,
                                   "filter_plus_aggregate_required_gbs": (req_choose + alg_agg) / (t_choose + t_agg) / 1e6},
                       workload=workload)


def hot_kernels_gcn(eng, agg_mod, data, shards, dev_nodes, cap, W, K, flush, dev):
    """C4: select-all + aggregate (rsqrt norm, self union) alone; bytes = (4F + 4) per neighbour row + output."""
    import torch
    from pcgnn_b200 import _lib

    F_ = data.feat.shape[1]
    st_nodes = dev_nodes[W].clone()
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for _ in range(2):
            eng.aggregate(eng.select_all(st_nodes, True, cap, _lib.NORM_RSQRT))
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with _lib.capture(g):
        sel = eng.select_all(st_nodes, True, cap, _lib.NORM_RSQRT)
        eng.aggregate(sel)
    t = alg = 0.0
    for s in range(K):
        i = W + s
        st_nodes.copy_(dev_nodes[i])
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        t += e0.elapsed_time(e1)
        nodes, _ = shards[i]
        sum_d = int(data.homo.degrees(0)[nodes].sum())
        alg += (4.0 * F_ + 4.0) * sum_d + 16.0 * len(nodes) + 4.0 * F_ * len(nodes)
        assert not sel.overflowed()
    kern = {"aggregate": {"ms": t / K, "alg_bytes": alg / K, "gbs": alg / t / 1e6, "launches_per_step": 2}}
    return kern, _roof(kern, "aggregate")


class _BatchRows:
    """Host view of a device-resident (row-partitioned) CSR restricted to the rows of some targets — all the
    reference ever touches (`adj_list[int(node)]` for the batch's nodes only, layers.py:219). Satisfies what
    oracle/port.py needs from a graph: n_rel and row(r, v)."""

    def __init__(self, graph, dev_graph, nodes):
        import torch

        self.n_rel = graph.n_rel
        indptr, indices = dev_graph
        self.rows = {}
        ip = graph.indptr
        for r in range(graph.n_rel):
            for v in np.unique(nodes):
                lv = int(v) - graph.row_lo
                b, e = int(ip[r * graph.n_nodes + lv]), int(ip[r * graph.n_nodes + lv + 1])
                self.rows[(r, int(v))] = indices[b:e].cpu().numpy()
        del torch

    def row(self, r, v):
        return self.rows[(r, int(v))]


def big_cpu_setup(args, dev):
    """C5 for the CPU arm: the partition is generated like the GPU arm generates it (on the GPU when there is one),
    then only the sampled batch rows, the feature table and the pool come to the host."""
    import torch
    from pcgnn_b200.synth_big import BigSpec, make_partition

    part = make_partition(BigSpec(nodes_per_rank=args.nodes_per_gpu, seed=SEED), 0, 1, dev)
    sample = min(args.cpu_sample, 64)           # the port (like the reference) builds a dense [B, U] mask: U ~ 3e5 here
    drawn = part.sample_batches(4, sample, SEED)
    batches = [(n.cpu().numpy().astype(np.int64), l.cpu().numpy()) for n, l in drawn]
    allnodes = np.concatenate([n for n, _ in batches])
    rows = _BatchRows(part.graph, part.graph.device(dev), allnodes)

    class D:
        pass

    d = D()
    d.feat = part.feat.cpu().numpy()
    d.graph = rows
    d.train_pos = part.train_pos.cpu().numpy().tolist()
    del part
    if torch.cuda.is_available():
        torch.cuda.empty_cache()
    return d, batches, sample


def run_reference(args):
    """--impl reference: the oracle port on the host cores, same config/metric/unit."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from pcgnn_b200.synth import make_graph

    spec, batch, embed, desc = WORKLOADS[args.workload]
    world = max(args.gpus, 1)
    if args.workload == "big":
        dev = torch.device("cuda", 0) if torch.cuda.is_available() else torch.device("cpu")
        data, batches, sample = big_cpu_setup(args, dev)
        params = init_params(data.feat.shape[1], embed, 3, SEED)
        note = ("oracle/port.py on %d targets per step with ONLY the batch rows of the CSR on the host (what the "
                "reference reads, layers.py:219); its dense [B,U] mask makes larger samples infeasible" % sample)
    else:
        data = make_graph(spec, seed=SEED)
        params = init_params(data.feat.shape[1], embed, data.graph.n_rel, SEED)
        batches = make_batches(data, 4, batch, SEED)
        sample = min(args.cpu_sample, batch)
        note = (f"full train step of oracle/port.py on the first {sample} targets of each {batch}-target batch "
                f"(Python loop per target like the reference)")
    rate, sec = cpu_port_rate(data, params, batches, sample, args.steps, args.warmup, gcn=args.workload.endswith("_gcn"))
    gb = batch if args.scaling == "strong" else batch * world
    line = {
        "impl": "reference", "metric": "train target-nodes/sec (fwd+bwd)", "value": rate, "unit": "target-nodes/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(desc, gb, world, args.scaling),
        "cpu_baseline": {"value": rate, "unit": "target-nodes/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": note + f"; host has {os.cpu_count()} cpus"},
        "e2e": {"value": rate, "unit": "target-nodes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def reference_loop_arm(data, params, host_nodes, host_labels, dev, W, K, flush, is_gcn, fast=False):
    """The reference's own training loop, unchanged (model_handler.py:124, :142-156), on a fresh model:
        optimizer = torch.optim.Adam(filter(requires_grad, params), lr, weight_decay)
        optimizer.zero_grad(); loss = model.loss(batch_nodes: list, Variable(cuda.LongTensor(batch_label)))
        loss.backward(); optimizer.step()            (+ loss.item(): the D2H of the step's result)
    Returns the summed CUDA-event ms of K steps (labels are numpy on the host when a step starts).
    fast: the same loop after ``pcgnn_b200.fastloop.enable()`` (loss.backward() hands out the replay's gradients without
    the autograd engine; optimizer.step() of the caller's torch.optim.Adam runs the package's one-kernel Adam)."""
    import torch
    from pcgnn_b200 import fastloop
    from pcgnn_b200.testing import build_cuda_pcgnn

    if fast:
        fastloop.enable()

    if is_gcn:
        model = build_cuda_gcn(data, params, dev)
    else:
        model = build_cuda_pcgnn(data.feat, data.graph, sorted(data.train_pos), params, rho=RHO, alpha=ALPHA, device=dev)
    opt = torch.optim.Adam(filter(lambda p: p.requires_grad, model.parameters()), lr=LR, weight_decay=WD)

    def step(i):
        opt.zero_grad()
        lab = torch.from_numpy(host_labels[i]).to(dev)              # model_handler.py:150 (cuda LongTensor of labels)
        loss = model.loss(host_nodes[i], lab)
        loss.backward()
        opt.step()
        return loss.item()

    for s_ in range(W):
        step(s_)
    torch.cuda.synchronize()
    evs = []
    for s_ in range(K):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step(W + s_)
        e1.record()
        evs.append((e0, e1))
    torch.cuda.synchronize()
    if fast:
        fastloop.disable()
    return sum(a.elapsed_time(b) for a, b in evs)


def dp_self_check(model, gstep, data, params, global_batches, shards, dev, rank, world, is_gcn):
    """Outside the timed region, world > 1: (1) the first step's loss, averaged over the ranks (equal shards), equals
    the loss of the whole global batch on ONE GPU (data parallel == large batch); (2) after the steps the replicas are
    bit-identical."""
    import torch
    import torch.distributed as dist
    from pcgnn_b200.testing import build_cuda_pcgnn

    n, l = shards[0]
    loss0 = gstep.run(n, l).clone()
    torch.cuda.synchronize()
    tot = loss0.double().clone()
    dist.all_reduce(tot)
    mean_loss = float(tot.item()) / world
    gn, gl = global_batches[0]
    if is_gcn:
        single = build_cuda_gcn(data, params, dev)
    else:
        single = build_cuda_pcgnn(data.feat, data.graph, sorted(data.train_pos), params, rho=RHO, alpha=ALPHA, device=dev)
        single.inter1.graph_cache = False
    want = float(single.loss(gn.tolist(), torch.from_numpy(gl).to(dev)).item())
    assert abs(mean_loss - want) <= 1e-5 * abs(want), f"data-parallel loss {mean_loss} != global-batch loss {want}"
    for i in range(1, 4):
        gstep.run(*shards[i])
    torch.cuda.synchronize()
    flat = torch.cat([p.detach().reshape(-1) for p in model.parameters() if p.requires_grad])
    every = [torch.empty_like(flat) for _ in range(world)]
    dist.all_gather(every, flat)
    assert all(torch.equal(every[0], e) for e in every), "replicas differ after data-parallel steps"
    if rank == 0:
        print(f"dp self-check ok: world {world}, step-1 loss {mean_loss:.7f} == global-batch loss {want:.7f}, "
              f"replicas bit-identical after 4 steps", file=sys.stderr)
    return mean_loss, want


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, loss, model):
    """What a caller of the timed train step ends up with after its last step: the step's loss over the global batch
    (`loss.npy`; with several GPUs the mean of the ranks' shard losses) and every trainable parameter after the step's
    optimizer update (`<parameter name>.npy`), float32. The inputs (graph, initial weights, batches) are seeded, so
    two builds run with the same arguments can be compared file by file."""
    arrays = {"loss": loss.detach().float().reshape(1)}
    arrays.update((name, p.detach().float()) for name, p in model.named_parameters() if p.requires_grad)
    total = sum(a.numel() * 4 for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs, more than the {DUMP_LIMIT_BYTES} allowed")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="yelp", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: the workload's batch per GPU; strong: the workload's batch in total, dealt to the GPUs")
    ap.add_argument("--check-only", action="store_true", help="world > 1: run the data-parallel self-check and exit")
    ap.add_argument("--cpu-sample", type=int, default=1024, help="targets per CPU-baseline step (bounded sample of a batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="do not use CUDA graphs for the device-resident step")
    ap.add_argument("--torch-adam", action="store_true",
                    help="NCCL all-reduce + torch.optim.Adam instead of the fused peer-memory exchange + Adam kernel")
    ap.add_argument("--nccl-scores", action="store_true",
                    help="workload big: exchange the score slices with an NCCL all-gather instead of peer-memory stores")
    ap.add_argument("--nodes-per-gpu", type=int, default=1_250_000, help="workload big: rows of the CSR held per GPU")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's loss (over the global batch) and the trained "
                         "parameters to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.check_only):
        ap.error("--dump-outputs needs the timed steps of --impl ours")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    from pcgnn_b200.parallel import FusedAdam, GradAllReduce, PeerComm
    from pcgnn_b200.synth import make_graph
    from pcgnn_b200.testing import build_cuda_pcgnn

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")        # keep NCCL's version banner off stdout (one JSON line)
        dist.init_process_group("nccl", device_id=dev)
    K, W = args.steps, max(args.warmup, 3)
    spec, wl_batch, embed, desc = WORKLOADS[args.workload]
    is_gcn = args.workload.endswith("_gcn")
    is_big = args.workload == "big"
    strong = args.scaling == "strong" and not is_big
    global_batch = wl_batch if strong else wl_batch * world
    if global_batch % world:
        raise SystemExit(f"global batch {global_batch} does not divide over {world} ranks")
    batch = global_batch // world                                  # targets per GPU
    n_b = W + K + 4
    if is_big:
        # C5: every rank generates and holds only its own row range of the CSR; features, scores and the pool
        # are global. Each rank draws its share of the global batch from its own nodes (targets live with
        # their rows), so the only exchanges per step are the score-slice all-gather and the gradient sum.
        from pcgnn_b200.synth_big import BigSpec, make_partition

        part = make_partition(BigSpec(nodes_per_rank=args.nodes_per_gpu, seed=SEED), rank, world, dev)
        data = part
        F_, R = part.feat.shape[1], part.graph.n_rel
        params = init_params(F_, embed, R, SEED)
        model = build_cuda_pcgnn_device(part.feat, part.graph, part.train_pos, params, dev)
        inter = model.inter1
        if world > 1:
            # self-check of the exchange: slice kernel + all-gather must equal the whole table computed locally
            e_ = inter.engine()
            e_.set_features(inter.features.weight)
            e_.score_table(inter.label_clf.weight, inter.label_clf.bias)
            whole = e_.score.clone()
            if args.nccl_scores:
                e_.score.zero_()
                e_.score_group = dist.group.WORLD          # slice kernel | NCCL all-gather (between two graphs)
            else:
                e_.enable_score_broadcast(dist.group.WORLD)  # slice kernel storing into every rank's table (one graph)
            e_.score_table(inter.label_clf.weight, inter.label_clf.bias)
            torch.cuda.synchronize()
            dist.barrier()
            assert torch.equal(whole, e_.score), "score exchange differs from the locally computed table"
            del whole
        drawn = part.sample_batches(n_b, batch, SEED + rank)
        shards = [(n.cpu().numpy().astype(np.int64), l.cpu().numpy()) for n, l in drawn]
        global_batches = None
        torch.cuda.synchronize()
        desc += f"; this run: {part.n_global} nodes, {int(part.graph.indptr[-1]) * world / 1e6:.0f}M CSR entries, pool {int(part.train_pos.shape[0])}"
    elif is_gcn:
        data = make_graph(spec, seed=SEED)
        F_, R = data.feat.shape[1], data.graph.n_rel
        params = init_params(F_, embed, R, SEED)
        model = build_cuda_gcn(data, params, dev)
        inter = model.enc.aggregator             # the module that owns the engine / slot capacity
    else:
        data = make_graph(spec, seed=SEED)
        F_, R = data.feat.shape[1], data.graph.n_rel
        params = init_params(F_, embed, R, SEED)
        model = build_cuda_pcgnn(data.feat, data.graph, sorted(data.train_pos), params, rho=RHO, alpha=ALPHA, device=dev)
        inter = model.inter1
    reducer = GradAllReduce(model.parameters()).attach()
    if args.torch_adam:     # NCCL all-reduce between two CUDA graphs + torch's fused Adam (the baseline arrangement)
        opt = torch.optim.Adam([p for p in model.parameters() if p.requires_grad], lr=LR, weight_decay=WD,
                               capturable=True, fused=True)
    else:                   # gradient exchange over NVLink peer memory + Adam in one kernel inside the step graph
        opt = FusedAdam(reducer, lr=LR, weight_decay=WD, comm=PeerComm(reducer.flat.numel()))
    fused = not args.torch_adam
    if not is_big:
        # global batches, identical on every rank; this rank's share dealt by total row length
        global_batches = make_batches(data, n_b, global_batch, SEED)
        weight = data.homo.degrees(0).astype(np.int64) if is_gcn else \
            sum(data.graph.degrees(r).astype(np.int64) for r in range(R))
        shards = [deal(n, l, weight, rank, world) for n, l in global_batches]
    dev_nodes = [torch.from_numpy(n.astype(np.int32)).to(dev) for n, _ in shards]
    dev_labels = [torch.from_numpy(l).to(dev) for _, l in shards]
    host_nodes = [n.tolist() for n, _ in shards]
    host_labels = [l for _, l in shards]
    if is_gcn:
        eng = inter._get_engine()
        eng.set_features(inter.features.weight)
        cap = max(inter.slots_bound(n) for n, _ in shards)
    else:
        eng = inter.engine()
        eng.set_features(inter.features.weight)
        cap = max(eng.slots_bound(n.astype(np.int32), inter.thresholds, RHO, True) for n, _ in shards)
    inter.cap_slots_hint = cap
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)      # > 126 MB L2

    def finish_step():
        if not fused:
            reducer()
            if world > 1:
                reducer.flat.div_(world)
        opt.step()                                               # fused: exchange + Adam + gradient clear

    def step_device_eager(i):
        if not fused:
            reducer.zero()
        loss = model.loss(dev_nodes[i], dev_labels[i])
        loss.backward()
        finish_step()
        return loss

    def step_host_eager(i):
        if not fused:
            reducer.zero()
        lab = torch.from_numpy(host_labels[i]).to(dev)
        loss = model.loss(host_nodes[i], lab)
        loss.backward()
        finish_step()
        return loss.item()                                       # D2H of the step's result

    use_graph = not args.no_graph
    gstep = None
    if use_graph:
        from pcgnn_b200.runtime import GraphedTrainStep

        gstep = GraphedTrainStep(model, opt, batch, cap, reducer=reducer, world=world, warmup_batch=shards[0])

        def step_device(i):
            return gstep.run_device(dev_nodes[i], dev_labels[i])

        def step_host(i):
            return gstep.run_item(shards[i][0], host_labels[i])        # host numpy ids + labels: H2D, replay, D2H loss
    else:
        step_device, step_host = step_device_eager, step_host_eager

    check = None
    if world > 1 and use_graph and not is_big:
        check = dp_self_check(model, gstep, data, params, global_batches, shards, dev, rank, world, is_gcn)
    if args.check_only:
        if world == 1 and rank == 0:
            print("dp self-check skipped: one GPU", file=sys.stderr)
        if world > 1:
            dist.destroy_process_group()
        return

    def timed(fn, first):
        """(summed event ms of K steps, what the last step returned)"""
        evs = []
        for s in range(K):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn(first + s)
            e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in evs), out

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    sampler = ClockSampler(local)
    # ---- device-resident inputs (value) ----
    for s in range(W):
        step_device(s)
    barrier()
    sampler.start()
    ms_dev, last_loss = timed(step_device, W)
    sampler.sample()
    barrier()
    ms_dev = max_over_ranks(ms_dev)
    if args.dump_outputs:
        # taken before the arms below train the same model further
        if gstep is not None and gstep.overflowed():
            raise SystemExit("--dump-outputs: a timed step overflowed its slot capacity, its outputs are incomplete")
        loss = last_loss.detach().float().reshape(1).clone()
        if world > 1:                  # equal shards: the mean of the ranks' losses is the loss of the global batch
            dist.all_reduce(loss)
            loss /= world
        if rank == 0:
            dump_outputs(args.dump_outputs, loss, model)
    # ---- host inputs through the step-graph API ----
    for s in range(W):
        step_host(s)
    barrier()
    ms_graph_host, _ = timed(step_host, W)
    barrier()
    ms_graph_host = max_over_ranks(ms_graph_host)
    if gstep is not None:
        assert not gstep.overflowed()
    # ---- host inputs through the REFERENCE's own loop (1 GPU: the reference is single-GPU) ----
    ms_ref_loop = ms_ref_loop_fast = None
    if world == 1 and not is_big:
        ms_ref_loop = reference_loop_arm(data, params, host_nodes, host_labels, dev, W, K, flush, is_gcn)
        ms_ref_loop_fast = None if is_gcn else \
            reference_loop_arm(data, params, host_nodes, host_labels, dev, W, K, flush, is_gcn, fast=True)
    sampler.stop_flag = True

    # ---- hot-path kernels alone (roofline), same batches. Each group is captured into its own CUDA graph
    # (static input buffers) so the events bracket GPU work only, not the host's launch calls. ----
    if hasattr(inter, "scores_external"):
        inter.scores_external = False
    kern, roof = hot_kernels_gcn(eng, inter, data, shards, dev_nodes, cap, W, K, flush, dev) if is_gcn else \
        hot_kernels_pcgnn(eng, inter, data, shards, dev_nodes, dev_labels, cap, W, K, flush, dev, batch, args.workload)

    # ---- the same steps from a device-resident epoch plan (one upload for all batches, no host work per step); last, and
    # guarded: an extra line of the report must never cost the report ----
    ms_plan = None
    if gstep is not None and fused and not is_big:
        try:
            gstep.load_plan([(shards[s][0], host_labels[s]) for s in range(W + K)])
            for s in range(W):
                gstep.run_planned()
            barrier()
            ms_plan, _ = timed(lambda i: gstep.run_planned(), W)
            barrier()
            ms_plan = max_over_ranks(ms_plan)
            assert not gstep.overflowed()
        except Exception as exc:          # noqa: BLE001
            print(f"epoch-plan arm skipped: {exc!r}", file=sys.stderr)
            ms_plan = None

    if rank == 0:
        total_nodes = global_batch * K
        io = {"h2d_bytes_per_step": batch * 4 + batch * 8, "d2h_bytes_per_step": 4}
        e2e_graph = {"value": total_nodes / (ms_graph_host / 1e3), "unit": "target-nodes/s", "ms_per_step": ms_graph_host / K,
                     "call": "runtime.GraphedTrainStep.run_item(numpy_ids, numpy_labels) -> float  (the host batch is packed into "
                             "one pinned buffer; ONE graph launch: the step's first kernel reads the 12 KB of ids / labels from "
                             "that pinned host memory over PCIe into HBM (pcg_pool_scores_stage), a copy kernel stores the loss "
                             "into a pinned word (pcg_stage); one event wait)", **io}
        line = {
            "metric": "train target-nodes/sec (fwd+bwd)", "value": total_nodes / (ms_dev / 1e3),
            "unit": "target-nodes/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_dev / K,
            "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": config_dict(desc, global_batch, world, "strong" if strong else "weak"),
            "e2e": e2e_graph,
            "gpu_launches": (GCN_KERNELS_PER_STEP if is_gcn else MY_KERNELS_PER_STEP) * K,
            "mode": "cuda-graph replay (runtime.GraphedTrainStep)" if use_graph else "eager",
            "roofline": roof, "kernels": kern, "clocks": sampler.result(),
        }
        if ms_plan is not None:
            line["e2e_epoch_plan"] = {
                "value": total_nodes / (ms_plan / 1e3), "unit": "target-nodes/s", "ms_per_step": ms_plan / K,
                "call": "runtime.GraphedTrainStep.load_plan(all batches) once, then run_planned() per step: the recorded step "
                        "fetches its batch from the device-resident plan through a device cursor and files its loss in a "
                        "device array (no host data per step)",
                "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
        if ms_ref_loop is not None:
            line["e2e_reference_loop"] = {
                "value": total_nodes / (ms_ref_loop / 1e3), "unit": "target-nodes/s", "ms_per_step": ms_ref_loop / K,
                "call": "the reference's loop unchanged (model_handler.py:124, :142-156): torch.optim.Adam; opt.zero_grad(); "
                        "model.loss(list_of_ids, cuda LongTensor(labels)); backward(); opt.step(); loss.item() -- served by "
                        "the package's CUDA-graph cache; host-bound: torch's Adam.step and the autograd engine are ~60% "
                        "of it (profiles/replay_cost.py)", **io}
            if ms_ref_loop_fast is not None:
                line["e2e_reference_loop_fast"] = {
                    "value": total_nodes / (ms_ref_loop_fast / 1e3), "unit": "target-nodes/s",
                    "ms_per_step": ms_ref_loop_fast / K,
                    "call": "the same unchanged loop after pcgnn_b200.fastloop.enable(): loss.backward() stores the replay's "
                            "gradients without the autograd engine, the caller's torch.optim.Adam.step() runs the package's "
                            "one-kernel Adam through a pre-step hook", **io}
        if check is not None:
            line["dp_self_check"] = {"step1_loss_mean_over_ranks": check[0], "global_batch_loss_one_gpu": check[1],
                                     "replicas_bit_identical": True}
        if world == 1 and not args.no_cpu_baseline:
            if is_big:
                del model, gstep
                torch.cuda.empty_cache()
                cdata, cbatches, sample = big_cpu_setup(args, dev)
                rate, sec = cpu_port_rate(cdata, params, cbatches, sample, 3, 1)
                note = (f"3 full train steps of oracle/port.py on {sample} targets each ({sec * 1e3:.0f} ms each) with only "
                        f"the batch rows of the CSR on the host (what the reference reads, layers.py:219)")
            else:
                sample = min(args.cpu_sample, batch)
                rate, sec = cpu_port_rate(data, params, global_batches, sample, 12, 1, gcn=is_gcn)
                note = (f"12 full train steps of oracle/port.py on the first {sample} targets of a batch "
                        f"({sec * 1e3:.0f} ms each)")
            line["cpu_baseline"] = {"value": rate, "unit": "target-nodes/s", "cores": torch.get_num_threads(),
                                    "kind": "port", "sample": note + f"; host has {os.cpu_count()} cpus"}
            if not is_gcn and not is_big:
                line["cpu_baseline"]["c_port_choose_aggregate_nodes_per_s"] = c_port_rate(data, global_batches)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

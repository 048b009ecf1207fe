"""Evaluation pass on the idx_rest set at B = 1024: three ways to score it and compute its metrics, timed on the GPU.

  python profiles/bench_eval.py --workload {yelp,amazon,amazon_gcn,amazon_sage} [--passes 30] [--warmup 5] --out DIR

  yelp / amazon  PC-GNN (PCALayer) on the C2 / C1 graphs
  amazon_gcn     GCN(GCNEncoder(GCNAggregator)) on the C1 graph's union (C4)
  amazon_sage    GraphSage(Encoder(MeanAggregator), gcn=True), the reference's build (model_handler.py:97-98), on the
                 same union graph

  utils_test    utils.test as it is (the reference's loop: model.to_prob(list, labels) per batch with grad enabled,
                then metrics.binary_metrics)
  no_grad_loop  the same loop under torch.no_grad() (PC-GNN: one cached infer-graph replay + a pinned upload per batch;
                the baselines: their module path per batch, a pinned upload, the select-all, aggregate and encoder
                kernels, then torch's head and to_prob)
  eval_pass     runtime.GraphedEvalPass.run() (ids uploaded once; n batch-graph replays, one metrics graph, one wait)

Every timed pass ends in a synchronise (host clock around it). max_abs_dprob compares each variant's to_prob output with
that of utils.test's loop body (log-probabilities for amazon_sage). The card's name and power limit are read with nvidia-smi in the same run. The whole
working set (C2: 45,954 x 32 fp32 features and an 8.0M-entry CSR, about 39 MB) stays in the 126 MB L2 across passes: the
numbers are warm-cache numbers, which is the regime of a validation pass inside a training run. The same holds for the
union graph of the baselines (11,944 x 25 features, an 8.5M-entry CSR, about 36 MB).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)

B = 1024
E = 64


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [x.strip() for x in q.split(",")]
    return {"name": name, "power_limit": power, "sm_max_clock": clock}


def build_baseline(d, sage, xavier):
    """GCN or GraphSage (MeanAggregator, Encoder(gcn=True)) on the union graph, frozen feature table, E = 64."""
    import torch
    import torch.nn as nn

    from pcgnn_b200 import graphsage as gs

    F_ = d.feat.shape[1]
    features = nn.Embedding(*d.feat.shape)
    features.weight = nn.Parameter(torch.from_numpy(np.ascontiguousarray(d.feat)), requires_grad=False)
    features = features.cuda()
    if sage:
        enc = gs.Encoder(features, F_, E, d.homo, gs.MeanAggregator(features, cuda=True), gcn=True, cuda=True)
        model = gs.GraphSage(2, enc)
    else:
        enc = gs.GCNEncoder(features, F_, E, d.homo, gs.GCNAggregator(features, cuda=True), cuda=True)
        model = gs.GCN(2, enc)
    with torch.no_grad():
        enc.weight.copy_(torch.from_numpy(xavier(E, F_)))
        model.weight.copy_(torch.from_numpy(xavier(2, E)))
    return model.cuda()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", choices=["yelp", "amazon", "amazon_gcn", "amazon_sage"], default="yelp")
    ap.add_argument("--passes", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    if a.passes < 20:
        raise SystemExit("--passes: at least 20 timed passes")

    import torch

    from pcgnn_b200.runtime import GraphedEvalPass
    from pcgnn_b200.synth import make_graph
    from pcgnn_b200.testing import build_cuda_pcgnn
    from pcgnn_b200.utils import test as utils_test

    if not torch.cuda.is_available():
        raise SystemExit("bench_eval.py measures on a CUDA device; none is visible")
    torch.cuda.set_device(0)
    info = gpu_info()
    baseline = a.workload in ("amazon_gcn", "amazon_sage")
    d = make_graph("amazon" if baseline else a.workload, seed=72)
    rng = np.random.default_rng(72)
    F_ = d.feat.shape[1]

    def xavier(r, c):
        lim = np.sqrt(6.0 / (r + c))
        return rng.uniform(-lim, lim, size=(r, c)).astype(np.float32)

    if baseline:
        model = build_baseline(d, a.workload == "amazon_sage", xavier)
    else:
        params = dict(intra=[xavier(2 * F_, E) for _ in range(d.graph.n_rel)], inter=xavier(F_ + d.graph.n_rel * E, E),
                      clf_w=xavier(2, F_), clf_b=np.zeros(2, np.float32), head=xavier(2, E))
        model = build_cuda_pcgnn(d.feat, d.graph, sorted(d.train_pos), params)
    nodes = [int(v) for v in d.idx_rest]
    labels = np.asarray(d.labels[d.idx_rest])
    n = len(nodes)

    def loop_probs(no_grad):
        out = []
        ctx = torch.no_grad() if no_grad else torch.enable_grad()
        with ctx:
            for s in range(0, n, B):
                p = model.to_prob(nodes[s:s + B], labels[s:s + B], train_flag=False)
                out.append((p[0] if isinstance(p, tuple) else p).detach())
        return torch.cat(out)

    ev = GraphedEvalPass(model, nodes, labels, B)

    def no_grad_loop():
        with torch.no_grad():
            utils_test(nodes, labels, model, B, print_line=False)

    variants = {
        "utils_test": lambda: utils_test(nodes, labels, model, B, print_line=False),
        "no_grad_loop": no_grad_loop,
        "eval_pass": ev.run,
    }
    for fn in variants.values():
        for _ in range(a.warmup):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in variants}
    for _ in range(a.passes):                     # alternate the variants: drift on a shared host hits all of them
        for k, fn in variants.items():
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            times[k].append(time.perf_counter() - t0)

    ref = loop_probs(False)
    probs = {"utils_test": ref, "no_grad_loop": loop_probs(True), "eval_pass": ev.probs()}
    m = ev.run()
    auc, recall, f1_macro, precision = utils_test(nodes, labels, model, B, print_line=False)
    res = {
        "workload": a.workload, "nodes": n, "batch": B, "batches": -(-n // B), "passes": a.passes, "warmup": a.warmup,
        "gpu": info, "l2": "working set L2-resident across passes (warm cache)",
        "variants": {},
        "eval_pass_metrics": m,
        "utils_test_metrics": {"auc": auc, "recall": recall, "f1_macro": f1_macro, "precision": precision},
    }
    for k, ts in times.items():
        ts = np.asarray(ts) * 1e3
        res["variants"][k] = {"ms_median": float(np.median(ts)), "ms_min": float(ts.min()), "ms_max": float(ts.max()),
                              "nodes_per_s": float(n / (np.median(ts) * 1e-3)),
                              "max_abs_dprob": float((probs[k] - ref).abs().max())}
    base = res["variants"]["utils_test"]["ms_median"]
    for k in res["variants"]:
        res["variants"][k]["speedup_vs_utils_test"] = base / res["variants"][k]["ms_median"]
    os.makedirs(a.out, exist_ok=True)
    path = os.path.join(a.out, f"bench_eval_{a.workload}.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: (v["ms_median"], v["max_abs_dprob"]) for k, v in res["variants"].items()}), info)


if __name__ == "__main__":
    main()

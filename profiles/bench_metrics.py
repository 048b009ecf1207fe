"""Cost of the device metrics: pcg_binary_metrics recorded as a CUDA graph (the metrics graph of GraphedEvalPass.run()),
the same graph with operating-point requests, and the eager curve read (GraphedEvalPass.curve() / metrics.device_curve
after the metrics), at n nodes.

  python profiles/bench_metrics.py [--sizes 27572,1000000,10000000] [--reps 50] [--warmup 5] --out DIR

  metrics_graph  one replay of a graph holding pcg_binary_metrics (sort, counts, best cuts, AP terms, final), CUDA
                 events around each replay
  points_graph   one replay of a graph holding pcg_binary_metrics then pcg_binary_points with 8 mixed requests
                 (GraphedEvalPass(..., operating_points=POINTS)), CUDA events; replays alternate with metrics_graph
  points_kernels pcg_binary_points alone (k_points_area + k_points_final) over the workspace the metrics left, CUDA
                 events
  curve          pcg_binary_curve (k_curve_scan + k_curve_write) over the workspace the metrics left, then the 8-byte
                 read of G: host clock around the call, which ends in that read (a synchronise)
  curve_kernels  the same two launches alone, CUDA events

Inputs: prob[1] uniform fp32 (almost all scores distinct, so G is close to n: the largest curve), 12 % positives, from
a fixed seed. n = 27,572 is the C2 validation set. Scores, labels and workspace are reused across repetitions, so up to
n = 10^6 the working set stays in the 126 MB L2 (warm cache); at 10^7 it does not (360 MB of workspace). The
card's name and power limit are read with nvidia-smi in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

# 8 mixed requests: review budgets, false-alarm ceilings and partial-AUC limits a fraud team would ask for
POINTS = dict(top_k=[100, 1000], fpr=[0.001, 0.01, 0.1], max_fpr=[0.01, 0.1, 1.0])

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="27572,1000000,10000000")
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    if a.reps < 20:
        raise SystemExit("--reps: at least 20 timed repetitions")

    import torch

    from bench_eval import gpu_info
    from pcgnn_b200 import _lib
    from pcgnn_b200.metrics import _curve_buffers, _point_requests, _read_curve

    if not torch.cuda.is_available():
        raise SystemExit("bench_metrics.py measures on a CUDA device; none is visible")
    torch.cuda.set_device(0)
    info = gpu_info()
    L = _lib.lib()
    res = {"gpu": info, "reps": a.reps, "warmup": a.warmup, "sizes": {}}
    for n in (int(x) for x in a.sizes.split(",")):
        rng = np.random.default_rng(n)
        prob = torch.from_numpy(rng.random((2, n), dtype=np.float32)).cuda()
        y = torch.from_numpy((rng.random(n) < 0.12).astype(np.int32)).cuda()
        ws = torch.empty(int(L.pcg_binary_metrics_workspace_bytes(n)), dtype=torch.uint8, device="cuda")
        out = torch.empty(_lib.METRICS_WORDS, dtype=torch.float64, device="cuda")
        bufs = _curve_buffers(n, prob.device)
        kind, arg = _point_requests(n, **POINTS)
        n_req = len(kind)
        kind_d, arg_d = torch.from_numpy(kind).cuda(), torch.from_numpy(arg).cuda()
        pws = torch.empty(int(L.pcg_binary_points_workspace_bytes(n, n_req)), dtype=torch.uint8, device="cuda")
        pts = torch.empty(n_req * _lib.POINT_WORDS, dtype=torch.float64, device="cuda")

        def metrics():
            _lib.check(L.pcg_binary_metrics(prob.data_ptr(), y.data_ptr(), n, out.data_ptr(), ws.data_ptr(), ws.numel(),
                                            _lib.stream_ptr()), "pcg_binary_metrics")

        def points():
            _lib.check(L.pcg_binary_points(ws.data_ptr(), ws.numel(), n, kind_d.data_ptr(), arg_d.data_ptr(), n_req,
                                           pts.data_ptr(), pws.data_ptr(), pws.numel(), _lib.stream_ptr()),
                       "pcg_binary_points")

        def metrics_points():
            metrics()
            points()

        def curve_kernels():
            thr, tp, fp, count = bufs
            _lib.check(L.pcg_binary_curve(ws.data_ptr(), ws.numel(), n, thr.data_ptr(), tp.data_ptr(), fp.data_ptr(),
                                          count.data_ptr(), _lib.stream_ptr()), "pcg_binary_curve")

        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            metrics_points()                            # warm-up launches outside the capture
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with _lib.capture(g):
            metrics()
        gp = torch.cuda.CUDAGraph()
        with _lib.capture(gp):
            metrics_points()
        for _ in range(a.warmup):
            gp.replay()
            g.replay()
            _read_curve(ws, n, bufs)
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(4)]
        t_graph, t_pgraph, t_pkern, t_curve, t_kern = [], [], [], [], []
        G = None
        for _ in range(a.reps):
            ev[2][0].record()
            gp.replay()
            ev[2][1].record()
            torch.cuda.synchronize()
            t_pgraph.append(ev[2][0].elapsed_time(ev[2][1]))
            ev[3][0].record()
            points()
            ev[3][1].record()
            torch.cuda.synchronize()
            t_pkern.append(ev[3][0].elapsed_time(ev[3][1]))
            ev[0][0].record()
            g.replay()
            ev[0][1].record()
            torch.cuda.synchronize()
            t_graph.append(ev[0][0].elapsed_time(ev[0][1]))
            t0 = time.perf_counter()
            G = int(_read_curve(ws, n, bufs)[0].numel())
            t_curve.append((time.perf_counter() - t0) * 1e3)
            ev[1][0].record()
            curve_kernels()
            ev[1][1].record()
            torch.cuda.synchronize()
            t_kern.append(ev[1][0].elapsed_time(ev[1][1]))
        m = dict(zip(_lib.METRICS_KEYS, out.cpu().tolist()))
        row = {"groups": G, "n_pos": m["n_pos"], "ap": m["ap"], "recall_at_k": m["recall_at_k"],
               "points": POINTS, "point_words": pts.cpu().tolist()}
        for k, ts in (("metrics_graph", t_graph), ("points_graph", t_pgraph), ("points_kernels", t_pkern),
                      ("curve", t_curve), ("curve_kernels", t_kern)):
            ts = np.asarray(ts)
            row[k] = {"ms_median": float(np.median(ts)), "ms_min": float(ts.min()), "ms_max": float(ts.max())}
        res["sizes"][str(n)] = row
        print(n, json.dumps({k: row[k]["ms_median"] for k in ("metrics_graph", "points_graph", "points_kernels", "curve",
                                                             "curve_kernels")}), flush=True)
        del g, gp
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bench_metrics.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(info))


if __name__ == "__main__":
    main()

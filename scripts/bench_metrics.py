"""Time one scan's evaluation metric set on the GPU (lidiff_b200.metrics) and check it against the previous shim path and the CPU
oracle on the same inputs.

    python scripts/bench_metrics.py --out <dir> [--repeats 5]

The pair is synthetic and eval-sized (real SemanticKITTI crop sizes are not at hand):
  * "ground truth": 12 synthetic KITTI-shaped scans (lidiff_b200.synth.synthetic_scan, 131 k points each) with 3 cm jitter, cut to
    z in (-4, 4.4) and to 50 m range -> ~1.5 M points;
  * "prediction": 6 x 180 k points resampled from 6 of those scans with 5 cm jitter (6 offsets per point after refinement), 2 % of
    them moved 20 m up (outside the ground truth's z crop) -> 1.08 M points.
Parts, each timed with CUDA events after warm-up (median of --repeats): both nearest-distance directions, precision / recall counts at
100 thresholds (both directions), the voxel histograms at 0.5 / 0.2 / 0.1 m (IoU; the 0.5 m call also yields JSD 3D and BEV), and
the whole set as lidiff_b200.tools.eval_path runs it through the metric classes (host copies and arithmetic included).
Writes <out>/bench_metrics.json with the GPU name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from lidiff_b200 import metrics as m  # noqa: E402
from lidiff_b200.synth import synthetic_scan  # noqa: E402


def make_pair():
    g = np.random.default_rng(0)
    scans = [synthetic_scan(s) for s in range(12)]
    gt = np.concatenate(scans) + g.normal(size=(sum(len(s) for s in scans), 3)) * 0.03
    gt = gt[(gt[:, 2] > -4.0) & (gt[:, 2] < 4.4) & (np.sqrt((gt ** 2).sum(1)) < 50.0)]
    pred = np.concatenate([s[g.integers(0, len(s), 180000)] for s in scans[:6]])
    pred = pred + g.normal(size=pred.shape) * 0.05
    out = g.random(len(pred)) < 0.02
    pred[out, 2] += 20.0
    return gt, pred


def timed(fn, repeats, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), ts, out


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable: {e}"
    return {"torch_device_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--no-shim", action="store_true", help="skip the previous shim path (_knn) comparison")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    res = {"gpu": gpu_info()}
    gt_np, pred_np = make_pair()
    res["sizes"] = {"ground_truth": len(gt_np), "prediction": len(pred_np)}
    gt, pred = m._cloud(gt_np), m._cloud(pred_np)
    thr = np.linspace(0.05, 0.1, 100)
    parts = {}
    parts["nn_pred_to_gt"], _, d_pg = timed(lambda: m.nn_distance(pred, gt), args.repeats)
    parts["nn_gt_to_pred"], _, d_gp = timed(lambda: m.nn_distance(gt, pred), args.repeats)
    parts["pr_counts_both"], _, cnts = timed(lambda: (m.threshold_counts(d_pg, thr), m.threshold_counts(d_gp, thr)), args.repeats)
    hist = {}
    for v in (0.5, 0.2, 0.1):
        parts[f"voxel_hist_{v}"], _, hist[v] = timed(lambda v=v: m.voxel_hist_compare(gt, pred, v, 50.0), args.repeats)

    def cli_set():                                      # one scan of tools/eval_path.py
        h = m.voxel_hist_compare(gt, pred, 0.5, 50.)
        rm, iou, cd, pr = m.RMSE(), m.CompletionIoU(), m.ChamferDistance(), m.PrecisionRecall(0.05, 0.1, 100)
        for o in (rm, iou, cd, pr):
            o.update(gt, pred)
        return h, rm.compute(), iou.compute(), cd.compute(), pr.compute_auc()
    parts["eval_path_scan_total"], ts, cli = timed(cli_set, args.repeats)
    res["ms"] = parts
    res["ms_kernel_parts_sum"] = sum(v for k, v in parts.items() if k != "eval_path_scan_total")
    res["eval_path_scan_total_all_repeats_ms"] = ts
    d_pg1 = m.nn_distance(pred, gt).cpu().numpy()
    d_pg = d_pg.cpu().numpy()
    d_gp = d_gp.cpu().numpy()
    res["repeat_bit_identical"] = bool(np.array_equal(d_pg, d_pg1)) and m.voxel_hist_compare(gt, pred, 0.1, 50.0) == hist[0.1]
    res["values"] = {"rmse": float(cli[1][0]), "chamfer": float(cli[3][0]), "iou": {str(k): float(v) for k, v in cli[2].items()},
                     "pr_re_f1_auc": [float(x) for x in cli[4]], "jsd_3d": hist[0.5]["jsd_3d"], "jsd_bev": hist[0.5]["jsd_bev"],
                     "hist": {str(k): v for k, v in hist.items()}}

    # the same inputs through the CPU oracle (scipy k-d tree + sparse histograms)
    sys.path.insert(0, ROOT)
    from oracle import metrics as om
    t0 = time.time()
    o_pg, o_gp = om.nn_distance(pred_np, gt_np), om.nn_distance(gt_np, pred_np)
    t_nn = time.time() - t0
    t0 = time.time()
    o_hist = {v: om.hist_compare(gt_np, pred_np, v, 50.0) for v in (0.5, 0.2, 0.1)}
    t_hist = time.time() - t0
    chk = {"nn_max_abs_diff_vs_kdtree": float(max(np.abs(d_pg - o_pg).max(), np.abs(d_gp - o_gp).max())),
           "threshold_counts_equal": bool(np.array_equal(cnts[0], [(d_pg < t).sum() for t in thr])
                                          and np.array_equal(cnts[1], [(d_gp < t).sum() for t in thr])),
           "occupancy_equal": all(hist[v][k] == o_hist[v][k] for v in hist for k in ("n_a", "n_b", "occ_a", "occ_b", "occ_ab")),
           "jsd_max_rel_diff": max(abs(hist[v][k] - o_hist[v][k]) / abs(o_hist[v][k]) for v in hist for k in ("jsd_3d", "jsd_bev"))}
    res["oracle_cpu_s"] = {"nn_both_kdtree": t_nn, "sparse_hist_3_sizes": t_hist, "cpu_count": os.cpu_count()}

    if not args.no_shim:                               # the open3d shim's previous GPU path: bucketed fp32 cdist + fp64 re-evaluation
        from lidiff_b200.shims.open3d.geometry import _knn

        def shim(q, r):
            _, idx = _knn(q.float(), r.float(), 1)
            return (q - r[idx[:, 0]]).norm(dim=1)
        t_shim, _, s_pg = timed(lambda: shim(pred, gt), 1, warmup=1)
        t_shim2, _, s_gp = timed(lambda: shim(gt, pred), 1, warmup=0)
        res["shim_knn_ms"] = {"nn_pred_to_gt": t_shim, "nn_gt_to_pred": t_shim2}
        chk["shim_max_abs_diff"] = float(max(np.abs(s_pg.cpu().numpy() - d_pg).max(), np.abs(s_gp.cpu().numpy() - d_gp).max()))
    res["checks"] = chk
    line = json.dumps(res)
    print(line)
    with open(os.path.join(args.out, "bench_metrics.json"), "w") as f:
        f.write(json.dumps(res, indent=1) + "\n")
    ok = (chk["nn_max_abs_diff_vs_kdtree"] <= 1e-9 and chk["threshold_counts_equal"] and chk["occupancy_equal"]
          and chk["jsd_max_rel_diff"] <= 1e-12 and res["repeat_bit_identical"])
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()

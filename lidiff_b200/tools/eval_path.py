"""Evaluation of completed scans against the accumulated sequence map — counterpart of the reference's
`python lidiff/utils/eval_path.py -p <results>/refine/` with the same options, the same per-scan output lines and the same
`res_log.yaml` (JSON) keys, every metric computed on the GPU (lidiff_b200.metrics).

    python -m lidiff_b200.tools.eval_path -p results/exp/refine/ --data ./Datasets/SemanticKITTI/dataset/sequences/08
    python -m lidiff_b200.tools.eval_path -d diff.ckpt -r refine.ckpt -t 50 --data <sequence>     # complete the scans first
    python -m lidiff_b200.tools.eval_path --random-weights -t 2 --data <sequence>                 # plumbing, no checkpoints

Without -d / --random-weights the prediction of scan `velodyne/<n>.bin` is `<path>/<n>.ply` (the `refine/` directory that
lidiff_b200.tools.diff_completion_pipeline writes); otherwise DiffCompletion completes the scan and its refined cloud is scored.
The ground truth is the sequence's `map_clean.npy` cropped at max_range around the scan's pose (poses.txt, corrected by calib.txt's
Tr as Tr^-1 P Tr), moved into the scan frame, cut to z in (-4, 4.4) and to the 10 m voxels the input scan occupies.
res_log.yaml goes to the directory part of --path (its parent for a path without a trailing slash).
"""
from __future__ import annotations

import json
import os
import re

import click
import numpy as np
import torch

from .. import metrics
from ..synth import read_ply_xyz

PATH_DATA = "./Datasets/SemanticKITTI/dataset/sequences/08"


def _natural(names):
    return sorted(names, key=lambda s: [int(t) if t.isdigit() else t for t in re.split(r"(\d+)", s)])


def _matrix(values):
    pose = np.zeros((4, 4))
    pose[0, 0:4] = values[0:4]
    pose[1, 0:4] = values[4:8]
    pose[2, 0:4] = values[8:12]
    pose[3, 3] = 1.0
    return pose


def parse_calibration(filename):
    calib = {}
    with open(filename) as f:
        for line in f:
            key, content = line.strip().split(":")
            calib[key] = _matrix([float(v) for v in content.strip().split()])
    return calib


def load_poses(calib_fname, poses_fname):
    """poses.txt rows as 4x4 matrices, as Tr^-1 . P . Tr when calib.txt exists"""
    tr_inv = tr = None
    if os.path.exists(calib_fname):
        tr = parse_calibration(calib_fname)["Tr"]
        tr_inv = np.linalg.inv(tr)
    poses = []
    with open(poses_fname) as f:
        for line in f:
            pose = _matrix([float(v) for v in line.strip().split()])
            poses.append(np.matmul(tr_inv, np.matmul(pose, tr)) if tr is not None else pose)
    return poses


def read_scan(bin_file, max_range):
    """(raw (n,4) float32 scan, input points (m,3) float32 closer than max_range)"""
    points = np.fromfile(bin_file, dtype=np.float32).reshape(-1, 4)
    dist = np.sqrt(np.sum(points[:, :3] ** 2, axis=-1))
    return points, points[dist < max_range, :3]


def read_prediction(ply_file, max_range):
    points = read_ply_xyz(ply_file)
    dist = np.sqrt(np.sum(points ** 2, axis=-1))
    return points[dist < max_range]


def ground_truth(pose, cur_scan, seq_map: torch.Tensor, max_range, viewpoint_voxel=10.0) -> torch.Tensor:
    """(k,3) fp64 CUDA tensor: map points closer than max_range to the pose's translation, in the scan frame, z in (-4, 4.4), in a
    voxel of the scan's viewpoint grid (open3d VoxelGrid.create_from_point_cloud: origin = min bound - half a voxel)"""
    dev = seq_map.device
    pose_t = torch.from_numpy(pose).to(dev)
    keep = torch.sum((seq_map - pose_t[:-1, -1]) ** 2, dim=-1) ** .5 < max_range
    gt = seq_map[keep]
    gt = (torch.cat((gt, torch.ones((gt.shape[0], 1), dtype=gt.dtype, device=dev)), dim=-1) @ torch.linalg.inv(pose_t).T)[:, :3]
    gt = gt[(gt[:, 2] > -4.) & (gt[:, 2] < 4.4)]
    scan = torch.as_tensor(np.asarray(cur_scan, dtype=np.float64), device=dev)
    if scan.shape[0] == 0 or gt.shape[0] == 0:
        return gt[:0]
    origin = scan.min(0).values - 0.5 * viewpoint_voxel
    vs = torch.floor((scan - origin) / viewpoint_voxel).long()
    vg = torch.floor((gt - origin) / viewpoint_voxel).long()
    lo = torch.minimum(vs.min(0).values, vg.min(0).values)
    span = torch.maximum(vs.max(0).values, vg.max(0).values) - lo + 1
    enc = lambda v: ((v[:, 0] - lo[0]) * span[1] + (v[:, 1] - lo[1])) * span[2] + (v[:, 2] - lo[2])
    return gt[torch.isin(enc(vg), torch.unique(enc(vs)))].contiguous()


@click.command()
@click.option("--path", "-p", type=str, default="", help="path to the scan sequence")
@click.option("--voxel_size", "-v", type=float, default=0.05, help="voxel size")
@click.option("--max_range", "-m", type=float, default=50, help="max range")
@click.option("--denoising_steps", "-t", type=int, default=50, help="number of denoising steps")
@click.option("--cond_weight", "-s", type=float, default=6.0, help="conditioning weights")
@click.option("--diff", "-d", type=str, help="run diffusion pipeline")
@click.option("--refine", "-r", type=str, help="path to the checkpoint for refinement net")
@click.option("--data", type=str, default=PATH_DATA, help="sequence directory (velodyne/, poses.txt, calib.txt, map_clean.npy)")
@click.option("--random-weights", is_flag=True, help="complete the scans with seeded random parameters instead of checkpoints")
def main(path, voxel_size, max_range, denoising_steps, cond_weight, diff, refine, data, random_weights):
    device = torch.device("cuda", torch.cuda.current_device())
    diff_completion = None
    if random_weights or diff:
        from ..pipeline import DiffCompletion
        if random_weights:
            from ..weights import random_state_dict
            sds = {k: random_state_dict(k, i) for i, k in enumerate(("enc", "diff", "refine"))}
            diff_completion = DiffCompletion(state_dicts=sds, denoising_steps=denoising_steps, cond_weight=cond_weight, device=device)
        else:
            diff_completion = DiffCompletion(diff, refine, denoising_steps, cond_weight, device=device)

    completion_iou = metrics.CompletionIoU()
    rmse = metrics.RMSE()
    chamfer_distance = metrics.ChamferDistance()
    precision_recall = metrics.PrecisionRecall(0.05, 2 * 0.05, 100)

    poses = load_poses(os.path.join(data, "calib.txt"), os.path.join(data, "poses.txt"))
    seq_map = torch.from_numpy(np.load(os.path.join(data, "map_clean.npy"))[:, :3].astype(np.float64)).to(device)
    jsd_3d, jsd_bev = [], []
    for pose, scan_name in zip(poses, _natural(os.listdir(os.path.join(data, "velodyne")))):
        raw, cur_scan = read_scan(os.path.join(data, "velodyne", scan_name), max_range)
        if diff_completion is None:
            pred = metrics._cloud(read_prediction(os.path.join(path, f'{scan_name.split(".")[0]}.ply'), max_range), device)
        else:
            refined, _ = diff_completion.complete_scan(raw)
            pred = metrics._cloud(refined, device)
        gt = ground_truth(pose, cur_scan, seq_map, max_range)

        hist = metrics.voxel_hist_compare(gt, pred, 0.5, 50.)          # compute_hist_metrics(gt, pred, bev=False / True)
        jsd_3d.append(hist["jsd_3d"])
        jsd_bev.append(hist["jsd_bev"])
        print(f"JSD 3D: {jsd_3d[-1]}")
        print(f"JSD BEV: {jsd_bev[-1]}")

        rmse.update(gt, pred)
        completion_iou.update(gt, pred)
        chamfer_distance.update(gt, pred)
        precision_recall.update(gt, pred)

        rmse_mean, rmse_std = rmse.compute()
        print(f"RMSE Mean: {rmse_mean}\tRMSE Std: {rmse_std}")
        thr_ious = completion_iou.compute()
        for v_size in thr_ious.keys():
            print(f"Voxel {v_size}cm IOU: {thr_ious[v_size]}")
        cd_mean, cd_std = chamfer_distance.compute()
        print(f"CD Mean: {cd_mean}\tCD Std: {cd_std}")
        pr, re_, f1 = precision_recall.compute_auc()
        print(f"Precision: {pr}\tRecall: {re_}\tF-Score: {f1}")

    print("\n\n=================== FINAL RESULTS ===================\n\n")
    print(f"JSD 3D: {np.array(jsd_3d).mean()}")
    print(f"JSD BEV: {np.array(jsd_bev).mean()}")
    print(f"RMSE Mean: {rmse_mean}\tRMSE Std: {rmse_std}")
    thr_ious = completion_iou.compute()
    for v_size in thr_ious.keys():
        print(f"Voxel {v_size}cm IOU: {thr_ious[v_size]}")
    cd_mean, cd_std = chamfer_distance.compute()
    print(f"CD Mean: {cd_mean}\tCD Std: {cd_std}")
    pr, re_, f1 = precision_recall.compute_auc()
    print(f"Precision: {pr}\tRecall: {re_}\tF-Score: {f1}")

    res_dict = {
        "jsd": float(np.array(jsd_bev).mean()),
        "jsd_noclip_3d": float(np.array(jsd_3d).mean()),
        "rmse_mean": float(rmse_mean), "rmse_std": float(rmse_std),
        "ious": {str(k): float(v) for k, v in thr_ious.items()},
        "cd_mean": float(cd_mean), "cd_std": float(cd_std),
        "pr": float(pr), "re": float(re_), "f1": float(f1),
    }
    log_dir = os.path.dirname(path) or "."
    with open(os.path.join(log_dir, "res_log.yaml"), "w+") as log_res:
        json.dump(res_dict, log_res)


if __name__ == "__main__":
    main()

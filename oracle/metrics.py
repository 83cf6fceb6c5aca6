"""CPU restatement of the evaluation metrics (lidiff/utils/metrics.py, histogram_metrics.py, eval_path.py) for the tests.

* nearest distance: scipy's cKDTree finds the neighbour, the distance is recomputed in fp64 as np.sqrt(((q - r)**2).sum(1));
* voxel histograms: searchsorted on the reference's np.linspace edges (np.histogramdd's rule) and np.unique on the flat bin keys,
  so the reference's 0.1 m grid (1000^3 bins) is feasible on the host;
* Jensen-Shannon: scipy's jensenshannon over the union of the occupied bins (bins empty in both clouds contribute nothing);
* the reference's class formulas and eval_path's ground-truth construction.
"""
from __future__ import annotations

import numpy as np
import scipy.integrate
from scipy.spatial import cKDTree
from scipy.spatial.distance import jensenshannon


def points_of(x):
    if hasattr(x, "points") and not isinstance(x, np.ndarray):
        x = x.points
    return np.asarray(x, dtype=np.float64)[:, :3]


def nn_distance(query, ref):
    q, r = points_of(query), points_of(ref)
    if len(q) == 0:
        return np.zeros(0)
    _, idx = cKDTree(r).query(q, workers=-1)
    return np.sqrt(((q - r[idx]) ** 2).sum(1))


def voxel_bins(p, voxel_size, max_range):
    """(m,) flat bin keys (ix*bins + iy)*bins + iz of the points np.histogramdd keeps, and bins"""
    bins = int(2 * max_range / voxel_size)
    edges = np.linspace(-max_range, max_range, bins + 1)
    p = points_of(p)
    idx = np.empty(p.shape, np.int64)
    for a in range(3):
        c = np.searchsorted(edges, p[:, a], side="right")
        c[p[:, a] == edges[-1]] -= 1
        idx[:, a] = c - 1
    ok = ((idx >= 0) & (idx < bins)).all(1)
    idx = idx[ok]
    return (idx[:, 0] * bins + idx[:, 1]) * bins + idx[:, 2], bins


def sparse_hist(p, voxel_size, max_range):
    """occupied flat bin keys (ascending) and their counts: the non-zero part of np.histogramdd(p, bins, range=[-R, R]^3)"""
    keys, _ = voxel_bins(p, voxel_size, max_range)
    return np.unique(keys, return_counts=True)


def _jsd_sparse(ka, ca, kb, cb):
    u = np.union1d(ka, kb)
    pa, pb = np.zeros(len(u)), np.zeros(len(u))
    pa[np.searchsorted(u, ka)] = ca
    pb[np.searchsorted(u, kb)] = cb
    return float(jensenshannon(pa, pb))


def hist_compare(a, b, voxel_size, max_range):
    """the quantities of lb2_voxel_hist_compare"""
    ka, ca = sparse_hist(a, voxel_size, max_range)
    kb, cb = sparse_hist(b, voxel_size, max_range)
    bins = int(2 * max_range / voxel_size)
    cola, zca = np.unique(ka // bins, return_counts=True)        # per (x, y) column: number of occupied z bins
    colb, zcb = np.unique(kb // bins, return_counts=True)
    return {"n_a": int(ca.sum()), "n_b": int(cb.sum()), "occ_a": len(ka), "occ_b": len(kb), "occ_ab": len(np.intersect1d(ka, kb)),
            "jsd_3d": _jsd_sparse(ka, ca, kb, cb), "jsd_bev": _jsd_sparse(cola, zca, colb, zcb)}


def compute_hist_metrics(pcd_gt, pcd_pred, bev=False):
    r = hist_compare(pcd_gt, pcd_pred, 0.5, 50.)
    return r["jsd_bev"] if bev else r["jsd_3d"]


class RMSE:
    def __init__(self):
        self.dists = []

    def update(self, gt_pcd, pt_pcd):
        self.dists.append(np.mean(nn_distance(pt_pcd, gt_pcd)))

    def compute(self):
        d = np.array(self.dists)
        return d.mean(), d.std()


class ChamferDistance(RMSE):
    def update(self, gt_pcd, pt_pcd):
        self.dists.append((np.mean(nn_distance(gt_pcd, pt_pcd)) + np.mean(nn_distance(pt_pcd, gt_pcd))) / 2)


class CompletionIoU:
    def __init__(self, voxel_sizes=(0.5, 0.2, 0.1)):
        self.voxel_sizes = list(voxel_sizes)
        self.conf_matrix = np.zeros((len(self.voxel_sizes), 3)).astype(np.uint64)

    def update(self, gt, pred):
        for i, v in enumerate(self.voxel_sizes):
            kg, _ = sparse_hist(gt, v, 50.)
            kp, _ = sparse_hist(pred, v, 50.)
            tp = len(np.intersect1d(kg, kp))
            self.conf_matrix[i] += np.array([tp, len(kg) - tp, len(kp) - tp], dtype=np.uint64)

    def compute(self):
        return {v: self.conf_matrix[i][0] / (self.conf_matrix[i][0] + self.conf_matrix[i][1] + self.conf_matrix[i][2] + 1e-15)
                for i, v in enumerate(self.voxel_sizes)}


class PrecisionRecall:
    def __init__(self, min_t, max_t, num):
        self.thresholds = np.linspace(min_t, max_t, num)
        self.pr = {t: [] for t in self.thresholds}
        self.re = {t: [] for t in self.thresholds}
        self.f1 = {t: [] for t in self.thresholds}

    def update(self, gt_pcd, pt_pcd):
        d_p, d_r = nn_distance(pt_pcd, gt_pcd), nn_distance(gt_pcd, pt_pcd)
        for t in self.thresholds:
            p = 100 / len(d_p) * len(np.where(d_p < t)[0])
            r = 100 / len(d_r) * len(np.where(d_r < t)[0])
            self.pr[t].append(p)
            self.re[t].append(r)
            self.f1[t].append(0 if p == 0 or r == 0 else 2 * p * r / (p + r))

    def compute_at_all_thresholds(self):
        m = lambda d: [sum(d[t]) / len(d[t]) for t in self.thresholds]
        return m(self.pr), m(self.re), m(self.f1)

    def compute_at_threshold(self, threshold):
        t = self.thresholds[np.abs(self.thresholds - threshold).argmin()]
        return sum(self.pr[t]) / len(self.pr[t]), sum(self.re[t]) / len(self.re[t]), sum(self.f1[t]) / len(self.f1[t]), t

    def compute_auc(self):
        dx = self.thresholds[1] - self.thresholds[0]
        perfect = scipy.integrate.simpson(np.ones_like(self.thresholds), dx=dx)
        return tuple(scipy.integrate.simpson(v, dx=dx) / perfect for v in self.compute_at_all_thresholds())


# ---- eval_path ground truth ------------------------------------------------------------------------------------------------------
def parse_calibration(filename):
    calib = {}
    with open(filename) as f:
        for line in f:
            key, content = line.strip().split(":")
            v = [float(x) for x in content.strip().split()]
            pose = np.zeros((4, 4))
            pose[0, :4], pose[1, :4], pose[2, :4], pose[3, 3] = v[0:4], v[4:8], v[8:12], 1.0
            calib[key] = pose
    return calib


def load_poses(calib_fname, poses_fname):
    tr = parse_calibration(calib_fname)["Tr"]
    poses = []
    with open(poses_fname) as f:
        for line in f:
            v = [float(x) for x in line.strip().split()]
            pose = np.zeros((4, 4))
            pose[0, :4], pose[1, :4], pose[2, :4], pose[3, 3] = v[0:4], v[4:8], v[8:12], 1.0
            poses.append(np.linalg.inv(tr) @ (pose @ tr))
    return poses


def ground_truth(pose, cur_scan, seq_map, max_range):
    """map crop at max_range around the pose, into the scan frame, z in (-4, 4.4), inside the 10 m voxel grid of the scan
    (origin = minimum bound - half a voxel)"""
    trans = pose[:-1, -1]
    gt = seq_map[np.sum((seq_map - trans) ** 2, axis=-1) ** .5 < max_range]
    gt = (np.concatenate((gt, np.ones((len(gt), 1))), axis=-1) @ np.linalg.inv(pose).T)[:, :3]
    gt = gt[(gt[:, 2] > -4.) & (gt[:, 2] < 4.4)]
    org = cur_scan.min(0) - 5.0
    keys = {tuple(k) for k in np.floor((cur_scan - org) / 10.0).astype(np.int64)}
    inside = np.array([tuple(k) in keys for k in np.floor((gt - org) / 10.0).astype(np.int64)], dtype=bool)
    return gt[inside]

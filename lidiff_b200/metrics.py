"""Evaluation metrics of completed scans on the GPU — lidiff/utils/metrics.py (RMSE, ChamferDistance, PrecisionRecall,
CompletionIoU) and lidiff/utils/histogram_metrics.py (compute_hist_metrics) with the reference's names, arguments and formulas.

The reference takes nearest distances from open3d's k-d tree and voxel statistics from dense np.histogramdd grids (1000^3 float64
bins per cloud at its default 0.1 m).  Here three CUDA kernels (lb2_cloud_nn_distance, lb2_voxel_hist_compare,
lb2_threshold_counts) produce the distances, counts and Jensen-Shannon sums, and the host repeats the reference's arithmetic on them
in the reference's order: from identical counts the outputs are bit-identical, from sums they agree to reordering.

Inputs: numpy arrays, torch tensors or anything with `.points` (the open3d shim's PointCloud); only the first three columns are used.
There is no CPU path: the plain functions raise on CPU tensors, the classes need a CUDA device.
"""
from __future__ import annotations

import ctypes

import numpy as np
import scipy.integrate
import torch

from . import _lib


def _handle(t):
    return _lib.get_handle(t.device)


def _cloud(x, device=None) -> torch.Tensor:
    """(n, 3) contiguous fp64 CUDA tensor of a numpy array / torch tensor / object with `.points`"""
    if hasattr(x, "points") and not isinstance(x, (np.ndarray, torch.Tensor)):
        x = np.asarray(x.points)
    if isinstance(x, torch.Tensor):
        t = x.detach()
        if not t.is_cuda:
            t = t.to(device or "cuda")
    else:
        t = torch.from_numpy(np.ascontiguousarray(np.asarray(x, dtype=np.float64))).to(device or "cuda")
    t = t.reshape(t.shape[0], -1) if t.dim() != 2 else t
    return t[:, :3].to(torch.float64).contiguous()


def _require_cuda(*ts, what):
    for t in ts:
        if not isinstance(t, torch.Tensor) or not t.is_cuda:
            raise RuntimeError(f"{what}: CUDA tensors required (no CPU fallback)")


def nn_distance(query: torch.Tensor, ref: torch.Tensor) -> torch.Tensor:
    """dist[i] = min_j |query[i] - ref[j]| in fp64 on the device; equals numpy's np.sqrt(((q - r)**2).sum(1)) for the nearest r bit
    for bit (open3d's compute_point_cloud_distance).  An empty query gives an empty result."""
    _require_cuda(query, ref, what="nn_distance")
    q = query[:, :3].to(torch.float64).contiguous()
    r = ref[:, :3].to(torch.float64).contiguous()
    nq, nr = q.shape[0], r.shape[0]
    dist = torch.empty(nq, dtype=torch.float64, device=q.device)
    if nq == 0:
        return dist
    if nr == 0:
        raise ValueError("nn_distance: empty reference cloud")
    h = _handle(q)
    scratch = torch.empty(h.cloud_nn_scratch_bytes(nq, nr), dtype=torch.uint8, device=q.device)
    h.cloud_nn_distance(q, nq, r, nr, scratch, dist)
    return dist


def threshold_counts(d: torch.Tensor, thresholds) -> np.ndarray:
    """counts[t] = #{i : d[i] < thresholds[t]} (ascending thresholds), int64 numpy array"""
    _require_cuda(d, what="threshold_counts")
    d = d.to(torch.float64).contiguous()
    thr = torch.as_tensor(np.asarray(thresholds, dtype=np.float64), device=d.device)
    counts = torch.empty(thr.numel(), dtype=torch.int64, device=d.device)
    _handle(d).threshold_counts(d, d.numel(), thr, thr.numel(), counts)
    return counts.cpu().numpy()


_EDGES = {}


def _edges(max_range, bins, device):
    key = (float(max_range), int(bins), str(device))
    if key not in _EDGES:                                   # the reference's per-axis edges, np.linspace(-R, R, bins + 1)
        _EDGES[key] = torch.from_numpy(np.linspace(-max_range, max_range, bins + 1)).to(device)
    return _EDGES[key]


def voxel_hist_compare(a: torch.Tensor, b: torch.Tensor, voxel_size: float, max_range: float) -> dict:
    """Both clouds on np.histogramdd's grid of the reference (bins = int(2 * max_range / voxel_size) per axis over
    [-max_range, max_range]): points in range (n_a, n_b), occupied voxels (occ_a, occ_b, occ_ab) and the Jensen-Shannon distances
    of histogram_metrics.compute_jsd with a as the first argument, of the raw counts (jsd_3d) and of the per-column numbers of
    occupied z voxels (jsd_bev)."""
    _require_cuda(a, b, what="voxel_hist_compare")
    a = a[:, :3].to(torch.float64).contiguous()
    b = b[:, :3].to(torch.float64).contiguous()
    bins = int(2 * max_range / voxel_size)
    h = _handle(a)
    scratch = torch.empty(h.voxel_hist_scratch_bytes(a.shape[0], b.shape[0]), dtype=torch.uint8, device=a.device)
    out = torch.empty(ctypes.sizeof(_lib.VoxelHistResult), dtype=torch.uint8, device=a.device)
    h.voxel_hist_compare(a, a.shape[0], b, b.shape[0], _edges(max_range, bins, a.device), bins, scratch, out)
    r = _lib.VoxelHistResult.from_buffer_copy(out.cpu().numpy().tobytes())
    return {k: getattr(r, k) for k, _ in _lib.VoxelHistResult._fields_}


# ---- the reference's classes (lidiff/utils/metrics.py) ---------------------------------------------------------------------------
class RMSE:
    def __init__(self):
        self.dists = []

    def update(self, gt_pcd, pt_pcd):
        dist_pt_2_gt = nn_distance(_cloud(pt_pcd), _cloud(gt_pcd)).cpu().numpy()
        self.dists.append(np.mean(dist_pt_2_gt))

    def reset(self):
        self.dists = []

    def compute(self):
        dist = np.array(self.dists)
        return dist.mean(), dist.std()


class ChamferDistance:
    def __init__(self):
        self.dists = []

    def update(self, gt_pcd, pt_pcd):
        gt, pt = _cloud(gt_pcd), _cloud(pt_pcd)
        dist_pt_2_gt = nn_distance(pt, gt).cpu().numpy()
        dist_gt_2_pt = nn_distance(gt, pt).cpu().numpy()
        self.dists.append((np.mean(dist_gt_2_pt) + np.mean(dist_pt_2_gt)) / 2)

    def reset(self):
        self.dists = []

    def compute(self):
        cdist = np.array(self.dists)
        return cdist.mean(), cdist.std()


class CompletionIoU:
    """tp / (tp + fn + fp + 1e-15) of the occupied voxels of ground truth and prediction in [-50, 50]^3 at each voxel size"""

    def __init__(self, voxel_sizes=[0.5, 0.2, 0.1]):   # noqa: B006 (the reference's signature)
        self.voxel_sizes = voxel_sizes
        self.conf_matrix = np.zeros((len(self.voxel_sizes), 3)).astype(np.uint64)      # tp, fn, fp

    def update(self, gt, pred):
        max_range = 50.
        g, p = _cloud(gt), _cloud(pred)
        for i, vsize in enumerate(self.voxel_sizes):
            r = voxel_hist_compare(g, p, vsize, max_range)
            tp = r["occ_ab"]
            self.conf_matrix[i][0] += np.uint64(tp)
            self.conf_matrix[i][1] += np.uint64(r["occ_a"] - tp)
            self.conf_matrix[i][2] += np.uint64(r["occ_b"] - tp)

    def compute(self):
        res_vsizes = {}
        for i, vsize in enumerate(self.voxel_sizes):
            tp = self.conf_matrix[i][0]
            fn = self.conf_matrix[i][1]
            fp = self.conf_matrix[i][2]
            intersection = tp
            union = tp + fn + fp + 1e-15
            res_vsizes[vsize] = intersection / union
        return res_vsizes

    def reset(self):
        self.conf_matrix = np.zeros((len(self.voxel_sizes), 3)).astype(np.uint)


class PrecisionRecall:
    def __init__(self, min_t, max_t, num):
        self.thresholds = np.linspace(min_t, max_t, num)
        self.pr_dict = {t: [] for t in self.thresholds}
        self.re_dict = {t: [] for t in self.thresholds}
        self.f1_dict = {t: [] for t in self.thresholds}

    def update(self, gt_pcd, pt_pcd):
        gt, pt = _cloud(gt_pcd), _cloud(pt_pcd)
        dist_pt_2_gt = nn_distance(pt, gt)            # precision: predicted --> ground truth
        dist_gt_2_pt = nn_distance(gt, pt)            # recall: ground truth --> predicted
        order = np.argsort(self.thresholds, kind="stable")
        cnt_p, cnt_r = np.empty(len(order), np.int64), np.empty(len(order), np.int64)
        cnt_p[order] = threshold_counts(dist_pt_2_gt, self.thresholds[order])
        cnt_r[order] = threshold_counts(dist_gt_2_pt, self.thresholds[order])
        n_p, n_r = dist_pt_2_gt.numel(), dist_gt_2_pt.numel()
        for k, t in enumerate(self.thresholds):
            p = 100 / n_p * int(cnt_p[k])
            self.pr_dict[t].append(p)
            r = 100 / n_r * int(cnt_r[k])
            self.re_dict[t].append(r)
            if p == 0 or r == 0:
                f = 0
            else:
                f = 2 * p * r / (p + r)
            self.f1_dict[t].append(f)

    def reset(self):
        self.pr_dict = {t: [] for t in self.thresholds}
        self.re_dict = {t: [] for t in self.thresholds}
        self.f1_dict = {t: [] for t in self.thresholds}

    def compute_at_threshold(self, threshold):
        t = self.find_nearest_threshold(threshold)
        pr = sum(self.pr_dict[t]) / len(self.pr_dict[t])
        re = sum(self.re_dict[t]) / len(self.re_dict[t])
        f1 = sum(self.f1_dict[t]) / len(self.f1_dict[t])
        return pr, re, f1, t

    def compute_auc(self):
        dx = self.thresholds[1] - self.thresholds[0]
        perfect_predictor = scipy.integrate.simpson(np.ones_like(self.thresholds), dx=dx)
        pr, re, f1 = self.compute_at_all_thresholds()
        norm_pr_area = scipy.integrate.simpson(pr, dx=dx) / perfect_predictor
        norm_re_area = scipy.integrate.simpson(re, dx=dx) / perfect_predictor
        norm_f1_area = scipy.integrate.simpson(f1, dx=dx) / perfect_predictor
        return norm_pr_area, norm_re_area, norm_f1_area

    def compute_at_all_thresholds(self):
        pr = [sum(self.pr_dict[t]) / len(self.pr_dict[t]) for t in self.thresholds]
        re = [sum(self.re_dict[t]) / len(self.re_dict[t]) for t in self.thresholds]
        f1 = [sum(self.f1_dict[t]) / len(self.f1_dict[t]) for t in self.thresholds]
        return pr, re, f1

    def find_nearest_threshold(self, value):
        idx = (np.abs(self.thresholds - value)).argmin()
        return self.thresholds[idx]


# ---- lidiff/utils/histogram_metrics.py -------------------------------------------------------------------------------------------
def compute_hist_metrics(pcd_gt, pcd_pred, bev=False):
    """Jensen-Shannon distance of the 0.5 m histograms in [-50, 50]^3: of the raw counts, or (bev=True) of the per-(x, y)-column
    numbers of occupied z voxels"""
    r = voxel_hist_compare(_cloud(pcd_gt), _cloud(pcd_pred), 0.5, 50.)
    return r["jsd_bev"] if bev else r["jsd_3d"]

"""The CPU restatement of the evaluation metrics (oracle/metrics.py) against numpy's dense histograms, scipy and the recorded outputs
of the reference's metrics module; the pose / ground-truth arithmetic of lidiff_b200.tools.eval_path on a hand-built sequence."""
import json
import os

import numpy as np
import pytest
from scipy.spatial.distance import jensenshannon

from oracle import metrics as om

HERE = os.path.dirname(os.path.abspath(__file__))
REFERENCE = json.load(open(os.path.join(HERE, "golden", "reference_on_shims.json")))


def edge_cloud(seed, n=20000):
    """normal clouds plus points exactly on bin edges, at +-50 m and just outside the range"""
    g = np.random.default_rng(seed)
    p = g.normal(size=(n, 3)) * [15, 15, 2]
    e = g.integers(-100, 101, size=(600, 3)) * 0.5                       # multiples of 0.5 m: edges of every grid tested
    e[:100, 0] = 50.0
    e[100:200, 1] = -50.0
    e[200:250, 2] = np.nextafter(50.0, 100.0)                            # just outside: dropped
    e[250:300, 0] = np.nextafter(-50.0, -100.0)
    e[300:350] = 50.0
    return np.concatenate([p, e, g.uniform(-60, 60, size=(500, 3))])


@pytest.mark.parametrize("voxel", [2.0, 1.0, 0.5])
def test_sparse_histogram_equals_histogramdd(voxel):
    for seed in (0, 1):
        p = edge_cloud(seed)
        bins = int(2 * 50.0 / voxel)
        dense = np.histogramdd(p, bins=bins, range=([-50., 50.],) * 3)[0]
        keys, counts = om.sparse_hist(p, voxel, 50.0)
        nz = np.flatnonzero(dense.reshape(-1))
        assert np.array_equal(keys, nz)
        assert np.array_equal(counts, dense.reshape(-1)[nz].astype(np.int64))


def test_jsd_equals_dense_formula():
    a, b = edge_cloud(2), edge_cloud(3)[:15000] + 0.3
    r = om.hist_compare(a, b, 0.5, 50.0)
    ha = np.histogramdd(a, bins=200, range=([-50., 50.],) * 3)[0]
    hb = np.histogramdd(b, bins=200, range=([-50., 50.],) * 3)[0]

    def compute_jsd(hist_gt, hist_pred, bev):                            # histogram_metrics.compute_jsd
        g = hist_gt.sum(-1) if bev else hist_gt
        p = hist_pred.sum(-1) if bev else hist_pred
        return jensenshannon((g / g.sum()).flatten(), (p / p.sum()).flatten())

    assert r["jsd_3d"] == pytest.approx(compute_jsd(ha, hb, False), rel=1e-12, abs=0)
    assert r["jsd_bev"] == pytest.approx(compute_jsd(np.clip(ha, 0, 1), np.clip(hb, 0, 1), True), rel=1e-12, abs=0)
    occ_a, occ_b = ha.astype(bool), hb.astype(bool)
    assert (r["occ_a"], r["occ_b"], r["occ_ab"]) == (occ_a.sum(), occ_b.sum(), (occ_a & occ_b).sum())
    assert (r["n_a"], r["n_b"]) == (ha.sum(), hb.sum())


def seeded_clouds():
    g = np.random.default_rng(3)
    gt = g.normal(size=(6000, 3)) * [12, 12, 1.0]
    pred = gt[g.choice(6000, 4000, replace=False)] + g.normal(size=(4000, 3)) * 0.05
    return gt, pred


def test_oracle_classes_reproduce_the_reference_outputs():
    ref = REFERENCE["metrics"]
    gt, pred = seeded_clouds()
    cd, rm = om.ChamferDistance(), om.RMSE()
    cd.update(gt, pred)
    rm.update(gt, pred)
    pr = om.PrecisionRecall(0.05, 1.0, 20)
    pr.update(gt, pred)
    iou = om.CompletionIoU(voxel_sizes=[2.0, 1.0, 0.5])
    iou.update(gt, pred)
    assert cd.compute()[0] == pytest.approx(ref["chamfer"][0], rel=1e-12) and cd.compute()[1] == 0.0
    assert rm.compute()[0] == pytest.approx(ref["rmse"][0], rel=1e-12)
    assert [float(x) for x in pr.compute_at_threshold(0.1)] == ref["precision_recall_at_0.1"]
    assert [float(x) for x in pr.compute_auc()] == ref["precision_recall_auc"]
    assert {str(k): float(v) for k, v in iou.compute().items()} == ref["completion_iou"]


def write_sequence(root, n_scans=3, seed=0):
    """a SemanticKITTI-shaped sequence: velodyne/*.bin, poses.txt, calib.txt with a non-identity Tr, map_clean.npy (world frame)"""
    from lidiff_b200.synth import synthetic_scan
    g = np.random.default_rng(seed)
    os.makedirs(os.path.join(root, "velodyne"), exist_ok=True)
    c, s = np.cos(0.02), np.sin(0.02)
    tr = np.array([[c, -s, 0, 0.27], [s, c, 0, -0.08], [0, 0, 1, -0.12], [0, 0, 0, 1.0]])
    with open(os.path.join(root, "calib.txt"), "w") as f:
        f.write("P0: " + " ".join(["1"] + ["0"] * 11) + "\n")
        f.write("Tr: " + " ".join(repr(float(v)) for v in tr[:3].reshape(-1)) + "\n")
    poses, world = [], []
    with open(os.path.join(root, "poses.txt"), "w") as f:
        for k in range(n_scans):
            yaw = 0.1 * k
            p = np.array([[np.cos(yaw), -np.sin(yaw), 0, 3.0 * k], [np.sin(yaw), np.cos(yaw), 0, 0.5 * k], [0, 0, 1, 0.02 * k], [0, 0, 0, 1.0]])
            f.write(" ".join(repr(float(v)) for v in p[:3].reshape(-1)) + "\n")
            poses.append(np.linalg.inv(tr) @ p @ tr)
    for k in range(n_scans):
        scan = synthetic_scan(seed + k, beams=64, azimuths=512)            # 32 k points: enough for DiffCompletion's 18 k FPS
        raw = np.concatenate([scan, g.uniform(0, 1, (len(scan), 1))], 1).astype(np.float32)
        raw.tofile(os.path.join(root, "velodyne", f"{k:06d}.bin"))
        pts = np.concatenate([scan, np.ones((len(scan), 1))], 1) @ poses[k].T
        world.append(pts[:, :3] + g.normal(size=(len(scan), 3)) * 0.03)
    np.save(os.path.join(root, "map_clean.npy"), np.concatenate(world))
    return poses


def test_eval_path_poses_and_ground_truth_crop(tmp_path):
    import torch
    from lidiff_b200.tools import eval_path as ep
    poses_ref = write_sequence(str(tmp_path))
    poses = ep.load_poses(str(tmp_path / "calib.txt"), str(tmp_path / "poses.txt"))
    assert len(poses) == 3
    for p, q in zip(poses, poses_ref):
        assert np.allclose(p, q, rtol=0, atol=1e-12)
    assert np.array_equal(np.stack(poses), np.stack(om.load_poses(str(tmp_path / "calib.txt"), str(tmp_path / "poses.txt"))))
    seq_map = np.load(tmp_path / "map_clean.npy")
    for k, pose in enumerate(poses):
        _, cur = ep.read_scan(str(tmp_path / "velodyne" / f"{k:06d}.bin"), 50.0)
        gt = ep.ground_truth(pose, cur, torch.from_numpy(seq_map), 50.0).numpy()
        want = om.ground_truth(pose, cur.astype(np.float64), seq_map, 50.0)
        assert gt.shape == want.shape and len(gt) > 1000
        assert np.allclose(gt, want, rtol=0, atol=1e-9)
        assert (np.abs(gt[:, 2]) < 4.4).all()

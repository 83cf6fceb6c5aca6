"""Evaluation metrics on the GPU (lidiff_b200.metrics) against brute-force numpy, scipy's k-d tree, the CPU restatement
(oracle/metrics.py) and the recorded outputs of the reference's metrics module; the eval_path CLI end to end."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import metrics as om

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
REFERENCE = json.load(open(os.path.join(HERE, "golden", "reference_on_shims.json")))


def cuda(x):
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64)).cuda()


def brute_nn(q, r, chunk=256):
    """min over r of sqrt((dx*dx + dy*dy) + dz*dz) in fp64, numpy's order"""
    out = np.empty(len(q))
    for a in range(0, len(q), chunk):
        qc = q[a:a + chunk]
        dx, dy, dz = (qc[:, None, k] - r[None, :, k] for k in range(3))
        out[a:a + chunk] = np.sqrt(((dx * dx + dy * dy) + dz * dz).min(1))
    return out


def kitti_like(seed, n):
    from lidiff_b200.synth import synthetic_scan
    p = synthetic_scan(seed)                                                # 131 k points
    return p[np.random.default_rng(seed).choice(len(p), n, replace=n > len(p))]


def nn_cases():
    g = np.random.default_rng(7)
    r = g.normal(size=(15000, 3)) * [10, 10, 1]
    yield "random", g.normal(size=(20000, 3)) * [10, 10, 1], r
    k = kitti_like(1, 20000)
    yield "kitti", k + g.normal(size=k.shape) * 0.1, kitti_like(2, 20000)
    d = np.repeat(g.normal(size=(2000, 3)), 5, axis=0)                     # every point five times
    yield "duplicates", np.concatenate([d[::3], d[:500] + 1e-3]), d
    xs, ys = np.meshgrid(np.arange(-70, 71, 1.0), np.arange(-70, 71, 1.0))
    plane = np.stack([xs.ravel(), ys.ravel(), np.zeros(xs.size)], 1)        # lattice: queries at cell centres tie with 4 points
    yield "lattice", np.stack([xs.ravel()[:19000] + 0.5, ys.ravel()[:19000] + 0.5, np.full(19000, 0.25)], 1), plane
    yield "far", r[:5000] + [1000.0, -1000.0, 1000.0], r
    yield "one_ref", g.normal(size=(3000, 3)), g.normal(size=(1, 3))


@pytest.mark.parametrize("case", ["random", "kitti", "duplicates", "lattice", "far", "one_ref"])
def test_nn_distance_is_bit_identical_to_brute_force(case):
    from lidiff_b200.metrics import nn_distance
    q, r = dict((c, (q, r)) for c, q, r in nn_cases())[case]
    d = nn_distance(cuda(q), cuda(r)).cpu().numpy()
    assert np.array_equal(d, brute_nn(q, r))


def test_nn_distance_empty_query_and_cpu_input():
    from lidiff_b200.metrics import nn_distance
    assert nn_distance(cuda(np.zeros((0, 3))), cuda(np.ones((5, 3)))).shape == (0,)
    with pytest.raises(RuntimeError):
        nn_distance(torch.zeros(4, 3, dtype=torch.float64), torch.zeros(4, 3, dtype=torch.float64))


def test_nn_distance_at_eval_size_matches_kdtree_and_repeats():
    from scipy.spatial import cKDTree
    from lidiff_b200.metrics import nn_distance
    g = np.random.default_rng(11)
    r = np.concatenate([kitti_like(s, 120000) for s in range(9)])           # 1.08 M
    q = r[g.permutation(len(r))[:1000000]] + g.normal(size=(1000000, 3)) * 0.05
    q[:20000] += [0.0, 0.0, 30.0]                                          # some far outside the reference's z range
    tq, tr = cuda(q), cuda(r)
    d1 = nn_distance(tq, tr).cpu().numpy()
    d2 = nn_distance(tq, tr).cpu().numpy()
    assert np.array_equal(d1, d2)
    assert np.abs(d1 - cKDTree(r).query(q, workers=-1)[0]).max() <= 1e-9


def hist_clouds(seed):
    g = np.random.default_rng(seed)
    a = np.concatenate([kitti_like(seed, 100000), g.integers(-500, 501, size=(3000, 3)) * 0.1,
                        np.array([[50.0, 0, 0], [-50.0, 50.0, -50.0], [np.nextafter(50.0, 99), 0, 0], [0, -50.0000001, 0]])])
    b = a[g.choice(len(a), 80000, replace=False)] + g.normal(size=(80000, 3)) * 0.05
    return a, b


@pytest.mark.parametrize("voxel", [0.5, 0.2, 0.1])
def test_voxel_hist_equals_the_oracle(voxel):
    from lidiff_b200.metrics import voxel_hist_compare
    a, b = hist_clouds(5)
    r1 = voxel_hist_compare(cuda(a), cuda(b), voxel, 50.0)
    r2 = voxel_hist_compare(cuda(a), cuda(b), voxel, 50.0)
    want = om.hist_compare(a, b, voxel, 50.0)
    for k in ("n_a", "n_b", "occ_a", "occ_b", "occ_ab"):
        assert r1[k] == want[k], k
    for k in ("jsd_3d", "jsd_bev"):
        assert r1[k] == pytest.approx(want[k], rel=1e-12, abs=0), k
    assert r1 == r2


def test_threshold_counts_equal_numpy():
    from lidiff_b200.metrics import threshold_counts
    g = np.random.default_rng(9)
    d = np.abs(g.normal(size=300000)) * 0.1
    thr = np.linspace(0.05, 0.1, 100)
    d[:1000] = thr[g.integers(0, 100, 1000)]                                # exactly on thresholds: strict <
    got = threshold_counts(cuda(d), thr)
    assert np.array_equal(got, np.array([len(np.where(d < t)[0]) for t in thr]))


def seeded_clouds():
    g = np.random.default_rng(3)
    gt = g.normal(size=(6000, 3)) * [12, 12, 1.0]
    pred = gt[g.choice(6000, 4000, replace=False)] + g.normal(size=(4000, 3)) * 0.05
    return gt, pred


def test_gpu_classes_reproduce_the_reference_outputs():
    from lidiff_b200 import metrics as m
    from lidiff_b200.shims.open3d.geometry import PointCloud
    ref = REFERENCE["metrics"]
    gt, pred = seeded_clouds()
    pg, pp = PointCloud(gt), PointCloud(pred)
    cd, rm = m.ChamferDistance(), m.RMSE()
    cd.update(pg, pp)
    rm.update(gt, torch.from_numpy(pred))
    pr = m.PrecisionRecall(0.05, 1.0, 20)
    pr.update(pg, pp)
    iou = m.CompletionIoU(voxel_sizes=[2.0, 1.0, 0.5])
    iou.update(pg, pp)
    assert cd.compute()[0] == pytest.approx(ref["chamfer"][0], rel=1e-12, abs=0)
    assert rm.compute()[0] == pytest.approx(ref["rmse"][0], rel=1e-12, abs=0)
    assert [float(x) for x in pr.compute_at_threshold(0.1)] == ref["precision_recall_at_0.1"]
    assert [float(x) for x in pr.compute_auc()] == ref["precision_recall_auc"]
    assert {str(k): float(v) for k, v in iou.compute().items()} == ref["completion_iou"]


def test_default_completion_iou_and_jsd_on_full_scans():
    from lidiff_b200 import metrics as m
    g = np.random.default_rng(4)
    gt = kitti_like(3, 180000)
    pred = kitti_like(4, 180000) + g.normal(size=(180000, 3)) * 0.05
    iou, want = m.CompletionIoU(), om.CompletionIoU()
    iou.update(gt, pred)
    want.update(gt, pred)
    assert np.array_equal(iou.conf_matrix, want.conf_matrix)
    assert iou.compute() == want.compute()
    for bev in (False, True):
        assert m.compute_hist_metrics(gt, pred, bev) == pytest.approx(om.compute_hist_metrics(gt, pred, bev), rel=1e-12, abs=0)


def test_eval_path_cli_end_to_end(tmp_path):
    from test_metrics_oracle import write_sequence
    from lidiff_b200.tools import eval_path as ep
    from lidiff_b200.tools.diff_completion_pipeline import write_ply
    seq = tmp_path / "seq"
    poses = write_sequence(str(seq))
    pred_dir = tmp_path / "exp" / "refine"
    os.makedirs(pred_dir)
    g = np.random.default_rng(1)
    for k in range(3):
        _, cur = ep.read_scan(str(seq / "velodyne" / f"{k:06d}.bin"), 50.0)
        p = np.repeat(cur.astype(np.float64), 2, axis=0) + g.normal(size=(2 * len(cur), 3)) * 0.05
        write_ply(str(pred_dir / f"{k:06d}.ply"), p)
    ep.main.main(["-p", str(pred_dir), "--data", str(seq)], standalone_mode=False)
    res = json.load(open(tmp_path / "exp" / "res_log.yaml"))

    seq_map = np.load(seq / "map_clean.npy")
    iou, rmse, cd, pr = om.CompletionIoU(), om.RMSE(), om.ChamferDistance(), om.PrecisionRecall(0.05, 0.1, 100)
    j3, jb = [], []
    for k, pose in enumerate(poses):
        _, cur = ep.read_scan(str(seq / "velodyne" / f"{k:06d}.bin"), 50.0)
        pred = ep.read_prediction(str(pred_dir / f"{k:06d}.ply"), 50.0)
        gt = om.ground_truth(ep.load_poses(str(seq / "calib.txt"), str(seq / "poses.txt"))[k], cur.astype(np.float64), seq_map, 50.0)
        j3.append(om.compute_hist_metrics(gt, pred, False))
        jb.append(om.compute_hist_metrics(gt, pred, True))
        for o in (iou, rmse, cd, pr):
            o.update(gt, pred)
    assert res["ious"] == {str(k): float(v) for k, v in iou.compute().items()}
    want = {"jsd": np.mean(jb), "jsd_noclip_3d": np.mean(j3), "rmse_mean": rmse.compute()[0], "rmse_std": rmse.compute()[1],
            "cd_mean": cd.compute()[0], "cd_std": cd.compute()[1]}
    want.update(dict(zip(("pr", "re", "f1"), pr.compute_auc())))
    for key, v in want.items():
        assert res[key] == pytest.approx(v, rel=1e-9, abs=1e-12), key

    out = tmp_path / "rw" / "log"
    os.makedirs(out.parent)
    ep.main.main(["--random-weights", "-t", "2", "-p", str(out), "--data", str(seq)], standalone_mode=False)
    res = json.load(open(tmp_path / "rw" / "res_log.yaml"))
    vals = [res[k] for k in ("jsd", "jsd_noclip_3d", "rmse_mean", "rmse_std", "cd_mean", "cd_std", "pr", "re", "f1")] + list(res["ious"].values())
    assert len(res["ious"]) == 3 and np.isfinite(vals).all()

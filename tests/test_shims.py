"""Import shims of SURVEY.md 8f-1: pytorch_lightning / natsort / open3d stand-ins the reference's inference script needs."""
import importlib
import json
import os
import sys

import numpy as np
import pytest
import torch

import lidiff_b200.shims as sh


@pytest.fixture(scope="module", autouse=True)
def _shims_on_path():
    sh.install()
    for m in ("open3d", "natsort", "pytorch_lightning"):          # a real install (none in this image) would be shadowed on purpose
        sys.modules.pop(m, None)
    yield


def test_natsorted_orders_numbers_naturally():
    from natsort import natsorted
    assert natsorted(["10.ply", "9.ply", "000100.ply", "1.ply", "a2", "a10"]) == ["1.ply", "9.ply", "10.ply", "000100.ply", "a2", "a10"]
    assert natsorted(["b3", "b20"], reverse=True) == ["b20", "b3"]


def test_lightning_module_hparams_device_and_partial_state_dict(tmp_path):
    from pytorch_lightning.core.lightning import LightningModule
    import yaml

    class M(LightningModule):
        def __init__(self, hp):
            super().__init__()
            self.save_hyperparameters(hp)
            self.lin = torch.nn.Linear(3, 2)

    m = M({"diff": {"t_steps": 1000}, "data": {"resolution": 0.05}})
    assert m.hparams["diff"]["t_steps"] == 1000 and m.device == torch.device("cpu")
    m.hparams["data"]["max_range"] = 50.0                                   # the reference mutates and dumps it (pipeline:49-56)
    assert yaml.safe_load(yaml.dump(m.hparams))["data"] == {"resolution": 0.05, "max_range": 50.0}
    sd = {"lin.weight": torch.ones(2, 3), "somebody.else": torch.zeros(1)}   # Lightning ckpt dicts hold all sub-models: strict=False
    res = m.load_state_dict(sd, strict=False)
    assert "lin.bias" in res.missing_keys and "somebody.else" in res.unexpected_keys and bool((m.lin.weight == 1).all())
    import pytorch_lightning as pl
    with pytest.raises(NotImplementedError):
        pl.Trainer(gpus=1)


def test_open3d_pointcloud_and_ply_round_trip(tmp_path):
    import open3d as o3d
    g = np.random.default_rng(0)
    pts = g.normal(size=(257, 3)) * [5, 5, 0.01]                               # a thin slab: normals ~ +-z
    pcd = o3d.geometry.PointCloud()
    pcd.points = o3d.utility.Vector3dVector(pts)
    assert np.array(pcd.points).shape == (257, 3) and not pcd.has_normals()
    for ascii_ in (False, True):
        f = str(tmp_path / f"a{int(ascii_)}.ply")
        o3d.io.write_point_cloud(f, pcd, write_ascii=ascii_)
        back = np.array(o3d.io.read_point_cloud(f).points)
        assert np.allclose(back, pts, rtol=0, atol=0 if not ascii_ else 1e-8)
    pcd.estimate_normals()
    n = np.asarray(pcd.normals)
    assert pcd.has_normals() and np.allclose(np.linalg.norm(n, axis=1), 1, atol=1e-5) and (np.abs(n[:, 2]) > 0.9).mean() > 0.9
    f = str(tmp_path / "n.ply")
    o3d.io.write_point_cloud(f, pcd)
    back = o3d.io.read_point_cloud(f)
    assert back.has_normals() and np.allclose(np.asarray(back.normals), n)
    with pytest.raises(RuntimeError):
        o3d.utility.Vector3dVector(np.zeros((4, 2)))
    from lidiff_b200.synth import read_ply_xyz                                   # the package's own reader agrees with the shim's writer
    assert np.allclose(read_ply_xyz(f), pts)


@pytest.mark.skipif(torch.cuda.is_available(), reason="CPU-only behaviour")
def test_open3d_fps_fails_loudly_without_gpu():
    import open3d as o3d
    pcd = o3d.geometry.PointCloud(np.zeros((10, 3)))
    with pytest.raises(RuntimeError):
        pcd.farthest_point_down_sample(3)


REFERENCE = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_on_shims.json")))


def resolve(dotted):
    """import the longest importable prefix of `dotted`, then walk the remaining attributes"""
    parts = dotted.split(".")
    for n in range(len(parts), 0, -1):
        try:
            obj = importlib.import_module(".".join(parts[:n]))
        except ImportError:
            continue
        for a in parts[n:]:
            obj = getattr(obj, a)
        return obj
    raise ImportError(dotted)


def test_reference_pipeline_script_imports_on_the_shims():
    """every name the reference's inference script (lidiff/tools/diff_completion_pipeline.py), its network module
    (lidiff/models/minkunet.py) and its metrics module (lidiff/utils/metrics.py) take from a shimmed package resolves on the shims
    (the names are recorded in tests/golden/reference_on_shims.json by tests/golden/make_reference_goldens.py)"""
    names = REFERENCE["shim_names"]
    assert set(names) == {"lidiff/tools/diff_completion_pipeline.py", "lidiff/models/minkunet.py", "lidiff/utils/metrics.py"}
    for path, dotted in names.items():
        for d in dotted:
            assert resolve(d) is not None, f"{path}: {d}"
    from pytorch_lightning.core.lightning import LightningModule
    import MinkowskiEngine as ME
    import natsort
    import open3d as o3d
    assert isinstance(LightningModule, type) and issubclass(LightningModule, torch.nn.Module)
    assert issubclass(o3d.geometry.PointCloud, o3d.geometry.Geometry)
    assert o3d.__version__.endswith("lidiff_b200.shim") and callable(natsort.natsorted)
    assert ME.__name__ == "MinkowskiEngine"


def test_reference_metrics_module_runs_on_the_open3d_shim():
    """SURVEY 8f-4: what the reference's lidiff/utils/metrics.py (RMSE, ChamferDistance, PrecisionRecall, CompletionIoU) computed on
    the open3d shim (recorded in tests/golden/reference_on_shims.json) equals the same quantities from the shim's nearest-neighbour
    distances, and those distances equal scipy's exact k-d tree"""
    from scipy.spatial import cKDTree
    import open3d as o3d
    ref = REFERENCE["metrics"]
    g = np.random.default_rng(3)
    gt = g.normal(size=(6000, 3)) * [12, 12, 1.0]
    pred = gt[g.choice(6000, 4000, replace=False)] + g.normal(size=(4000, 3)) * 0.05
    pg, pp = o3d.geometry.PointCloud(gt), o3d.geometry.PointCloud(pred)
    d_pg = np.asarray(pp.compute_point_cloud_distance(pg))
    d_gp = np.asarray(pg.compute_point_cloud_distance(pp))
    assert np.allclose(d_pg, cKDTree(gt).query(pred)[0], rtol=0, atol=1e-9) and np.allclose(d_gp, cKDTree(pred).query(gt)[0], rtol=0, atol=1e-9)
    assert abs(ref["chamfer"][0] - 0.5 * (d_pg.mean() + d_gp.mean())) < 1e-12 and abs(ref["rmse"][0] - d_pg.mean()) < 1e-12
    p, r, f1, t = ref["precision_recall_at_0.1"]
    assert abs(p - 100.0 * (d_pg < t).mean()) < 1e-9 and abs(r - 100.0 * (d_gp < t).mean()) < 1e-9 and 0 < f1 <= 100
    assert all(0 <= v <= 100.000001 for v in ref["precision_recall_auc"])     # percentages, normalised by the perfect predictor
    iou = {float(k): v for k, v in ref["completion_iou"].items()}             # (the default 0.1 m grid is a 1000^3 float64 histogram: 8 GB)
    assert set(iou) == {2.0, 1.0, 0.5} and 0 < iou[0.5] <= iou[1.0] <= iou[2.0] <= 1
    assert ref["prediction_is_empty"] == [False, True]
    assert isinstance(pp, o3d.geometry.Geometry) and len(np.asarray(pp.points)) == 4000
    # viewpoint mask of the training collation (collations.py:44-50): voxel-grid membership at 10 m
    grid = o3d.geometry.VoxelGrid.create_from_point_cloud(pp, voxel_size=10.0)
    inc = np.array(grid.check_if_included(o3d.utility.Vector3dVector(gt)))
    org = pred.min(0) - 5.0
    keys = {tuple(k) for k in np.floor((pred - org) / 10.0).astype(int)}
    assert np.array_equal(inc, np.array([tuple(k) in keys for k in np.floor((gt - org) / 10.0).astype(int)]))

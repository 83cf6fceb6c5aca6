"""Records what the original LiDiff code computes on the import shims, so the tests that compare against it run without it:

    python tests/golden/make_reference_goldens.py <path to a LiDiff checkout>

writes
  * tests/golden/reference_on_shims.json — the parameter names and shapes of the reference's MinkGlobalEnc / MinkUNetDiff /
    MinkUNet, every attribute of a shimmed package (MinkowskiEngine, open3d, diffusers, pytorch_lightning, natsort, pykeops) that
    its inference script, network module and metrics module name, and the outputs of its metrics (lidiff/utils/metrics.py) on
    seeded point clouds;
  * tests/golden/reference_diffcompletion.npz — the preprocessed scan and the two (refined, post) results of the reference's
    DiffCompletion.complete_scan on two consecutive scans under torch.manual_seed(123), from synthetic Lightning checkpoints.

Everything runs on the CPU: the CUDA library is replaced by tests/fake_backend.py and `.cuda()` by a no-op, as in the tests.
The mirror (lidiff_b200.pipeline.DiffCompletion) is checked to give the same bytes before anything is written.
"""
import ast
import importlib
import importlib.util
import json
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
sys.path[:0] = [ROOT, TESTS]

import lidiff_b200.shims as sh                                       # noqa: E402
from test_reference_on_shims import complete_two_scans, cpu_only, lightning_checkpoints    # noqa: E402

SHIMMED = ("MinkowskiEngine", "open3d", "diffusers", "pytorch_lightning", "natsort", "pykeops")


def drop_modules(*names):
    for k in [k for k in sys.modules if any(k == m or k.startswith(m + ".") for m in names)]:
        sys.modules.pop(k)


def shim_names(path):
    """dotted names of shimmed-package attributes a source file reaches through its import aliases (`ME.utils.batched_coordinates`,
    `o3d.geometry.PointCloud`, `from diffusers import X` -> `diffusers.X`)"""
    tree = ast.parse(open(path).read())
    alias, names = {}, set()
    for node in ast.walk(tree):
        if isinstance(node, ast.Import):
            for a in node.names:
                if a.name.split(".")[0] in SHIMMED:
                    alias[a.asname or a.name.split(".")[0]] = a.name if a.asname else a.name.split(".")[0]
                    names.add(a.name)
        elif isinstance(node, ast.ImportFrom) and node.module and node.module.split(".")[0] in SHIMMED:
            for a in node.names:
                alias[a.asname or a.name] = f"{node.module}.{a.name}"
                names.add(f"{node.module}.{a.name}")
    for node in ast.walk(tree):
        if isinstance(node, ast.Attribute):
            chain, n = [], node
            while isinstance(n, ast.Attribute):
                chain.append(n.attr)
                n = n.value
            if isinstance(n, ast.Name) and n.id in alias:
                names.add(".".join([alias[n.id]] + chain[::-1]))
    # keep the longest chains only: resolving a.b.c resolves a.b
    return sorted(x for x in names if not any(y.startswith(x + ".") for y in names))


def state_dict_shapes(ref):
    sh.install()
    spec = importlib.util.spec_from_file_location("ref_minkunet", os.path.join(ref, "lidiff/models/minkunet.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return {name: {k: list(v.shape) for k, v in getattr(mod, name)(in_channels=3, **kw).state_dict().items()}
            for name, kw in (("MinkGlobalEnc", {}), ("MinkUNetDiff", {}), ("MinkUNet", {"out_channels": 18}))}


def metrics_outputs(ref):
    """the seeded point clouds of tests/test_shims.py through the reference's metric classes"""
    sh.install()
    drop_modules("open3d", "lidiff")
    sys.path.insert(0, ref)
    try:
        import open3d as o3d
        metrics = importlib.import_module("lidiff.utils.metrics")
        metrics.torch = torch                                     # the module uses `torch.Tensor` without importing torch
        g = np.random.default_rng(3)
        gt = g.normal(size=(6000, 3)) * [12, 12, 1.0]
        pred = gt[g.choice(6000, 4000, replace=False)] + g.normal(size=(4000, 3)) * 0.05
        pg, pp = o3d.geometry.PointCloud(gt), o3d.geometry.PointCloud(pred)
        cd, rm = metrics.ChamferDistance(), metrics.RMSE()
        cd.update(pg, pp); rm.update(pg, pp)
        pr = metrics.PrecisionRecall(0.05, 1.0, 20)
        pr.update(pg, pp)
        iou = metrics.CompletionIoU(voxel_sizes=[2.0, 1.0, 0.5])
        iou.update(pg, pp)
        return {"chamfer": [float(x) for x in cd.compute()], "rmse": [float(x) for x in rm.compute()],
                "precision_recall_at_0.1": [float(x) for x in pr.compute_at_threshold(0.1)],
                "precision_recall_auc": [float(x) for x in pr.compute_auc()],
                "completion_iou": {str(k): float(v) for k, v in iou.compute().items()},
                "prediction_is_empty": [bool(metrics.Metrics3D().prediction_is_empty(pp)),
                                        bool(metrics.Metrics3D().prediction_is_empty(np.zeros((0, 3))))]}
    finally:
        sys.path.remove(ref)
        drop_modules("lidiff")


def diffcompletion_outputs(ref, tmp):
    from lidiff_b200.pipeline import DiffCompletion as Mirror
    from lidiff_b200.synth import synthetic_scan
    from oracle.pipeline import farthest_point_sample as fps_cpu
    with pytest.MonkeyPatch.context() as mp:
        cpu_only(mp, tmp)
        sys.path.insert(0, ref)
        drop_modules("lidiff")
        try:
            mod = importlib.import_module("lidiff.tools.diff_completion_pipeline")

            def fps(self, n):                     # open3d's farthest point sampling is a CUDA kernel in the shim: the oracle's CPU one
                pts = np.asarray(self.points)
                return type(self)(pts[fps_cpu(pts, int(n))])
            mp.setattr(mod.o3d.geometry.PointCloud, "farthest_point_down_sample", fps)
            n_points = 2000
            diff_path, refine_path = lightning_checkpoints(tmp, n_points)
            raw = synthetic_scan(9, beams=16, azimuths=256)
            r = mod.DiffCompletion(diff_path, refine_path, 2, 6.0)
            pre = r.preprocess_scan(raw)
            out_ref = complete_two_scans(r, raw)
            out_mir = complete_two_scans(Mirror(diff_path, refine_path, 2, 6.0, device="cpu", engine=False), pre, preprocessed=True)
        finally:
            sys.path.remove(ref)
            drop_modules("lidiff")
    for (ra, pa), (rb, pb) in zip(out_ref, out_mir):
        assert pa.shape == pb.shape and np.array_equal(pa, pb) and np.array_equal(ra, rb), "reference on shims vs mirror"
    z = {"pre": pre.numpy()}
    for n, (refined, post) in enumerate(out_ref):
        z[f"refined{n}"], z[f"post{n}"] = refined, post
    return z


def main():
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    ref = os.path.abspath(sys.argv[1])
    import tempfile
    torch.set_num_threads(os.cpu_count() or 1)
    out = {"state_dict_shapes": state_dict_shapes(ref),
           "shim_names": {f: shim_names(os.path.join(ref, f)) for f in
                          ("lidiff/tools/diff_completion_pipeline.py", "lidiff/models/minkunet.py", "lidiff/utils/metrics.py")},
           "metrics": metrics_outputs(ref)}
    with open(os.path.join(HERE, "reference_on_shims.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    with tempfile.TemporaryDirectory() as tmp:
        z = diffcompletion_outputs(ref, tmp)
    np.savez_compressed(os.path.join(HERE, "reference_diffcompletion.npz"), **z)
    print("wrote reference_on_shims.json and reference_diffcompletion.npz")


if __name__ == "__main__":
    main()

"""The reference's OWN inference class on the import shims (SURVEY.md 8f-1, a16; VERDICT r1 item 8), recorded in
tests/golden/reference_diffcompletion.npz by tests/golden/make_reference_goldens.py: LiDiff's `DiffCompletion(diff_path,
refine_path, T, s)` built from synthetic Lightning-format checkpoints (ctor :15-56: torch.load, save_hyperparameters, strict=False
state-dict loads, scheduler construction) ran `complete_scan(points)` (:117-169) end to end — preprocess (open3d FPS),
points_to_tensor, the guided sampling loop over the ME / diffusers shims, postprocess, refinement, 6x offsets — for two consecutive
scans under one torch seed (the reference never resets its scheduler between scans).  This repo's mirror
`lidiff_b200.pipeline.DiffCompletion` must give the same point counts and the same points (within TOL_M) from the same
checkpoints and the same preprocessed scan.

The CUDA library is replaced by tests/fake_backend.py (CPU stand-in under the same C-ABI-shaped handle) and `.cuda()` is a no-op:
what runs is every line of the mirror's host code and of the shims; the kernels themselves are covered by the -m gpu suites."""
import os
import sys

import numpy as np
import pytest
import torch

import fake_backend
from conftest import make_scan

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_diffcompletion.npz")
# On the machine and thread count that recorded the reference, the mirror reproduces it bit for bit.  Elsewhere MKL's kernel
# choice and the thread count reorder fp32 sums: 0.09 mm is the largest deviation seen over AVX-512 / AVX2 / SSE4.2 BLAS and
# 1 / 3 / 8 threads.  The point counts after postprocess must match exactly.
TOL_M = 1e-3


def cpu_only(mp, tmp):
    """shims on the path, the fake CUDA backend, `.cuda()` / `.to('cuda')` kept on the CPU, cwd in `tmp`"""
    import lidiff_b200.shims as sh
    sh.install()
    for m in ("open3d", "natsort", "pytorch_lightning", "MinkowskiEngine", "diffusers", "pykeops"):
        for k in [k for k in sys.modules if k == m or k.startswith(m + ".")]:
            sys.modules.pop(k)
    fake_backend.install(mp)
    mp.setattr(torch.Tensor, "cuda", lambda self, *a, **k: self)
    mp.setattr(torch.nn.Module, "cuda", lambda self, *a, **k: self)
    orig_to = torch.Tensor.to

    def to_cpu_instead_of_cuda(self, *a, **k):                                      # minkunet.py:395 `.to(torch.device('cuda'))`
        is_cuda = lambda x: (isinstance(x, torch.device) and x.type == "cuda") or (isinstance(x, str) and x.startswith("cuda"))
        a = tuple(torch.device("cpu") if is_cuda(x) else x for x in a)
        if is_cuda(k.get("device")):
            k["device"] = torch.device("cpu")
        return orig_to(self, *a, **k)
    mp.setattr(torch.Tensor, "to", to_cpu_instead_of_cuda)
    mp.chdir(tmp)                                                                   # the reference's ctor writes ./results/<exp>/


def lightning_checkpoints(tmp_path, n_points):
    """what LiDiff's training writes: {'hyper_parameters': config.yaml dict, 'state_dict': {<submodule>.<param>: tensor}}"""
    from oracle.pipeline import calibrated_state_dicts
    scan = make_scan(n_points // 10, 4)
    sds = calibrated_state_dicts(scan, seed=3)
    hp = {"experiment": {"id": "test"},
          "data": {"resolution": 0.05, "num_points": n_points, "max_range": 50.0, "dataloader": "KITTI"},
          "train": {"uncond_w": 6.0, "uncond_prob": 0.1, "lr": 1e-4},
          "diff": {"beta_start": 3.5e-5, "beta_end": 0.007, "beta_func": "linear", "t_steps": 1000, "s_steps": 50, "reg_weight": 5.0},
          "model": {"out_dim": 96}}
    sd_diff = {f"partial_enc.{k}": v for k, v in sds["enc"].items()}
    sd_diff.update({f"model.{k}": v for k, v in sds["diff"].items()})
    sd_ref = {f"model_refine.{k}": v for k, v in sds["refine"].items()}
    d, r = os.path.join(str(tmp_path), "diff_net.ckpt"), os.path.join(str(tmp_path), "refine_net.ckpt")
    torch.save({"epoch": 19, "hyper_parameters": hp, "state_dict": sd_diff}, d)
    torch.save({"epoch": 5, "hyper_parameters": hp, "state_dict": sd_ref}, r)
    return d, r


def complete_two_scans(pipe, scan, **kw):
    torch.manual_seed(123)
    return [pipe.complete_scan(scan, **kw) for _ in range(2)]      # second scan: multistep state carried over (no reset)


def test_reference_diffcompletion_runs_on_shims_and_equals_the_mirror(monkeypatch, tmp_path):
    from lidiff_b200.pipeline import DiffCompletion as Mirror
    from lidiff_b200.synth import range_filter, synthetic_scan
    cpu_only(monkeypatch, tmp_path)
    z = np.load(GOLD)
    n_points = 2000
    diff_path, refine_path = lightning_checkpoints(tmp_path, n_points)
    raw = synthetic_scan(9, beams=16, azimuths=256)                           # (4096, 3) incl. points the range filter drops
    mir = Mirror(diff_path, refine_path, 2, 6.0, device="cpu", engine=False)
    assert mir.hparams["data"]["num_points"] == n_points
    assert mir.hparams["diff"]["s_steps"] == 2 and len(mir.dpm_scheduler.timesteps) == 2
    pre = torch.from_numpy(z["pre"])                                          # the reference's preprocess_scan(raw)
    assert tuple(pre.shape) == (1, n_points, 3) and pre.dtype == torch.float64
    assert pre.shape[1] == range_filter(raw).shape[0] or pre.shape[1] == n_points
    outs = complete_two_scans(mir, pre, preprocessed=True)
    for n, (refined, post) in enumerate(outs):
        assert refined.shape == (6 * post.shape[0], 3) and np.isfinite(refined).all() and post.shape[0] > 0
        for name, a in (("post", post), ("refined", refined)):
            b = z[f"{name}{n}"]
            assert a.shape == b.shape and a.dtype == b.dtype, f"scan {n}: {name} {a.shape} {a.dtype}, reference {b.shape} {b.dtype}"
            err = float(np.abs(a.astype(np.float64) - b).max())
            print(f"scan {n}: {name} max |mirror - reference| = {err:.3e} m")
            assert err <= TOL_M, f"scan {n}: {name}, mirror vs reference on shims"
    assert not np.array_equal(outs[0][1], outs[1][1])                         # the two scans drew different noise

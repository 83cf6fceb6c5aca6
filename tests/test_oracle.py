"""CPU tests: the oracle against the committed known-answer values and structural invariants, and the
host-side logic of the product against the oracle.  No GPU needed."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import me_cpu as ome
from oracle import nets as onets
from oracle.dpm import DPMSolverSDE2M
from oracle.pipeline import DiffCompletionOracle, farthest_point_sample

GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "known_answers.json")))


def test_timestep_tables_match_golden():
    d = DPMSolverSDE2M()
    d.set_timesteps(50)
    assert d.timesteps.tolist() == GOLD["timesteps_50"]
    d.set_timesteps(1000)
    assert len(d.timesteps) == GOLD["timesteps_1000_len"]
    assert d.timesteps[:3].tolist() == GOLD["timesteps_1000_head"] and d.timesteps[-3:].tolist() == GOLD["timesteps_1000_tail"]
    d.set_timesteps(1)
    assert d.timesteps.tolist() == GOLD["timesteps_1"]
    for t, row in GOLD["tables"].items():
        t = int(t)
        assert float(d.alphas_cumprod[t]) == row["alphas_cumprod"]
        assert float(d.alpha_t[t]) == row["alpha_t"] and float(d.sigma_t[t]) == row["sigma_t"]
        assert float(d.lambda_t[t]) == row["lambda_t"]


def test_dpm_coefficients_match_golden():
    d = DPMSolverSDE2M()
    d.set_timesteps(50)
    for idx, key in ((0, "step_999_979"), (49, "step_20_0")):
        c = d.coefficients(idx)
        for k in ("h", "c_sample", "c_x0", "c_noise"):
            assert float(c[k]) == GOLD[key][k], (key, k)


def test_time_embedding_and_rounding_match_golden():
    e = onets.Net({}).timestep_embedding(torch.tensor([999]))[0]
    assert e[:4].tolist() == GOLD["temb_999_0_4"] and e[48:52].tolist() == GOLD["temb_999_48_52"]
    q = ome.quantize(torch.tensor([0.5, 1.5, 2.5, -0.5, -1.5]) * 0.05, 0.05, "div")
    assert q.tolist() == GOLD["round_half_even"]


def test_parameter_counts_match_reference():
    def n(sd):
        return sum(v.numel() for k, v in sd.items() if "running" not in k and "num_batches" not in k)
    assert n(onets.random_state_dict("diff")) == GOLD["param_counts"]["diff"]
    assert n(onets.random_state_dict("enc")) == GOLD["param_counts"]["enc"]
    assert n(onets.random_state_dict("refine", out_channels=18)) == GOLD["param_counts"]["refine18"]


def test_first_step_is_closed_form():
    """one first-order SDE step equals c_sample*s + c_x0*x0 + c_noise*z with the golden coefficients"""
    d = DPMSolverSDE2M()
    d.set_timesteps(50)
    g = torch.Generator().manual_seed(0)
    s = torch.randn(1, 64, 3, generator=g, dtype=torch.float64)
    eps = torch.randn(1, 64, 3, generator=g)
    z = torch.randn(1, 64, 3, generator=g)
    out = d.step(eps, 999, s, z)
    G = GOLD["step_999_979"]
    a, sg = GOLD["tables"]["999"]["alpha_t"], GOLD["tables"]["999"]["sigma_t"]
    x0 = (s - (torch.tensor(sg, dtype=torch.float32) * eps)) / torch.tensor(a, dtype=torch.float32)
    ref = G["c_sample"] * s + G["c_x0"] * x0 + (torch.tensor(G["c_noise"], dtype=torch.float32) * z).double()   # fp32 noise term (diffusers)
    assert torch.allclose(out, ref, rtol=0, atol=1e-12)


# ---- structural invariants of the sparse ops ---------------------------------------------------------
def _field_from_int_coords(C, F):
    return ome.TensorField(F, torch.cat([torch.zeros(C.shape[0], 1), C.float()], 1))


def test_sparse_conv_equals_dense_conv_on_full_grid():
    """on a completely filled cube a 3^3 sparse conv is a zero-padded dense cross-correlation"""
    n = 6
    zz, yy, xx = torch.meshgrid(torch.arange(n), torch.arange(n), torch.arange(n), indexing="ij")
    C = torch.stack([xx.reshape(-1), yy.reshape(-1), zz.reshape(-1)], 1)
    g = torch.Generator().manual_seed(1)
    F = torch.randn(C.shape[0], 4, generator=g, dtype=torch.float64)
    W = torch.randn(27, 4, 5, generator=g, dtype=torch.float64)
    x = _field_from_int_coords(C, F).sparse()
    y = ome.conv(x, W, 3)
    dense_in = F.reshape(n, n, n, 4).permute(3, 0, 1, 2)[None]              # (1,C,z,y,x)
    Wd = W.reshape(3, 3, 3, 4, 5).permute(4, 3, 0, 1, 2)                    # k = kx + 3ky + 9kz -> [kz][ky][kx]
    ref = torch.nn.functional.conv3d(dense_in, Wd, padding=1)[0].permute(1, 2, 3, 0).reshape(-1, 5)
    assert torch.allclose(y.F, ref, atol=1e-10)


def test_stride2_conv_and_transpose_are_adjoint():
    """<conv_s2(x), y> == <x, convT_s2(y)> with the same kernel: the transposed map is the swapped map"""
    g = torch.Generator().manual_seed(2)
    C = torch.randint(-9, 9, (300, 3), generator=g)
    F = torch.randn(300, 3, generator=g, dtype=torch.float64)
    x = _field_from_int_coords(C, F).sparse()
    W = torch.randn(8, 3, 6, generator=g, dtype=torch.float64)
    y = ome.conv(x, W, 2, stride=2)
    assert y.ts == 2 and (y.C[:, 1:] % 2 == 0).all()
    Y = torch.randn(y.F.shape, generator=g, dtype=torch.float64)
    back = ome.conv(y.replace(Y), W.transpose(1, 2).contiguous(), 2, stride=2, transposed=True)
    assert back.ts == 1 and back.F.shape == (x.F.shape[0], 3)
    assert torch.allclose((y.F * Y).sum(), (x.F * back.F).sum(), atol=1e-9)
    # every fine row has exactly one (coarse, k) parent
    maps = x.geom.kernel_map(2, 2, 2, True)
    assert sum(m[0].shape[0] for m in maps) == x.F.shape[0]


def test_voxelise_first_occurrence_order_and_mean():
    Cf = torch.tensor([[0, 5, 5, 5], [0, 1, 1, 1], [0, 5, 5, 5], [0, -3, 0, 2], [0, 1, 1, 1]], dtype=torch.float32)
    F = torch.arange(15, dtype=torch.float32).reshape(5, 3)
    s = ome.TensorField(F, Cf).sparse()
    assert s.C.tolist() == [[0, 5, 5, 5], [0, 1, 1, 1], [0, -3, 0, 2]]
    assert s.geom.inverse.tolist() == [0, 1, 0, 2, 1]
    assert torch.equal(s.F, torch.stack([(F[0] + F[2]) / 2, (F[1] + F[4]) / 2, F[3]]))
    lvl = s.geom.stride_level(2)
    assert lvl.tolist() == [[0, 4, 4, 4], [0, 0, 0, 0], [0, -4, 0, 2]]          # true floor for negatives


def test_argkmin_ties_pick_lowest_index():
    q = torch.tensor([[0, 0, 0, 0], [0, 4, 0, 0]])
    k = torch.tensor([[0, 2, 0, 0], [0, -2, 0, 0], [0, 2, 0, 0]])
    assert ome.match_part_to_full(q, k).tolist() == [0, 0]


def test_fps_matches_definition():
    g = np.random.default_rng(0)
    p = g.normal(size=(200, 3))
    sel = farthest_point_sample(p, 10)
    assert 0 in sel and len(set(sel.tolist())) == 10 and (np.diff(sel) > 0).all()


# ---- host logic of the product vs oracle ---------------------------------------------------------------
def test_product_scheduler_equals_oracle_bitwise():
    from lidiff_b200.scheduler import DPMSolverMultistepScheduler as S
    s = S(1000, 3.5e-5, 0.007, "linear", algorithm_type="sde-dpmsolver++", solver_order=2)
    for T in (50, 5):
        s.set_timesteps(T)
        o = DPMSolverSDE2M()
        o.set_timesteps(T)
        g = torch.Generator().manual_seed(T)
        x = torch.randn(1, 50, 3, dtype=torch.float64, generator=g)
        for i in range(T):
            eps, nz = torch.randn(1, 50, 3, generator=g), torch.randn(1, 50, 3, generator=g)
            a = s.step(eps, s.timesteps[i], x, noise=nz)["prev_sample"]
            b = o.step(eps, o.timesteps[i], x, nz)
            assert torch.equal(a, b), (T, i)
            x = a


def test_scheduler_rejects_other_configurations():
    from lidiff_b200.scheduler import DPMSolverMultistepScheduler as S
    with pytest.raises(NotImplementedError):
        S(1000, 1e-4, 0.02, "linear", algorithm_type="dpmsolver++")


def test_module_tree_has_reference_state_dict_keys():
    from lidiff_b200 import minkunet as mk
    for kind, cls, kw in (("enc", mk.MinkGlobalEnc, {}), ("diff", mk.MinkUNetDiff, {}), ("refine", mk.MinkUNet, {"out_channels": 18})):
        sd = cls(in_channels=3, **kw).state_dict()
        osd = onets.random_state_dict(kind, out_channels=kw.get("out_channels", 3))
        assert set(sd) == set(osd)
        assert all(tuple(sd[k].shape) == tuple(osd[k].shape) for k in sd)


def test_reference_minkunet_builds_on_shims_with_same_keys():
    """parameter names and shapes of the reference's MinkGlobalEnc / MinkUNetDiff / MinkUNet built on the shims (recorded in
    tests/golden/reference_on_shims.json by tests/golden/make_reference_goldens.py) are those of lidiff_b200.minkunet"""
    from lidiff_b200 import minkunet as mk
    ref = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_on_shims.json")))["state_dict_shapes"]
    for name, kw in (("MinkGlobalEnc", {}), ("MinkUNetDiff", {}), ("MinkUNet", {"out_channels": 18})):
        a = ref[name]
        b = getattr(mk, name)(in_channels=3, **kw).state_dict()
        assert set(a) == set(b) and all(tuple(a[k]) == tuple(b[k].shape) for k in a)


def test_oracle_end_to_end_small(small_scan, calibrated_sds):
    """two denoising steps (first + second order) and the refinement forward run and stay finite"""
    sd = calibrated_sds
    o = DiffCompletionOracle(sd["enc"], sd["diff"], sd["refine"], denoising_steps=50)
    scan = small_scan[:, ::5].contiguous()
    g = torch.Generator().manual_seed(3)
    start = torch.randn(scan.shape, generator=g)
    noise = torch.randn((2,) + tuple(scan.shape), generator=g)
    x_t, x_c, x_u = o.points_to_tensor(scan + start), o.points_to_tensor(scan), o.points_to_tensor(torch.zeros_like(scan))
    out = o.completion_loop(scan, x_t, x_c, x_u, noise, n_steps=2)
    assert out.shape == (scan.shape[1], 3) and np.isfinite(out).all()
    ref = o.refine.unet_refine(o.points_to_tensor(torch.from_numpy(out)[None]))
    assert ref.shape == (scan.shape[1], 18) and torch.isfinite(ref).all() and ref.abs().max() <= 1


def test_nn_match_against_scipy_kdtree():
    """independent check of the argKmin restatement (minkunet.py:403-418): scipy's exact k-d tree gives the same nearest distance
    for every query, and the same index wherever the nearest key is unique"""
    from scipy.spatial import cKDTree
    g = torch.Generator().manual_seed(21)
    keys = torch.cat([torch.zeros(3000, 1), torch.round(torch.randn(3000, 3, generator=g) * torch.tensor([300.0, 300.0, 30.0]) / 16) * 16], 1)
    q = torch.cat([torch.zeros(20000, 1), torch.round(torch.randn(20000, 3, generator=g) * torch.tensor([320.0, 320.0, 35.0]))], 1)
    idx = ome.match_part_to_full(q, keys).numpy()
    d_ref, i_ref = cKDTree(keys[:, 1:].numpy().astype(np.float64)).query(q[:, 1:].numpy().astype(np.float64), k=2)
    d_or = np.linalg.norm(q[:, 1:].numpy().astype(np.float64) - keys[idx, 1:].numpy().astype(np.float64), axis=1)
    assert np.array_equal(d_or, d_ref[:, 0])
    unique = d_ref[:, 1] > d_ref[:, 0]
    assert unique.mean() > 0.9 and np.array_equal(idx[unique], i_ref[unique, 0])
    ties = ~unique                                                          # among equidistant keys the lowest index wins (App. A.10)
    assert np.all(idx[ties] <= i_ref[ties].min(1))

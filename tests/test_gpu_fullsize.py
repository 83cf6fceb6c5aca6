"""Parity at the benchmark configuration and on the reference's own fixture (SURVEY.md 8d configs 1/2, VERDICT r1 item 2):
one engine step at N = 180 000 points against the committed oracle goldens (tests/golden/step_*.npz, written by
tests/golden/make_step_goldens.py with the CPU oracle; the oracle needs minutes per step at this size, the test seconds).
eps and x_next are compared on every 8th row, the refinement offsets on every 16th point, plus fp64 sums over the full arrays.

  * coordinates: level row counts, key checksums (sum and xor of the packed 64-bit keys of every level) and 3^3 pair counts
    BIT-EXACT;
  * guided eps and the update x_next - x_t: per element |a - b| <= 1e-3 (|b| + rms(b))  (SURVEY.md 8c-iii, north star 1e-3);
  * the refinement forward (MinkUNet, 6 offsets per point) through the fused engine: same rule.
The conv / linear weights are re-created from their seeds and checked against the digest in the fixture; the calibrated BatchNorm
tensors, the conditioning points and the digests of the noise tensors come from the fixture.
"""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def rule_violations(a, b, tol=1e-3):
    """fraction of elements outside |a-b| <= tol*(|b| + rms(b)) and the largest ratio"""
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    r = (a - b).abs() / (b.abs() + b.pow(2).mean().sqrt() + 1e-30)
    return float((r > tol).double().mean()), float(r.max())


def conditioning_points(z):
    """the 18 000 conditioning points (fp64): the synthetic scan's are regenerated from its seed and picked by index"""
    if "part_index" in z:
        from lidiff_b200.synth import range_filter, synthetic_scan
        return range_filter(synthetic_scan(0))[z["part_index"]]
    return z["part"].astype(np.float64)


def load_case(name):
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_step_goldens", os.path.join(GOLD, "make_step_goldens.py"))
    mk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mk)
    z = np.load(os.path.join(GOLD, f"step_{name}.npz"))
    sds = mk.seeded_state_dicts(0)
    assert mk.weights_digest(sds) == str(z["weights_digest"]), \
        "seeded weights differ from the ones the golden was computed with (torch CPU RNG changed?): regenerate the goldens"
    off = 0
    for key, size in zip(z["bn_keys"].tolist(), z["bn_sizes"].tolist()):
        net, k = key.split("/", 1)
        sds[net][k] = torch.from_numpy(z["bn_vals"][off:off + size].copy()).reshape(sds[net][k].shape)
        off += size
    scan = torch.tensor(conditioning_points(z)).repeat(10, 1)[None]
    start, step = mk.noises(scan.shape, 1234)
    assert mk.digest(start) == str(z["start_digest"]) and mk.digest(step) == str(z["step_digest"]), "seeded noise differs from the golden's"
    return z, sds, scan, start, step, mk


def packed_keys(C: np.ndarray) -> np.ndarray:
    C = C.astype(np.int64)
    off = 1 << 17
    return ((C[:, 0] << 54) | ((C[:, 1] + off) << 36) | ((C[:, 2] + off) << 18) | (C[:, 3] + off)).astype(np.uint64)


@pytest.mark.parametrize("case", ["synth180k", "000123"])
def test_engine_step_at_180k_points_matches_oracle_golden(case):
    from lidiff_b200.engine import DenoiseEngine
    z, sds, scan, start, step, _ = load_case(case)
    N, T, stride = scan.shape[1], int(z["T"]), int(z["stride"])
    assert N == 180_000
    eng = DenoiseEngine(sds["enc"], sds["diff"], device=DEV, n_points=N, denoising_steps=T)
    st = eng.start(scan, scan + start)
    x_t = st["xa"].clone()
    eps = torch.empty((N, 3), device=DEV)
    eng.step(0, st["xa"], st["xb"], st["ca"], st["cb"], st["x_init"], step[0, 0].to(DEV).contiguous(), st["x0s"], eps_out=eps)
    torch.cuda.synchronize()
    assert eng.h.read_status() == 0
    g = eng.geom
    rows = g.sizes()
    assert rows == z["level_rows"].tolist(), "level row counts"
    for l in range(5):
        keys = packed_keys(g.C[l][:rows[l]].cpu().numpy())
        assert int(keys.sum(dtype=np.uint64)) == int(z["level_key_sum"][l]) and int(np.bitwise_xor.reduce(keys)) == int(z["level_key_xor"][l]), f"level {l} coordinates"
    assert g.pairs[:5].tolist() == z["pairs3"].tolist(), "3^3 kernel-map pair counts"
    frac, worst = rule_violations(eps[::stride], z["eps"])
    upd = (st["xb"] - x_t)[::stride]
    upd_ref = torch.from_numpy(z["x_next"]) - x_t[::stride].cpu()
    frac_x, worst_x = rule_violations(upd, upd_ref)
    s = float(eps.double().sum())
    print(f"{case}: rows {rows}; eps worst ratio {worst:.2e} (violations {frac:.1e}), update worst {worst_x:.2e}; eps sum {s:.4f} vs {float(z['eps_sum']):.4f}")
    assert worst <= 1e-3, "guided eps vs oracle at 180k points (|a-b| <= 1e-3 (|b| + rms))"
    assert worst_x <= 1e-3, "x_next - x_t vs oracle"
    assert abs(s - float(z["eps_sum"])) <= 1e-3 * float(z["eps_abs_sum"])


def test_refinement_forward_matches_oracle_golden():
    """MinkUNet refinement forward + slice through the fused engine on the 180k-point reference scan (decoupled from the diffusion
    result: input = conditioning scan + 2 cm seeded noise, as in make_step_goldens.py)"""
    from lidiff_b200.engine import DenoiseEngine
    z, sds, scan, _, _, mk = load_case("000123")
    z = np.load(os.path.join(GOLD, "step_000123_refine.npz"))
    rin = (scan + 0.02 * torch.randn(scan.shape, generator=torch.Generator().manual_seed(99), dtype=scan.dtype)).float()
    assert mk.digest(rin) == str(z["refine_in_digest"])
    eng = DenoiseEngine(sds["enc"], sds["diff"], device=DEV, n_points=scan.shape[1], denoising_steps=1, sd_refine=sds["refine"])
    off = eng.refine_offsets(rin[0].to(DEV)).reshape(-1, 6, 3)
    torch.cuda.synchronize()
    frac, worst = rule_violations(off[::int(z["refine_stride"])], z["refine_offsets"])
    tot = float(off.double().abs().sum())
    print(f"refinement offsets: worst ratio {worst:.2e}, |sum| {tot:.3f} vs {float(z['refine_offsets_abs_sum']):.3f}")
    assert worst <= 1e-3
    assert abs(tot - float(z["refine_offsets_abs_sum"])) <= 1e-3 * float(z["refine_offsets_abs_sum"])


def test_complete_scan_chain_on_reference_fixture():
    """T=1 on 000123.ply: loop + postprocess + refinement + 6 offsets on the device; the surviving point count may differ from the
    oracle's only by points whose z / range sits within the fp32 tolerance of a threshold"""
    from lidiff_b200.engine import DenoiseEngine
    z, sds, scan, start, step, _ = load_case("000123")
    eng = DenoiseEngine(sds["enc"], sds["diff"], device=DEV, n_points=scan.shape[1], denoising_steps=1, sd_refine=sds["refine"])
    refined, post = eng.complete(scan, scan + start, step[:, 0].to(DEV))
    n_ref = int(z["post_rows"])
    print(f"complete(): {post.shape[0]} points survive postprocess (oracle {n_ref}); refined {refined.shape[0]}")
    assert refined.shape[0] == 6 * post.shape[0] and torch.isfinite(refined).all()
    assert abs(post.shape[0] - n_ref) <= 20

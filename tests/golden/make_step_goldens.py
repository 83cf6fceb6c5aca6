"""Generates the full-size step goldens the GPU parity tests are diffed against (SURVEY.md 8d configs 1 and 2, VERDICT r1 item 2):

    python tests/golden/make_step_goldens.py synth180k     # BASELINE configs[1] geometry: synthetic KITTI-shape scan, 180 000 points,
                                                           # first step of the T=50 schedule   -> tests/golden/step_synth180k.npz
    python tests/golden/make_step_goldens.py ply000123 <LiDiff checkout>/lidiff/Datasets/test/000123.ply
                                                           # the reference's own fixture preprocessed per
                                                           # tools/diff_completion_pipeline.py:92-105, T=1 (timesteps [999]) + refinement
                                                           #       -> tests/golden/step_000123.npz, tests/golden/step_000123_refine.npz

Everything is computed by the CPU oracle (fp32, `oracle/`) — about 2-4 minutes per case on 8 cores — so the tests only load the
result.  To keep the fixtures under 1 MB each they hold: the 18 000 conditioning points (for the synthetic scan their indices into
range_filter(synthetic_scan(0)), for the .ply its float32 values), the calibrated BatchNorm tensors (the conv / linear weights are
re-created from their seeds on the test machine and checked against a digest), digests of the noise tensors, per-level row counts
+ key checksums + pair counts (bit-exact quantities), every 8th row of eps / x_next, every 16th point of the refinement offsets
(in a file of their own), plus fp64 sums over the full arrays.  The .ply is read here only; the tests never need it.
"""
import hashlib
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import me_cpu as ome                                     # noqa: E402
from oracle.nets import random_state_dict                            # noqa: E402
from oracle.pipeline import DiffCompletionOracle, farthest_point_sample    # noqa: E402

STRIDE = 8
REFINE_STRIDE = 16


def digest(*tensors) -> str:
    h = hashlib.sha256()
    for t in tensors:
        h.update(np.ascontiguousarray(torch.as_tensor(t).detach().cpu().numpy()).tobytes())
    return h.hexdigest()


def seeded_state_dicts(seed=0):
    return dict(enc=random_state_dict("enc", seed), diff=random_state_dict("diff", seed + 1),
                refine=random_state_dict("refine", seed + 2, out_channels=18))


def weights_digest(sds) -> str:
    """digest of every tensor that is NOT a BatchNorm tensor (those travel in the fixture)"""
    ts = []
    for name in ("enc", "diff", "refine"):
        for k in sorted(sds[name]):
            if ".bn." not in k:
                ts.append(sds[name][k])
    return digest(*ts)


def calibrate(sds, scan, seed=0, sigma=0.5):
    """oracle.pipeline.calibrated_state_dicts on given state dicts: one forward sets the BN running stats"""
    g = torch.Generator().manual_seed(seed + 17)
    o = DiffCompletionOracle(sds["enc"], sds["diff"], sds["refine"])
    for n in (o.enc, o.diff, o.refine):
        n.calibrate, n.rng = True, g
    noisy = scan + sigma * torch.randn(scan.shape, generator=g, dtype=scan.dtype)
    x_t, x_c = o.points_to_tensor(noisy), o.points_to_tensor(scan)
    o.forward(x_t, x_t.sparse(), x_c, torch.tensor([500] * scan.shape[0]))
    o.refine.unet_refine(o.points_to_tensor(scan + 0.05 * torch.randn(scan.shape, generator=g, dtype=scan.dtype)))


def noises(shape, seed):
    g = torch.Generator().manual_seed(seed)
    start = torch.randn(shape, generator=g)
    step = torch.randn((1, 1) + tuple(shape[1:]), generator=g)
    return start, step


def level_stats(geom):
    rows, ksum, kxor, pairs = [], [], [], []
    for l in range(5):
        C = geom.stride_level(1 << l)
        keys = ome.pack_keys(C).astype(np.uint64)
        rows.append(C.shape[0])
        ksum.append(int(keys.sum(dtype=np.uint64)))
        kxor.append(int(np.bitwise_xor.reduce(keys)))
        pairs.append(int(sum(len(i) for i, _ in geom.kernel_map(1 << l, 3, 1))))
    return np.array(rows, np.int64), np.array(ksum, np.uint64), np.array(kxor, np.uint64), np.array(pairs, np.int64)


def main(case, ply=None):
    torch.set_num_threads(os.cpu_count() or 1)
    t0 = time.time()
    if case == "synth180k":
        from lidiff_b200.synth import range_filter, synthetic_scan
        raw = range_filter(synthetic_scan(0))
        T, refine = 50, False
    elif case == "ply000123":
        from lidiff_b200.synth import range_filter, read_ply_xyz
        raw = range_filter(read_ply_xyz(ply))
        T, refine = 1, True
    else:
        raise SystemExit(__doc__)
    print(f"{case}: {raw.shape[0]} points after the range filter; farthest point sampling to 18000 ...", flush=True)
    sel = farthest_point_sample(raw, 18000)
    part = raw[sel]
    scan = torch.tensor(part).repeat(10, 1)[None]                      # (1, 180000, 3) f64
    print(f"  FPS done ({time.time() - t0:.0f} s); calibrating BN", flush=True)
    sds = seeded_state_dicts(0)
    wd = weights_digest(sds)
    calibrate(sds, scan)
    start, step = noises(scan.shape, 1234)
    o = DiffCompletionOracle(sds["enc"], sds["diff"], sds["refine"], denoising_steps=T, cond_weight=6.0)
    x_t, x_c, x_u = o.points_to_tensor(scan + start), o.points_to_tensor(scan), o.points_to_tensor(torch.zeros_like(scan))
    print(f"  oracle step ({time.time() - t0:.0f} s)", flush=True)
    t1 = time.time()
    completed = o.completion_loop(scan, x_t, x_c, x_u, step, n_steps=1)
    t_step = time.time() - t1
    hist = o.trace["hist"][0]
    eps, x_next = hist["eps"][0].float(), hist["x_next"][0].float()
    rows, ksum, kxor, pairs = level_stats(o.trace["geom"])
    # the synthetic scan is regenerated from its seed on the test machine: its indices are enough; the .ply holds float32 values
    stored = dict(part_index=np.asarray(sel, np.int32)) if case == "synth180k" else dict(part=part.astype(np.float32))
    assert case == "synth180k" or np.array_equal(stored["part"].astype(np.float64), part)
    out = dict(**stored, stride=np.int64(STRIDE), weights_digest=np.array(wd), start_digest=np.array(digest(start)), step_digest=np.array(digest(step)),
               T=np.int64(T), level_rows=rows, level_key_sum=ksum, level_key_xor=kxor, pairs3=pairs,
               eps=eps[::STRIDE].numpy(), x_next=x_next[::STRIDE].numpy(),
               eps_sum=np.float64(eps.double().sum()), eps_abs_sum=np.float64(eps.double().abs().sum()),
               x_next_sum=np.float64(x_next.double().sum()), oracle_step_seconds=np.float64(t_step), oracle_threads=np.int64(torch.get_num_threads()))
    bn_keys, bn_vals = [], []
    for name in ("enc", "diff", "refine"):
        for k in sorted(sds[name]):
            if ".bn." in k and "num_batches" not in k:
                bn_keys.append(f"{name}/{k}")
                bn_vals.append(sds[name][k].detach().float().numpy().ravel())
    out["bn_keys"] = np.array(bn_keys)
    out["bn_sizes"] = np.array([v.size for v in bn_vals], np.int64)
    out["bn_vals"] = np.concatenate(bn_vals)
    name = "000123" if case == "ply000123" else case
    if refine:
        post = o.postprocess_scan(completed, scan)
        off = o.refine.unet_refine(o.points_to_tensor(torch.from_numpy(post)[None, :, :])).reshape(-1, 6, 3)
        out["post_rows"] = np.int64(post.shape[0])
        out["offsets_abs_sum"] = np.float64(off.double().abs().sum())
        # refinement parity decoupled from the diffusion result: input = conditioning scan + 2 cm seeded noise
        rin = (scan + 0.02 * torch.randn(scan.shape, generator=torch.Generator().manual_seed(99), dtype=scan.dtype)).float()
        off2 = o.refine.unet_refine(o.points_to_tensor(rin)).reshape(-1, 6, 3)
        np.savez_compressed(os.path.join(HERE, f"step_{name}_refine.npz"), refine_in_digest=np.array(digest(rin)),
                            refine_stride=np.int64(REFINE_STRIDE), refine_offsets=off2[::REFINE_STRIDE].numpy(),
                            refine_offsets_abs_sum=np.float64(off2.double().abs().sum()))
    path = os.path.join(HERE, f"step_{name}.npz")
    np.savez_compressed(path, **out)
    print(f"wrote {path} ({os.path.getsize(path) / 1e6:.2f} MB); oracle step {t_step:.1f} s; rows {rows.tolist()} pairs {pairs.tolist()}; total {time.time() - t0:.0f} s")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "", sys.argv[2] if len(sys.argv) > 2 else None)

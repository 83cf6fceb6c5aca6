#!/usr/bin/env python
"""Benchmark of the LiDiff denoising hot path (BASELINE.json metric: denoising steps/sec at 180K points,
T=50; scans sharded one per GPU).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference ...                     # CPU restatement of the reference path (oracle port)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/<name>.npy

A "step" is one denoising step of the sampling loop (voxelise + kernel maps, conditional +
unconditional MinkUNetDiff passes, guidance, DPM-Solver++ update, re-quantise) on one 180 000-point
synthetic KITTI-shaped scan with seeded random, BN-calibrated weights.  Under torchrun every rank runs
its own scan (weak scaling, no data-path collective); NCCL is used for the start/stop barriers and the
max-over-ranks time only.  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_POINTS = 180_000
T_STEPS = 50
GUIDANCE_W = 6.0
METRIC = "denoising_steps_per_sec_180k_pts_T50"
UNIT = "steps/s"


def log(msg):
    print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def usable_cpus() -> int:
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:                                    # cgroup v2 CPU quota of the container, if any
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=p["hbm_gbs"], tf=p.get("bf16_tflops_sustained", p["bf16_tflops"]), src="of measured (MEASURED_PEAKS.json, sustained)")
    return dict(hbm_gbs=6650.0, tf=1400.0, src="of fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs"""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()

    def summary(self):
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        reasons = []
        for name, col in (("hw_slowdown", 3), ("hw_thermal_slowdown", 4), ("sw_thermal_slowdown", 5), ("sw_power_cap", 6)):
            if any(len(r) > col and r[col].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons, "samples": len(sm)}


def build_inputs(device, seed):
    """synthetic KITTI-shaped scan -> preprocess_scan (range filter, FPS 18000, x10)  [outside the timed region]"""
    from lidiff_b200.preprocess import farthest_point_sample
    from lidiff_b200.synth import range_filter, synthetic_scan
    raw = torch.tensor(range_filter(synthetic_scan(seed)), device=device)
    sel = farthest_point_sample(raw, N_POINTS // 10)
    scan = raw[sel].repeat(10, 1)                                   # (180000, 3) fp64
    g = torch.Generator(device=device).manual_seed(1234 + seed)
    start = torch.randn(scan.shape, device=device, generator=g)
    return scan, start, g


def build_pipeline(device, scan, T=T_STEPS):
    from lidiff_b200.pipeline import DiffCompletion
    from lidiff_b200.weights import calibrate_bn, random_state_dict
    sds = {"enc": random_state_dict("enc", 0), "diff": random_state_dict("diff", 1), "refine": random_state_dict("refine", 2)}
    pipe = DiffCompletion(state_dicts=sds, denoising_steps=T, cond_weight=GUIDANCE_W, device=device,
                          hparams={"data": {"num_points": N_POINTS}}, engine=True)
    calibrate_bn(pipe, scan[None])                                  # seeded random weights with sane BN statistics
    return pipe


# ---------------------------------------------------------------------------------------------------------------
def sampled_steps(K: int, T: int):
    """the K schedule positions the timed region runs: all T steps in order when K >= T (wrapping), otherwise K positions
    spread evenly over the schedule (first and last included) — a short run costs what the full trajectory costs per step"""
    if K >= T:
        return [i % T for i in range(K)]
    return sorted({int(round(j * (T - 1) / max(K - 1, 1))) for j in range(K)}) if K > 1 else [0]


def csrc_digest():
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "lidiff_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh")):
            h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist
    from lidiff_b200.sharding import max_over_ranks
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    log("building inputs (synthetic scan, GPU farthest point sampling)")
    scan, start, g = build_inputs(device, seed=rank)
    log("building pipeline (seeded weights, BN calibration)")
    pipe = build_pipeline(device, scan, args.T)
    eng = pipe.engine()
    h = eng.h
    K, W, T = args.steps, args.warmup, eng.T
    steps = sampled_steps(K, T)
    K = len(steps)
    noise = torch.randn((T, N_POINTS, 3), device=device, generator=g)
    x_feats = (scan + start).float()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- untimed: the full T-step trajectory once; the loop state in front of every sampled step is kept --------------
    log(f"trajectory pass: {T} steps (untimed), snapshots in front of steps {steps}")
    st = eng.start(scan, x_feats)
    snaps = {}
    for i in range(T):
        if i in steps and i not in snaps:
            snaps[i] = (st["xa"].clone(), st["ca"].clone(), st["x0s"].clone())
        eng.advance(st, noise[i])
    torch.cuda.synchronize()

    bufs = tuple(eng._bufs[k] for k in ("x_a", "x_b", "c_a", "c_b"))       # the loop's ping-pong buffers; step 0 reads x_a / c_a

    def restore(i):
        xa, ca, x0s = snaps[i]
        # schedule position i always runs from the same ping-pong buffer as in the trajectory (captured step graphs are keyed on it)
        st["xa"], st["xb"], st["ca"], st["cb"] = bufs if i % 2 == 0 else (bufs[1], bufs[0], bufs[3], bufs[2])
        st["xa"].copy_(xa); st["ca"].copy_(ca); st["x0s"].copy_(x0s)
        st["i"] = i
        eng._have_x0 = i > 0

    log(f"warm-up {W} steps")
    for j in range(W):
        restore(steps[j % K])
        eng.advance(st, noise[steps[j % K]])
    torch.cuda.synchronize()

    # ---- timed region 1: inputs resident in HBM, no instrumentation -----------------------------------------------------
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    l0 = eng.launches()
    with ClockSampler(local_rank) as clocks:
        if args.profiler_range:
            torch.cuda.profiler.start()                 # `ncu --profile-from-start off` then sees exactly the timed region
        e0.record()
        for i in steps:
            restore(i)
            eng.advance(st, noise[i])
        e1.record()
        barrier()
        if args.profiler_range:
            torch.cuda.profiler.stop()
    launches = eng.launches() - l0
    ms = e0.elapsed_time(e1)
    log(f"timed region: {K} steps in {ms:.1f} ms")
    if h.read_status() & 1:
        raise RuntimeError("a coordinate left the supported key range during the benchmark")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, st, steps[-1])

    # ---- timed region 2: end to end through the public loop with HOST buffers ----------------------------------------------
    h_noise = torch.empty((K, N_POINTS, 3), dtype=torch.float32).pin_memory()      # the SDE noise of the K timed schedule positions
    h_noise.copy_(noise[steps])
    h_out = torch.empty((N_POINTS, 3), dtype=torch.float32).pin_memory()
    h_scan, h_start = scan.cpu().pin_memory(), x_feats.cpu().pin_memory()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    f0.record()
    st = eng.start(h_scan.to(device, non_blocking=True), h_start.to(device, non_blocking=True))
    for n, i in enumerate(steps):
        restore(i)
        eng.advance(st, None, host_noise=h_noise[n], host_out=h_out)
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    log(f"e2e region: {K} steps in {ms_e2e:.1f} ms")
    ms, ms_e2e = max_over_ranks(ms, device), max_over_ranks(ms_e2e, device)

    # ---- instrumented pass (separate from the headline): per-conv CUDA events + pair counts of the same K steps --------------
    eng.pair_hist = torch.zeros((K, 18), dtype=torch.int64, device=device)
    eng._hist_row = 0
    eng.conv_events, eng.layer_log = [], []
    torch.cuda.synchronize()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    for n, i in enumerate(steps):
        restore(i)
        eng.advance(st, noise[i])
        if n == 0:
            layers, eng.layer_log = eng.layer_log, None
    g1.record()
    torch.cuda.synchronize()
    ms_instr = g0.elapsed_time(g1)
    conv_events, eng.conv_events = eng.conv_events, None
    pair_hist, eng.pair_hist = eng.pair_hist.cpu().numpy(), None

    # ---- fixed-geometry micro-benchmark (SURVEY 8d-5): points = scan + sigma*randn, one schedule position each --------------
    fixed = {}
    if rank == 0 and not args.no_fixed:
        gf = torch.Generator(device=device).manual_seed(4321)
        for sigma, i in ((1.0, 0), (0.2, T // 2), (0.05, T - 1)):
            xs = (scan + sigma * torch.randn(scan.shape, device=device, generator=gf, dtype=scan.dtype)).float()
            st = eng.start(scan, xs)
            st["i"] = i
            reps = 3
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            xa0, ca0 = st["xa"].clone(), st["ca"].clone()
            for r in range(reps + 1):                 # first repetition untimed (captures the graph of this position on these buffers)
                if r == 1:
                    a.record()
                st["xa"], st["xb"], st["ca"], st["cb"] = bufs if i % 2 == 0 else (bufs[1], bufs[0], bufs[3], bufs[2])
                st["xa"].copy_(xa0); st["ca"].copy_(ca0); st["i"] = i
                eng._have_x0 = False
                eng.advance(st, noise[i])
            b.record()
            torch.cuda.synchronize()
            fixed[f"sigma_{sigma}"] = {"ms_per_step": round(a.elapsed_time(b) / reps, 3), "level_rows": eng.geom.sizes(),
                                       "pairs_3x3x3": eng.geom.pairs[:5].tolist()}
    # ---- BASELINE configs[4]: whole-scan completion through the public API (host numpy in, host numpy out) --------------------------
    scan_e2e = None
    if not args.no_scan:
        from lidiff_b200.synth import synthetic_scan
        raw = synthetic_scan(100 + rank)                                   # (131072, 3) float64 host array, before the range filter
        pipe.complete_scan(raw)                                            # untimed: graphs of the refinement-free path exist, buffers sized
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t_host = time.time()
        s0.record()
        refined, post = pipe.complete_scan(raw)
        s1.record()
        barrier()
        t_host = time.time() - t_host
        ms_scan = max_over_ranks(max(s0.elapsed_time(s1), 1e3 * t_host), device)
        scan_e2e = {"value": round(world / (ms_scan * 1e-3), 4), "unit": "scans/s", "ms_per_scan": round(ms_scan, 1), "scans_timed": world,
                    "points_in": int(raw.shape[0]), "points_out": int(refined.shape[0]),
                    "what": "DiffCompletion.complete_scan(raw numpy scan) -> refined numpy cloud: range filter (host, as the reference), GPU farthest "
                            "point sampling to 18000 (INSIDE the timed region), x10, T=50 guided denoising steps, postprocess, refinement "
                            "network forward, 6 offsets per point, copy back; wall clock incl. all host work, one scan per GPU"}
    if rank != 0:
        return None

    # ---- rooflines ---------------------------------------------------------------------------------------------------------
    peaks = measured_peaks()
    nconv = len(layers)
    geo = eng.geom
    pair_opt = int(h.get_option(0))                      # LB2_OPT_TC_PAIR: which Cout classes run on the CTA-pair kernel
    cls_of = lambda e: ("ffma" if not e["tc"] else ("cout256" if e["cout"] == 256 else ("cout128" if e["cout"] == 128 else "cout_le96")))
    acc = {c: dict(flops=0.0, bytes_gs=0.0, bytes_min=0.0, ms=0.0, n=0) for c in ("cout256", "cout128", "cout_le96", "ffma")}
    lvl_of_dm = {d.data_ptr(): l for l, d in enumerate(geo.d_n)}
    for n_ev, (a, b, j) in enumerate(conv_events):
        ent = layers[j % nconv]
        step_row = n_ev // nconv
        rows_out = pair_hist[step_row, 13 + lvl_of_dm[ent["d_m"]]]
        if ent["map"] is not None and ent["map"] in geo.map_id:
            slot = geo.map_id[ent["map"]]          # 0-4: 3^3 at level slot; 5-8: stride-2 into level slot-4; 9-12: transposed into level slot-9
            pairs = pair_hist[step_row, slot]
            lvl_in = slot if slot < 5 else (slot - 5 if slot < 9 else slot - 8)
            rows_in = pair_hist[step_row, 13 + lvl_in]
        else:                                   # 1x1 conv on the identity map: pairs = rows of that level
            pairs, rows_in = rows_out, rows_out
        c = acc[cls_of(ent)]
        c["flops"] += 2.0 * pairs * ent["cin"] * ent["cout"] * ent["npass"]
        c["bytes_gs"] += (pairs * (ent["cin"] + ent["cout"]) * 4.0 + pairs * 8.0) * ent["npass"]
        c["bytes_min"] += (rows_in * ent["cin"] * 4.0 + rows_out * ent["cout"] * 4.0 + pairs * 8.0) * ent["npass"]
        c["ms"] += a.elapsed_time(b)
        c["n"] += 1
    conv_ms = sum(c["ms"] for c in acc.values())
    tot = {k: sum(c[k] for c in acc.values()) for k in ("flops", "bytes_gs", "bytes_min", "n")}
    dom = max(acc, key=lambda k: acc[k]["ms"])
    d = acc[dom]
    names = {"cout256": ("k_spconv_tc_pair<256> (CTA-pair cta_group::2 sparse conv" if pair_opt >= 1 else "k_spconv_tc_n256 (sparse conv") + ", Cout 256: levels 3-4 + decoder level 3)",
             "cout128": ("k_spconv_tc_pair<128> (CTA-pair cta_group::2 sparse conv" if pair_opt >= 2 else "k_spconv_tc_small<4> (sparse conv") + ", Cout 128: level-3 encoder, level-2 decoder)",
             "cout_le96": "k_spconv_tc_small<1-3> (sparse conv, Cout 32 / 64 / 96: levels 0-2)", "ffma": "k_spconv_ffma (Cin=3 stem)"}
    traffic = traffic_src = None
    tpath = os.path.join(ROOT, "profiles", "r02_conv_dram_traffic.json")
    if os.path.exists(tpath):                         # ncu dram bytes per launch: only valid for the kernel sources it was captured on
        tj = json.load(open(tpath))
        if tj.get("csrc_digest") == csrc_digest():
            traffic, traffic_src = tj.get("traffic_bytes_per_launch", {}).get(dom), "profiles/r02_conv_dram_traffic.json (ncu --set full, same kernel sources)"
    ach = d["flops"] / max(d["ms"], 1e-9) / 1e9          # FLOP / ms / 1e9 = TFLOP/s
    roofline = {"kernel": names[dom], "bound": "tensor", "achieved": round(ach, 2), "peak": peaks["tf"], "unit": "TFLOP/s",
                "frac": round(ach / peaks["tf"], 4), "traffic": traffic, "traffic_source": traffic_src, "peak_source": peaks["src"],
                "algorithmic_flops_per_launch": d["flops"] / max(d["n"], 1), "avg_launch_ms": round(d["ms"] / max(d["n"], 1), 4), "launches": d["n"],
                "share_of_step": round(d["ms"] / ms_instr, 3),
                "note": "algorithmic FLOPs = 2*pairs*Cin*Cout per pass (SURVEY 8d); the FP16x3 operand split issues 3 MMAs per product, so "
                        "the tensor ceiling for this figure is peak/3; per-launch times from CUDA events around every conv launch in a separate "
                        "instrumented pass over the same steps",
                "all_conv": {"achieved_TFLOPs": round(tot["flops"] / conv_ms / 1e9, 2), "launches": tot["n"], "share_of_step": round(conv_ms / ms_instr, 3),
                             "gather_scatter_model_GBps": round(tot["bytes_gs"] / conv_ms / 1e6, 1),
                             "gather_scatter_frac_of_hbm": round(tot["bytes_gs"] / conv_ms / 1e6 / peaks["hbm_gbs"], 4),
                             "compulsory_GBps": round(tot["bytes_min"] / conv_ms / 1e6, 1), "hbm_peak_GBps": peaks["hbm_gbs"]},
                "by_class": {k: {"ms_per_step": round(c["ms"] / K, 3), "achieved_TFLOPs": round(c["flops"] / max(c["ms"], 1e-9) / 1e9, 2),
                                 "gather_scatter_GBps": round(c["bytes_gs"] / max(c["ms"], 1e-9) / 1e6, 1)} for k, c in acc.items() if c["n"]}}

    out = {"metric": METRIC, "value": round(K * world / (ms * 1e-3), 3), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
           "ms_per_step": round(ms / K, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "fp16x3 split tensor-core MMA, fp32 accumulate (fp32 CUDA cores for the Cin=3 stem), fp64 DPM update",
           "data": "synthetic",
           "config": {"workload": ("BASELINE configs[1]: one synthetic KITTI-shape scan of 180000 points per GPU, T=50 schedule, guidance s=6.0" if args.T == T_STEPS else
                                   f"BASELINE configs[3]: one synthetic KITTI-shape scan of 180000 points per GPU, full schedule set_timesteps({args.T}) = {T} steps, guidance s=6.0"),
                      "points": N_POINTS, "T": T, "guidance_w": GUIDANCE_W, "resolution_m": 0.05,
                      "schedule_positions_timed": steps,
                      "steps_note": "the full T-step trajectory runs once untimed; the timed region replays the listed schedule positions from the saved "
                                    "loop state (3 device copies per step, inside the timed region), so K < T samples the whole trajectory instead of its first K steps",
                      "weights": "seeded random init with reference parameter names, BN statistics calibrated on the scan",
                      "l2": "per-step working set (several GB of feature maps and maps) exceeds the 126 MB L2; no explicit flush",
                      "level_rows_first_last": [pair_hist[0, 13:18].tolist(), pair_hist[-1, 13:18].tolist()]},
           "clocks": clocks.summary(),
           "e2e": {"value": round(K * world / (ms_e2e * 1e-3), 3), "unit": UNIT, "h2d_bytes_per_step": N_POINTS * 3 * 4,
                   "d2h_bytes_per_step": N_POINTS * 3 * 4,
                   "what": "same schedule positions through DenoiseEngine.start/advance with pinned HOST buffers: scan + start uploaded, per-step SDE noise H2D and x_t D2H inside the timed region"},
           "gpu_launches": int(launches), "roofline": roofline, "fixed_geometry": fixed, "scan_e2e": scan_e2e,
           "engine": {"cuda_graphs": bool(eng.use_graphs), "graph_replays": int(eng.graph_replays), "lean_activations": bool(eng.lean),
                      "tc_pair": int(h.get_option(0))}}
    if world == 1 and not args.no_cpu_baseline:
        log("cpu baseline leg")
        out["cpu_baseline"] = cpu_reference(scan.cpu(), pipe, steps=2, warmup=1)
    return out


def dump_outputs(out_dir, st, i):
    """what the last timed step handed its caller, as .npy files: the next noisy points x_t (the loop's output), the DPM-Solver++
    x0 prediction it keeps for the next step and the quantised coordinates of x_t; all 180 000 rows (about 9 MB).  The inputs
    are seeded, but the untimed trajectory in front of a late schedule position compounds the order of atomic accumulations:
    two runs of one build on a B200 agreed to 2e-6 m in the median row, and under 1 % of the rows differed by more than 1 mm."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"x_t": st["xa"].float(), "x0_pred": st["x0s"].double(), "coords": st["ca"].float()}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.cpu().numpy())
    with open(os.path.join(out_dir, "meta.json"), "w") as f:
        json.dump({"schedule_position": int(i), "points": N_POINTS, "arrays": {k: list(v.shape) for k, v in arrays.items()}}, f)
    log(f"outputs of schedule position {i} written to {out_dir}: {', '.join(arrays)}")


# ---------------------------------------------------------------------------------------------------------------
def wedge(scan: torch.Tensor, frac: float) -> torch.Tensor:
    """the points of an azimuthal sector holding `frac` of the scan: same local density as the full scan (a random subsample
    would thin the neighbourhoods and change the cost per point)"""
    az = torch.atan2(scan[:, 1], scan[:, 0])
    cut = torch.quantile(az.double(), min(max(frac, 0.0), 1.0))
    return scan[az.double() <= cut]


CPU_SECTOR = 0.125       # share of the noisy points x_t (an azimuthal sector) one CPU-reference step runs on


def cpu_reference(scan, pipe, steps, warmup):
    """CPU restatement of the reference path (oracle port) on the host cores.  ONE definition for both uses (the cpu_baseline leg and
    --impl reference): a full denoising step (conditional + unconditional pass incl. the conditioning encoder the reference re-runs in
    each pass, nearest-neighbour matching, guidance, DPM update) in which the NOISY points x_t are a 45-degree azimuthal sector of the
    scan (1/8 of the points, same point density) while the conditioning scan x_cond stays complete — so the U-Net work and the
    (queries x keys) nearest-neighbour search shrink by 8 and the encoder work does not.  Full-scan time per step is then
    2 t_enc + 8 (t_step - 2 t_enc) with t_enc timed once; steps/s = 1 / that.  (A sector of x_cond as well would make the brute-force
    matching 64x cheaper and overstate the CPU 3.8x: measured 0.0637 against 0.0167 steps/s on the whole scan, profiles/r02_*.)"""
    from oracle.pipeline import DiffCompletionOracle
    cores = usable_cpus()
    torch.set_num_threads(cores)
    log(f"cpu reference: {cores} threads")
    sd_e = {k: v.detach().cpu() for k, v in pipe.partial_enc.state_dict().items()}
    sd_d = {k: v.detach().cpu() for k, v in pipe.model.state_dict().items()}
    o = DiffCompletionOracle(sd_e, sd_d, None, denoising_steps=T_STEPS, cond_weight=GUIDANCE_W)
    g = torch.Generator().manual_seed(99)
    sub = wedge(scan, CPU_SECTOR)
    n_s = sub.shape[0]
    x_cond = o.points_to_tensor(scan[None])
    o.enc.global_enc(x_cond)                                    # untimed: thread pool, allocator and page faults of a first call
    t0 = time.time()
    o.enc.global_enc(x_cond)
    t_enc = time.time() - t0
    log(f"cpu reference: conditioning encoder on the whole scan {t_enc:.2f} s")

    def one_step(pts):
        x = pts[None] + torch.randn((1,) + tuple(pts.shape), generator=g, dtype=pts.dtype)
        nz = torch.randn((1, 1) + tuple(pts.shape), generator=g)
        t0 = time.time()
        o.completion_loop(pts[None], o.points_to_tensor(x), x_cond, o.points_to_tensor(torch.zeros_like(scan[None])), nz, n_steps=1)
        return time.time() - t0

    total = max(steps + warmup, 1)
    log(f"cpu reference: {total} step(s), x_t = a {n_s}-point sector, x_cond = the whole scan")
    for _ in range(warmup):
        one_step(sub)
    ts = []
    for _ in range(steps):
        ts.append(one_step(sub))
        log(f"cpu reference: step took {ts[-1]:.2f} s")
    t_step = sum(ts) / len(ts)
    t_full = 2.0 * t_enc + (t_step - 2.0 * t_enc) * (N_POINTS / n_s)
    return {"value": round(1.0 / t_full, 5), "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{steps} denoising step(s) after {warmup} untimed of the oracle (fp32 torch-CPU restatement of the ME/KeOps/diffusers path, all host threads): noisy points = a "
                      f"45-degree azimuthal sector ({n_s} of the {N_POINTS} points, same density), conditioning scan complete; {t_step:.2f} s per sampled step, "
                      f"conditioning encoder {t_enc:.2f} s per pass; full-scan estimate 2 t_enc + {N_POINTS / n_s:.1f} (t_step - 2 t_enc) = {t_full:.1f} s per step "
                      f"(measured on the whole scan: 59.7 s per step on 16 cores)"}


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path (oracle port; MinkowskiEngine/pykeops/
    diffusers cannot be installed or compiled here, see DESIGN.md) on the host cores; rank 0 only."""
    if rank != 0:
        return None
    from lidiff_b200 import minkunet as mk  # module definitions only (parameter names/shapes), CPU tensors
    from lidiff_b200.synth import range_filter, synthetic_scan
    from lidiff_b200.weights import random_state_dict
    from oracle.pipeline import farthest_point_sample

    class P:      # minimal stand-in holding the same seeded weights the CUDA arm uses (uncalibrated BN: timing only)
        pass
    p = P()
    p.partial_enc, p.model = mk.MinkGlobalEnc(in_channels=3), mk.MinkUNetDiff(in_channels=3)
    p.partial_enc.load_state_dict(random_state_dict("enc", 0))
    p.model.load_state_dict(random_state_dict("diff", 1))
    raw = range_filter(synthetic_scan(0))
    rng = np.random.default_rng(0)
    sel = np.sort(rng.choice(raw.shape[0], N_POINTS // 10, replace=False))      # FPS is preprocessing, outside the metric
    scan = torch.tensor(raw[sel]).repeat(10, 1)
    cb = cpu_reference(scan, p, steps=max(args.steps, 1), warmup=args.warmup)
    K = max(args.steps, 1)
    return {"metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": world, "steps": K, "warmup": args.warmup,
            "ms_per_step": round(1e3 / max(cb["value"], 1e-12), 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": "BASELINE configs[1]: one synthetic KITTI-shape scan of 180000 points, T=50 schedule, guidance s=6.0",
                       "points": N_POINTS, "T": T_STEPS, "guidance_w": GUIDANCE_W},
            "cpu_baseline": cb, "gpu_launches": 0,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-fixed", action="store_true", help="skip the fixed-geometry sigma micro-benchmark")
    ap.add_argument("--profiler-range", action="store_true", help="cudaProfilerStart/Stop around the timed region (for ncu --profile-from-start off)")
    ap.add_argument("--no-scan", action="store_true", help="skip the whole-scan (configs[4]) measurement")
    ap.add_argument("--T", type=int, default=T_STEPS, help="schedule length (1000 = BASELINE configs[3])")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    # stdout carries exactly ONE line, the result JSON: libraries that print to fd 1 (NCCL's version banner does) are sent to
    # stderr for the whole run, the JSON is written to the saved descriptor at the end
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())

    if args.impl == "reference":
        out = run_reference(args, rank, world)
        if out is not None:
            emit(out)
        return
    if args.warmup < 3:
        args.warmup = 3
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    out = run_ours(args, rank, world, local_rank)
    if out is not None:
        emit(out)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

"""Fused denoising engine: the sampling loop of
/root/reference/lidiff/tools/diff_completion_pipeline.py:148-169 restructured for the B200
(SURVEY.md App. D), every arithmetic step a call into the C-ABI CUDA library, no host
synchronisation inside the loop (row counts stay in device scalars), buffers sized once.

Exact restructurings relative to the operator-by-operator path (results equal up to fp32 summation
order):
  D.1  gate MLPs hoisted to the <= M_part distinct rows and split into step-invariant and
       time-dependent halves; `x*w` is fused into the producing convolution's epilogue;
  D.2  the conditional encoder output is computed once per scan, the unconditional one (a single
       voxel at the origin) once per engine; the 8 unconditional gate rows for all T steps are
       precomputed;
  D.3  both guidance passes run through every convolution in ONE launch (shared maps/weights);
       the stem (identical for both passes) runs once;
  D.4  head + guidance on voxel rows, then one fused per-point kernel: devoxelise, guidance,
       DPM-Solver++(2M) SDE update in fp64, next TensorField features + coordinates;
  D.5  eval-mode BatchNorm folded into a per-channel affine epilogue (+ReLU, + residual add);
  ME.cat is never materialised (second K segment of the consuming convolution).
"""
from __future__ import annotations

import math
import os
from collections import ChainMap

import numpy as np
import torch

from . import _lib
from ._lib import ConvDesc, ConvIO, DpmCoef, ScatterDesc
from .scheduler import DPMSolverMultistepScheduler

GATE_NAMES = ("stage1", "stage2", "stage3", "stage4", "up1", "up2", "up3", "up4")
GATE_LEVEL = (0, 1, 2, 3, 4, 3, 2, 1)
# level -> tau of the dense / residual split of the Cout-256 convolutions (Geometry).  Measured on a B200 (bench.py, 180k points):
# level 3 at tau 0.5 takes the Cout-256 class from 8.95 to 8.44 ms/step; level 4 (fewer sparse offsets per super-tile) is slower split
SPLIT_TAU = {3: 0.5}
BN_EPS = 1e-5


class ConvLayer:
    """conv weight + folded eval-BatchNorm affine (SURVEY.md App. D.5)"""

    def __init__(self, h, sd, pconv, pbn, device):
        W = sd[f"{pconv}.kernel"].detach().to(device=device, dtype=torch.float32)
        if W.dim() == 2:
            W = W[None]
        self.W = W.contiguous()
        self.kvol, self.cin, self.cout = self.W.shape
        self.name = pconv
        if pbn is not None:
            g = lambda k: sd[f"{pbn}.bn.{k}"].detach().to(device=device, dtype=torch.float32)
            scale = g("weight") / torch.sqrt(g("running_var") + BN_EPS)
            self.scale = scale.contiguous()
            self.shift = (g("bias") - g("running_mean") * scale).contiguous()
        else:
            self.scale = self.shift = None
        self.Wp = h.pack_weights(self.W)          # tensor-core image (None when unsupported)
        # gather-GEMM-scatter split of a 3^3 conv: off-centre offsets through lb2_spconv_scatter, centre as a 1x1 conv
        self.Wc = self.Wpc = None
        if self.kvol == 27 and self.Wp is not None and h.scatter_supported(self.cin, 0, self.cout, 27):
            self.Wc = self.W[13:14].contiguous()
            self.Wpc = h.pack_weights(self.Wc)


class Linear:
    def __init__(self, sd, p, device, cols=None):
        w = sd[f"{p}.weight"].detach().to(device=device, dtype=torch.float32)
        self.w = (w if cols is None else w[:, cols[0]:cols[1]]).contiguous()
        self.b = sd[f"{p}.bias"].detach().to(device=device, dtype=torch.float32).contiguous()
        self.n_out, self.n_in = self.w.shape


class Act:
    """One activation of the fused engine: the fp32 tensor `f` (P, cap, C) and / or its fp16 split companion `h` (P, cap, 2C,
    row = [hi | lo]).  Activations that only convolutions consume exist as the companion alone (half the epilogue's store traffic);
    `f` is kept where a non-convolution consumer reads it (gate multiply, head / gate linears, downsample residuals)."""
    __slots__ = ("f", "h", "P", "cap", "C")

    def __init__(self, P, cap, C, f, h):
        self.P, self.cap, self.C, self.f, self.h = P, cap, C, f, h


def _ptr(t, p):
    return None if t is None else t[min(p, t.shape[0] - 1)].data_ptr()


def _net_layers(h, sd, device, decoder: bool):
    L = {}

    def add(pconv, pbn):
        L[pconv] = ConvLayer(h, sd, pconv, pbn, device)

    def res(p):
        add(f"{p}.net.0", f"{p}.net.1")
        add(f"{p}.net.3", f"{p}.net.4")
        if f"{p}.downsample.0.kernel" in sd:
            add(f"{p}.downsample.0", f"{p}.downsample.1")

    add("stem.0", "stem.1")
    add("stem.3", "stem.4")
    for n in range(1, 5):
        add(f"stage{n}.0.net.0", f"stage{n}.0.net.1")
        res(f"stage{n}.1")
        res(f"stage{n}.2")
    if decoder:
        for n in range(1, 5):
            add(f"up{n}.0.net.0", f"up{n}.0.net.1")
            res(f"up{n}.1.0")
            res(f"up{n}.1.1")
    return L


class Geometry:
    """Device-resident coordinate manager of one point set: 5 levels of voxel rows + hash grids, the
    3^3 / 2^3-stride / transposed kernel maps, all at a fixed row capacity, row counts on device."""

    def __init__(self, h, n_cap: int, with_up: bool = True, levels: int = 5, use_pairs: bool = True):
        dev = h.device
        self.h, self.n_cap, self.levels, self.use_pairs = h, n_cap, levels, use_pairs
        i32 = dict(dtype=torch.int32, device=dev)
        self.C = [torch.zeros((n_cap, 4), **i32) for _ in range(levels)]
        self.d_n = [torch.zeros(1, **i32) for _ in range(levels)]
        self.grid = [h.new_grid(n_cap) for _ in range(levels)]
        self.inv = [torch.zeros(n_cap, **i32) for _ in range(levels)]     # [0]: point -> voxel; [l]: fine row -> coarse row
        self.nbr3 = [torch.empty((27, n_cap), **i32) for _ in range(levels)]
        self.nbr_dn = [None] + [torch.empty((8, n_cap), **i32) for _ in range(levels - 1)]
        self.nbr_up = [torch.empty((8, n_cap), **i32) for _ in range(levels - 1)] + [None] if with_up else None
        self.scratch = h.unique_scratch(n_cap)
        self.counts = torch.empty(n_cap, **i32)
        # (in,out) pair counters filled by lb2_kernel_map: [0:5] 3^3 per level, [5:9] stride-2 (out level 1..4),
        # [9:13] transposed (out level 0..3); [13:18] row counts per level (copied from d_n)
        self.pairs = torch.zeros(18, dtype=torch.int64, device=dev)
        self.map_id = {}
        # execution order of the output rows of each map (rows bucketed by neighbour mask, lb2_row_order)
        self.mask_of = {}                                    # map -> its per-row neighbour bit mask (conv kernels skip absent offsets)
        self.ro_scratch = torch.zeros((h.row_order_scratch_bytes(n_cap) + 3) // 4, **i32)
        self.ro_scratch_late = self.to_scratch_late = None      # second scratch set: maps built on a side stream (build(late_stream=...))
        self.perm3 = [torch.zeros(n_cap, **i32) for _ in range(levels)]
        self.perm_dn = [None] + [torch.zeros(n_cap, **i32) for _ in range(levels - 1)]
        self.perm_up = [torch.zeros(n_cap, **i32) for _ in range(levels - 1)] + [None] if with_up else None
        self.perm_of = {}
        # cost order of the 128-row tiles / 256-row super-tiles of every map (static LPT schedule of the persistent conv kernels)
        self.use_tile_order = os.environ.get("LB2_TILE_ORDER", "1") != "0"
        self.map_self = os.environ.get("LB2_MAP_SELF", "1") != "0"
        self.tile_order_of = {}
        self.to_scratch = torch.zeros((n_cap + 127) // 128, **i32)
        # per-offset (in,out) pair lists of the 3^3 maps of the sparse levels (gather-GEMM-scatter form)
        self.morton_levels = set(int(c) for c in os.environ.get("LB2_MORTON_LEVELS", "") if c.isdigit())
        self.pair_levels = min(3, levels)
        self.pair_level_set = set(int(c) for c in os.environ.get("LB2_SCATTER_LEVELS", "") if c.isdigit())
        self.pairs_of = {}
        self.pl_scratch = torch.zeros(64, **i32)
        want = [use_pairs and l in self.pair_level_set for l in range(self.pair_levels)]     # 208 B/row per level: only where asked for
        self.pair_in = [torch.zeros(26 * n_cap, **i32) if w else None for w in want]
        self.pair_out = [torch.zeros(26 * n_cap, **i32) if w else None for w in want]
        self.koff = [torch.zeros(28, **i32) for _ in range(self.pair_levels)]
        self.tile_off = [torch.zeros(28, **i32) for _ in range(self.pair_levels)]
        # dense / residual split of the 3^3 maps of the dense levels for the Cout-256 convolutions (lb2_tile_split): per 256-row
        # super-tile, the offsets that fewer than tau * 256 rows have leave the CTA-pair kernel and run as compacted pair lists
        # through lb2_spconv_scatter.  LB2_SPLIT_TAU="3:0.5,4:0.5" (level:tau, tau = 0 = off) overrides SPLIT_TAU.
        env = os.environ.get("LB2_SPLIT_TAU")
        tau = dict(SPLIT_TAU) if env is None else {int(a): float(b) for a, b in (kv.split(":") for kv in env.split(",") if kv)}
        ok = use_pairs and h.scatter_supported(256, 0, 256, 27)
        self.split_min_rows = {l: math.ceil(t * 256) for l, t in tau.items() if ok and 0 < t and l < levels}
        self.split_of = {}                                   # nbr pointer -> (dense mask, tile orders, pair_in, pair_out, koff, tile_off)
        self.split_bufs = {l: (torch.zeros(n_cap, **i32), torch.zeros(n_cap, **i32),
                               (torch.zeros((n_cap + 127) // 128, **i32), torch.zeros((n_cap + 255) // 256, **i32)),
                               torch.zeros(27 * n_cap, **i32), torch.zeros(27 * n_cap, **i32), torch.zeros(28, **i32), torch.zeros(28, **i32),
                               torch.zeros(64, **i32))      # pair-list counters: one set per level (levels build on different streams)
                           for l in self.split_min_rows}

    def build(self, coords_f: torch.Tensor, n_points: int, after_levels=None, late_stream=None, late_done=None):
        """coords_f (n_points,4) fp32 integer-valued [b,x,y,z] -> all levels and maps (async).  `after_levels()` is called once the
        coordinate levels (C, inv, d_n, grids) are enqueued and before the kernel maps: work that only needs the levels can be
        put on another stream there and overlap with the map construction.
        late_stream / late_done: the maps the network needs first (3^3 of levels 0-1, stride-2 into level 1) are built on the current
        stream, all others on `late_stream` (own scratch buffers), `late_done` recorded behind them: the caller waits for it in front
        of the first layer of stage 2, so ~0.6 ms of map construction hides behind the stem and stage-1 convolutions."""
        h, N = self.h, self.n_cap
        h.unique_build(coords_f, None, None, n_points, 0, self.grid[0], self.C[0], self.inv[0], self.d_n[0], self.scratch)
        for l in range(1, self.levels):
            h.unique_build(None, self.C[l - 1], self.d_n[l - 1], N, 1 << l, self.grid[l], self.C[l], self.inv[l], self.d_n[l], self.scratch)
        if after_levels is not None:
            after_levels()
        self.pairs.zero_()

        def one(grid, l_out, ks, step, nbr, perm, slot, ro_scratch=None, to_scratch=None):
            ro_scratch = self.ro_scratch if ro_scratch is None else ro_scratch
            to_scratch = self.to_scratch if to_scratch is None else to_scratch
            mask = self.mask_of.get(nbr.data_ptr())
            if mask is None:
                mask = self.mask_of[nbr.data_ptr()] = torch.zeros(N, dtype=torch.int32, device=nbr.device)
            if ks == 3 and self.map_self:            # a level onto itself: symmetric pair set, half the hash probes
                h.kernel_map_self(grid, self.C[l_out], self.d_n[l_out], N, step, nbr, N, self.pairs[slot:slot + 1], mask)
            else:
                h.kernel_map(grid, self.C[l_out], self.d_n[l_out], N, ks, step, nbr, N, self.pairs[slot:slot + 1], mask)
            # 3^3 maps of the levels with many neighbours per row: rows of equal mask in Morton order (compact tiles, L2 locality)
            morton = ks == 3 and l_out in self.morton_levels
            h.row_order(mask, self.d_n[l_out], N, ks ** 3, perm, ro_scratch, self.C[l_out] if morton else None, l_out)
            if self.use_tile_order:
                to = self.tile_order_of.get(nbr.data_ptr())
                if to is None:
                    to = self.tile_order_of[nbr.data_ptr()] = (torch.zeros((N + 127) // 128, dtype=torch.int32, device=nbr.device),
                                                               torch.zeros((N + 255) // 256, dtype=torch.int32, device=nbr.device))
                h.tile_order(mask, perm, self.d_n[l_out], N, to[0], to[1], to_scratch)
            self.map_id[nbr.data_ptr()] = slot
            self.perm_of[nbr.data_ptr()] = perm

        def map3(l, **kw):
            one(self.grid[l], l, 3, 1 << l, self.nbr3[l], self.perm3[l], l, **kw)
            if l in self.split_min_rows:
                dense, res, to, p_in, p_out, koff, toff, scratch = self.split_bufs[l]
                mask, perm = self.mask_of[self.nbr3[l].data_ptr()], self.perm3[l]
                h.tile_split(mask, perm, self.d_n[l], N, 27, self.split_min_rows[l], dense, res)
                h.tile_order(dense, perm, self.d_n[l], N, to[0], to[1], kw.get("to_scratch", self.to_scratch))
                h.pair_list(self.nbr3[l], N, self.d_n[l], N, 27, -1, p_in, p_out, koff, toff, scratch, row_mask=res)
                self.split_of[self.nbr3[l].data_ptr()] = (dense, to, p_in, p_out, koff, toff)
            if l < self.pair_levels and self.use_pairs and l in self.pair_level_set:
                h.pair_list(self.nbr3[l], N, self.d_n[l], N, 27, 13, self.pair_in[l], self.pair_out[l], self.koff[l], self.tile_off[l], self.pl_scratch)
                self.pairs_of[self.nbr3[l].data_ptr()] = l

        def map_dn(l, **kw):
            one(self.grid[l - 1], l, 2, 1 << (l - 1), self.nbr_dn[l], self.perm_dn[l], 4 + l, **kw)

        def map_up(l, **kw):
            one(self.grid[l + 1], l, 2, -(1 << l), self.nbr_up[l], self.perm_up[l], 9 + l, **kw)

        split = late_stream is not None and self.levels >= 3 and not (self.use_pairs and self.pair_level_set)
        early3 = (0, 1) if split else tuple(range(self.levels))
        early_dn = (1,) if split else tuple(range(1, self.levels))
        if split:
            if self.ro_scratch_late is None:
                self.ro_scratch_late, self.to_scratch_late = torch.zeros_like(self.ro_scratch), torch.zeros_like(self.to_scratch)
            kw = dict(ro_scratch=self.ro_scratch_late, to_scratch=self.to_scratch_late)
            late_stream.wait_stream(torch.cuda.current_stream())          # levels, grids and the zeroed pair counters
            with torch.cuda.stream(late_stream):
                for l in range(2, self.levels):                           # in the order the network needs them
                    map_dn(l, **kw)
                    map3(l, **kw)
                if self.nbr_up is not None:
                    for l in range(self.levels - 2, -1, -1):
                        map_up(l, **kw)
                late_done.record(late_stream)
        for l in early3:
            if l >= 1 and l in early_dn:
                map_dn(l)
            map3(l)
        for l in early_dn:
            if l not in early3:
                map_dn(l)
        if not split and self.nbr_up is not None:
            for l in range(self.levels - 1):
                map_up(l)

    def voxel_mean(self, feats, n_points, out):
        self.h.voxel_mean(feats, self.inv[0], n_points, feats.shape[1], self.d_n[0], self.n_cap, out, self.counts)

    def sizes(self):
        return [int(d.item()) for d in self.d_n]


class _PairLookup:
    """nbr tensor pointer -> (geometry, level) for maps that have pair lists (the step geometry only)"""

    def __init__(self, geom):
        self.geom = geom

    def get(self, ptr):
        l = self.geom.pairs_of.get(ptr)
        return None if l is None else (self.geom, l)


class DenoiseEngine:
    def __init__(self, sd_enc: dict, sd_diff: dict, *, device="cuda", n_points=180000, denoising_steps=50,
                 cond_weight=6.0, resolution=0.05, t_steps=1000, beta_start=3.5e-5, beta_end=0.007,
                 div_mode=1, conv_algo=_lib.ALGO_AUTO, batch_coord=0.0, sd_refine: dict | None = None, max_range=50.0):
        self.device = torch.device(device)
        self.h = _lib.get_handle(self.device)
        self.N = int(n_points)
        self.w = float(cond_weight)
        self.resolution = float(resolution)
        self.div_mode = int(div_mode)
        self.conv_algo = conv_algo
        h, dev = self.h, self.device
        self.enc = _net_layers(h, sd_enc, dev, decoder=False)
        self.diff = _net_layers(h, sd_diff, dev, decoder=True)
        # refinement network (MinkUNet, minkunet.py:500-619): same stem / stages / ups without gates, head 96 -> 20 -> 18 + tanh
        self.refine = _net_layers(h, sd_refine, dev, decoder=True) if sd_refine is not None else None
        self.refine_head = (Linear(sd_refine, "last.0", dev), Linear(sd_refine, "last.2", dev)) if sd_refine is not None else None
        self.max_range = float(max_range)
        self.sched = DPMSolverMultistepScheduler(num_train_timesteps=t_steps, beta_start=beta_start, beta_end=beta_end,
                                                 beta_schedule="linear", algorithm_type="sde-dpmsolver++", solver_order=2)
        self.sched.set_timesteps(denoising_steps)
        self.T = len(self.sched.timesteps)
        # gate / head MLPs (minkunet.py:165-181 ..., :376-380)
        self.latent = [(Linear(sd_diff, f"latent_{g}.0", dev), Linear(sd_diff, f"latent_{g}.2", dev)) for g in GATE_NAMES]
        self.temp = [(Linear(sd_diff, f"{g}_temp.0", dev), Linear(sd_diff, f"{g}_temp.2", dev)) for g in GATE_NAMES]
        self.lat_p, self.lat_t, self.lat_2 = [], [], []
        for g in GATE_NAMES:
            half = sd_diff[f"latemp_{g}.0.weight"].shape[1] // 2
            pc, tc = ((half, 2 * half), (0, half)) if g == "up1" else ((0, half), (half, 2 * half))   # :461 swaps the cat order
            self.lat_p.append(Linear(sd_diff, f"latemp_{g}.0", dev, cols=pc))
            self.lat_t.append(Linear(sd_diff, f"latemp_{g}.0", dev, cols=tc))
            self.lat_2.append(Linear(sd_diff, f"latemp_{g}.2", dev))
        self.head = (Linear(sd_diff, "last.0", dev), Linear(sd_diff, "last.2", dev))
        self._bufs = {}
        self._graphs = {}
        self.use_row_order = True
        self.use_scatter = True
        self.use_split = True            # fp16 hi/lo companions + cp.async gathers in the tensor-core kernels
        # lean activations: tensors that only convolutions read are kept as the split companion alone (LB2_LEAN=0: fp32 + companion everywhere)
        self.lean = os.environ.get("LB2_LEAN", "1") != "0" and not os.environ.get("LB2_SCATTER_LEVELS")
        self._acts = {}
        self._perm_lookup = {}
        self._tile_order_lookup = {}
        self.geom = Geometry(h, self.N, with_up=True)
        self._perm_lookup = self.geom.perm_of
        self._mask_lookup = self.geom.mask_of
        self._tile_order_lookup = self.geom.tile_order_of
        self._pairs_lookup = _PairLookup(self.geom)
        self.geom_cond = None
        self.part_cap = 0
        self.nn_algo = os.environ.get("LB2_NN_ALGO", "tree")             # "tree" (box hierarchy) or "grid" (lattice shell search): same results
        # NN matches + gate tables on a second stream, concurrent with the kernel-map construction (LB2_SIDE_STREAM=0: all on one stream)
        self.use_side_stream = os.environ.get("LB2_SIDE_STREAM", "1") != "0" and torch.cuda.is_available() and self.device.type == "cuda"
        if self.use_side_stream:
            self._side = torch.cuda.Stream(device=self.device)
            self._side_done = torch.cuda.Event()
            self._side2 = torch.cuda.Stream(device=self.device)       # gate tables (depend on the step index only)
            self._side2_done = torch.cuda.Event()
            self._side3 = torch.cuda.Stream(device=self.device)       # kernel maps of levels 2-4 + all transposed maps
            self._side3_done = torch.cuda.Event()
        self.late_maps = self.use_side_stream and os.environ.get("LB2_LATE_MAPS", "1") != "0"
        # optional instrumentation (bench.py): per-conv CUDA events + layer inventory + pair-count history
        self.conv_events = None          # list of (start, end, layer_index) when enabled
        self.layer_log = None            # list of dict(map, lvl, cin, cout, kvol, npass, tc) recorded during one step
        self.pair_hist = None            # (steps, 18) int64 device tensor when enabled
        self._hist_row = 0
        self._conv_counter = 0
        self._have_x0 = False            # the multistep state (x0_state buffer) holds a prediction of an earlier step
        # CUDA graphs: one graph per (schedule position, ping-pong parity, solver order) captured on first use after an eager
        # warm-up step; all row counts are device scalars and every buffer is persistent, so a graph stays valid across scans
        self.use_graphs = os.environ.get("LB2_GRAPHS", "1") != "0" and torch.cuda.is_available() and self.device.type == "cuda"
        self._graphs = {}
        self._eager_steps = 0
        self.graph_replays = 0
        self.replayed_launches = 0       # kernels launched through graph replays (the library's own counter only sees eager launches)
        self._captured_launches = 0
        self._prepare_time_tables()
        self._prepare_uncond()

    # ------------------------------------------------------------------------------------------------
    @classmethod
    def from_modules(cls, pipe, **kw):
        sd_e = {k: v for k, v in pipe.partial_enc.state_dict().items()}
        sd_d = {k: v for k, v in pipe.model.state_dict().items()}
        hp = pipe.hparams
        if getattr(pipe, "model_refine", None) is not None:
            kw.setdefault("sd_refine", {k: v for k, v in pipe.model_refine.state_dict().items()})
        kw.setdefault("max_range", hp["data"].get("max_range", 50.0))
        return cls(sd_e, sd_d, device=pipe.device, n_points=hp["data"]["num_points"], denoising_steps=hp["diff"]["s_steps"],
                   cond_weight=pipe.w_uncond, resolution=hp["data"]["resolution"], t_steps=hp["diff"]["t_steps"],
                   beta_start=hp["diff"]["beta_start"], beta_end=hp["diff"]["beta_end"], **kw)

    def buf(self, name, shape, dtype=torch.float32):
        t = self._bufs.get(name)
        if t is None or tuple(t.shape) != tuple(shape) or t.dtype != dtype:
            if t is not None:
                self._graphs.clear()                 # a captured step graph may point at the buffer being replaced
            t = torch.zeros(shape, dtype=dtype, device=self.device)
            self._bufs[name] = t
        return t

    # ---- activations (fp32 tensor and / or fp16 split companion), allocated once per name ------------------------------
    def act(self, name, P, cap, C, f32=True, split=True) -> Act:
        split = bool(split and self.use_split and self.conv_algo != _lib.ALGO_FFMA and C % 8 == 0)
        f32 = bool(f32 or not split)
        a = self._acts.get(name)
        if a is None or (a.P, a.cap, a.C) != (P, cap, C) or (a.f is not None) != f32 or (a.h is not None) != split:
            if a is not None:
                self._graphs.clear()                 # a captured step graph may point at the activation being replaced
            f = torch.zeros((P, cap, C), dtype=torch.float32, device=self.device) if f32 else None
            hh = torch.zeros((P, cap, 2 * C), dtype=torch.float16, device=self.device) if split else None
            a = self._acts[name] = Act(P, cap, C, f, hh)
        return a

    # ---- small dense helpers ------------------------------------------------------------------------
    def _linear(self, x, lin: Linear, out, act=0, m_cap=None, d_m=None, prebias=None, pre_act=0, bias=True):
        m_cap = x.shape[0] if m_cap is None else m_cap
        self.h.linear(x, x.stride(0), lin.w, lin.b if bias else None, None, 0, m_cap, d_m, lin.n_in, lin.n_out, act,
                      out, out.stride(0), prebias, pre_act)
        return out

    def _head(self, x, head, out, out_act, d_m):
        """`last` of the U-Nets (minkunet.py:376-380, :585-588) on voxel rows: Linear + LeakyReLU(0.1) + Linear (+ tanh) in one launch
        for all passes; x (npass, cap, n_in), out (npass, cap, n_out)."""
        l0, l1 = head
        self.h.head_mlp(x, x.stride(1), x.stride(0), l0.w, l0.b, l1.w, l1.b, x.shape[1], d_m, l0.n_in, l0.n_out, l1.n_out, out_act,
                        x.shape[0], out, out.stride(1), out.stride(0))

    def _timestep_embedding(self, ts: torch.Tensor) -> torch.Tensor:
        """MinkUNetDiff.get_timestep_embedding (minkunet.py:390-401) for all T steps at once."""
        half = 48
        freq = torch.from_numpy(np.exp(np.arange(0, half) * -(np.log(10000) / (half - 1)))).float().to(self.device)
        arg = ts.to(self.device)[:, None] * freq[None, :]
        return torch.cat([torch.sin(arg), torch.cos(arg)], dim=1).contiguous()

    def _prepare_time_tables(self):
        """bvec[g] (T, hidden_g) = W1t . temp_g(temb(t)) + b1 for every step (time-only half of each gate)."""
        T, dev = self.T, self.device
        temb = self._timestep_embedding(self.sched.timesteps)
        self.bvec = []
        for g in range(8):
            l0, l2 = self.temp[g]
            u = self._linear(temb, l0, torch.empty((T, l0.n_out), device=dev), act=1)
            tv = self._linear(u, l2, torch.empty((T, l2.n_out), device=dev))
            self.bvec.append(self._linear(tv, self.lat_t[g], torch.empty((T, self.lat_t[g].n_out), device=dev)))

    def _gate_tables(self, A_list, rows_cap, d_rows, step, tag):
        """table_g = W2 . leaky(A_g + bvec_g[step]) + b2  -> (rows_cap, C_g) per gate"""
        out = []
        for g in range(8):
            t = self.buf(f"gate_{tag}_{g}", (rows_cap, self.lat_2[g].n_out))
            self._linear(A_list[g], self.lat_2[g], t, m_cap=rows_cap, d_m=d_rows, prebias=self.bvec[g][step], pre_act=1)
            out.append(t)
        return out

    def _part_A(self, part_F, rows_cap, d_rows, tag):
        """A_g = W1p . latent_g(part_F)   (step-invariant half of each gate)"""
        A = []
        for g in range(8):
            l0, l2 = self.latent[g]
            h1 = self._linear(part_F, l0, self.buf(f"lat_h_{tag}", (rows_cap, l0.n_out)), act=1, m_cap=rows_cap, d_m=d_rows)
            p = self._linear(h1, l2, self.buf(f"lat_p_{tag}", (rows_cap, l2.n_out)), m_cap=rows_cap, d_m=d_rows)
            a = self.buf(f"lat_A_{tag}_{g}", (rows_cap, self.lat_p[g].n_out))     # persistent: captured step graphs point at it
            A.append(self._linear(p, self.lat_p[g], a, m_cap=rows_cap, d_m=d_rows, bias=False))
        return A

    # ---- convolution helper ---------------------------------------------------------------------------
    def _conv(self, lay: ConvLayer, nbr, d_m, cap, in1: Act, in2: Act = None, out: Act = None, residual: Act = None, relu=True,
              gate=None, out_gated: Act = None, npass=1):
        """in1 / in2 / residual / out / out_gated: activations with P in {1, npass} passes; gate: list per pass of (table, idx-or-None).
        A residual that exists as a companion only is read as hi + lo by the epilogue."""
        d = ConvDesc()
        d.c1 = in1.C
        d.c2 = in2.C if in2 is not None else 0
        assert d.c1 + d.c2 == lay.cin, (d.c1, d.c2, lay.cin)
        f = lambda a: None if a is None else a.f
        hh = lambda a: None if a is None else a.h
        pre = None
        geom_lvl = self._pairs_lookup.get(nbr.data_ptr()) if (nbr is not None and self.use_scatter and lay.Wpc is not None
                                                               and self.conv_algo != _lib.ALGO_FFMA) else None
        split = None
        if (geom_lvl is None and nbr is not None and lay.cout == 256 and lay.kvol == 27 and lay.Wp is not None
                and self.conv_algo != _lib.ALGO_FFMA):
            split = self.geom.split_of.get(nbr.data_ptr())
        if split is not None:
            # sparse offsets of each super-tile: out_split[pair_out] += in[pair_in] @ W[k], added by the pair kernel's epilogue
            dense, to_dense, p_in, p_out, koff, toff = split
            pre = self.buf(f"split.{lay.cout}", (2, cap, lay.cout))
            sd = ScatterDesc()
            sd.c1, sd.c2, sd.cout, sd.kvol = d.c1, d.c2, lay.cout, 27
            sd.weight_packed = lay.Wp.data_ptr()
            sd.pair_in, sd.pair_out, sd.koff, sd.tile_off = p_in.data_ptr(), p_out.data_ptr(), koff.data_ptr(), toff.data_ptr()
            sd.npass = npass
            for p in range(npass):
                sd.in1[p], sd.in2[p], sd.out[p] = _ptr(f(in1), p), _ptr(f(in2), p), pre[p].data_ptr()
                sd.in1_h[p], sd.in2_h[p] = _ptr(hh(in1), p), _ptr(hh(in2), p)
            sd.d_zero_rows, sd.zero_rows_cap = d_m.data_ptr(), cap
        elif geom_lvl is not None:
            # off-centre pairs: out_scatter[pair_out] += in[pair_in] @ W[k]; the centre runs below as a 1x1 conv with pre_add
            g, l = geom_lvl
            pre = self.buf(f"scatter.{lay.cout}", (2, cap, lay.cout))
            sd = ScatterDesc()
            sd.c1, sd.c2, sd.cout, sd.kvol = d.c1, d.c2, lay.cout, 27
            sd.weight_packed = lay.Wp.data_ptr()
            sd.pair_in, sd.pair_out = g.pair_in[l].data_ptr(), g.pair_out[l].data_ptr()
            sd.koff, sd.tile_off = g.koff[l].data_ptr(), g.tile_off[l].data_ptr()
            sd.npass = npass
            for p in range(npass):
                sd.in1[p], sd.in2[p], sd.out[p] = _ptr(f(in1), p), _ptr(f(in2), p), pre[p].data_ptr()
                sd.in1_h[p], sd.in2_h[p] = _ptr(hh(in1), p), _ptr(hh(in2), p)
            sd.d_zero_rows, sd.zero_rows_cap = d_m.data_ptr(), cap
        else:
            sd = None
        map_ptr = nbr.data_ptr() if nbr is not None else None
        centre = pre is not None and split is None
        d.cout, d.kvol = lay.cout, (1 if centre else lay.kvol)
        d.weight = (lay.Wc if centre else lay.W).data_ptr()
        wp = lay.Wpc if centre else lay.Wp
        d.weight_packed = wp.data_ptr() if wp is not None else None
        d.scale = lay.scale.data_ptr() if lay.scale is not None else None
        d.shift = lay.shift.data_ptr() if lay.shift is not None else None
        d.relu = 1 if relu else 0
        if centre:
            nbr = None                               # centre offset = identity map
        d.nbr = nbr.data_ptr() if nbr is not None else None
        d.nbr_stride = nbr.stride(0) if nbr is not None else cap
        d.d_mout = d_m.data_ptr() if d_m is not None else None
        d.mout_cap, d.npass = cap, npass
        perm = self._perm_lookup.get(nbr.data_ptr()) if (nbr is not None and self.use_row_order) else None
        d.row_perm = perm.data_ptr() if perm is not None else None
        mask = self._mask_lookup.get(nbr.data_ptr()) if nbr is not None else None
        if split is not None:
            mask = split[0]
        d.row_mask = mask.data_ptr() if mask is not None else None
        to = self._tile_order_lookup.get(nbr.data_ptr()) if (nbr is not None and perm is not None) else None
        if split is not None and to is not None:
            to = split[1]
        d.tile_order128 = to[0].data_ptr() if to is not None else None
        d.tile_order256 = to[1].data_ptr() if to is not None else None
        res_h = hh(residual) if (residual is not None and residual.f is None) else None
        for p in range(npass):
            gt = gi = None
            if gate is not None:
                gt = gate[p][0].data_ptr()
                gi = gate[p][1].data_ptr() if gate[p][1] is not None else None
            d.io[p] = ConvIO(_ptr(f(in1), p), _ptr(f(in2), p), _ptr(f(residual), p), _ptr(f(out), p), gt, gi, _ptr(f(out_gated), p),
                             pre[p].data_ptr() if pre is not None else None,
                             _ptr(hh(in1), p), _ptr(hh(in2), p), _ptr(hh(out), p), _ptr(hh(out_gated), p), _ptr(res_h, p))
        if self.layer_log is not None:
            self.layer_log.append(dict(name=lay.name, scatter=sd is not None, map=map_ptr, d_m=d_m.data_ptr() if d_m is not None else None,
                                       cin=lay.cin, cout=lay.cout, kvol=lay.kvol, npass=npass,
                                       tc=bool(lay.Wp is not None and self.conv_algo != _lib.ALGO_FFMA)))
        if self.conv_events is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            if sd is not None:
                self.h.spconv_scatter(sd)
            self.h.spconv(d, self.conv_algo)
            e1.record()
            self.conv_events.append((e0, e1, self._conv_counter))
            self._conv_counter += 1
        else:
            if sd is not None:
                self.h.spconv_scatter(sd)
            self.h.spconv(d, self.conv_algo)

    def _res(self, L, p, geom, lvl, in1: Act, in2: Act, npass, tag, gate=None, want_plain=True, lean=False, out_f32=False):
        """ResidualBlock (minkunet.py:51-80).  lean: the intermediate and the block output exist as split companions only (the
        1x1 downsample branch, read once as a residual, as fp32 only); out_f32 keeps an fp32 copy of the block output."""
        cap = geom.n_cap
        nbr, d_m = geom.nbr3[lvl], geom.d_n[lvl]
        cmid = L[f"{p}.net.0"].cout
        hbuf = self.act(f"{tag}.h", npass, cap, cmid, f32=not lean)
        self._conv(L[f"{p}.net.0"], nbr, d_m, cap, in1, in2, out=hbuf, npass=npass)
        if f"{p}.downsample.0" in L:
            sbuf = self.act(f"{tag}.s", npass, cap, cmid, split=not lean)
            self._conv(L[f"{p}.downsample.0"], None, d_m, cap, in1, in2, out=sbuf, relu=False, npass=npass)
        else:
            assert in2 is None
            sbuf = in1
        out = self.act(f"{tag}.o", npass, cap, cmid, f32=(not lean) or out_f32) if want_plain else None
        og = self.act(f"{tag}.g", npass, cap, cmid, f32=not lean) if gate is not None else None
        self._conv(L[f"{p}.net.3"], nbr, d_m, cap, hbuf, None, out=out, residual=sbuf, relu=True, gate=gate, out_gated=og, npass=npass)
        return out, og

    def _encoder(self, L, geom, F0: Act, npass, tag, gates=None, lean=False, before_gates=None, before_stage2=None):
        """stem + 4 stages.  gates: None (MinkGlobalEnc / refinement net) or per-gate list of per-pass (table, idx)."""
        cap = geom.n_cap
        s0 = self.act(f"{tag}.stem0", 1, cap, 32, f32=not lean)
        self._conv(L["stem.0"], geom.nbr3[0], geom.d_n[0], cap, F0, out=s0, npass=1)
        x0 = self.act(f"{tag}.x0", 1, cap, 32, f32=(not lean) or gates is not None)     # the gate multiply reads fp32
        self._conv(L["stem.3"], geom.nbr3[0], geom.d_n[0], cap, s0, out=x0, npass=1)
        skips = [x0]
        if gates is not None:
            if before_gates is not None:
                before_gates()
            cur = self.act(f"{tag}.x0g", npass, cap, 32, f32=not lean)
            for p in range(npass):
                tb, ix = gates[0][p]
                self.h.gate_mul(x0.f[0], tb, ix, geom.d_n[0], cap, 32, cur.f[p] if cur.f is not None else None,
                                cur.h[p] if cur.h is not None else None)
        else:
            cur = x0
        for n in range(1, 5):
            if n == 2 and before_stage2 is not None:
                before_stage2()
            a = self.act(f"{tag}.s{n}a", npass, cap, L[f"stage{n}.0.net.0"].cout, f32=not lean)
            self._conv(L[f"stage{n}.0.net.0"], geom.nbr_dn[n], geom.d_n[n], cap, cur, out=a, npass=npass)
            b, _ = self._res(L, f"stage{n}.1", geom, n, a, None, npass, f"{tag}.s{n}r1", lean=lean)
            g = gates[n] if gates is not None else None
            x, xg = self._res(L, f"stage{n}.2", geom, n, b, None, npass, f"{tag}.s{n}r2", gate=g, lean=lean)
            skips.append(x)
            cur = xg if gates is not None else x
        return skips, cur

    def _decoder(self, L, geom, skips, cur: Act, npass, tag, gates, lean=False):
        """4 ups; the last block's output keeps its fp32 tensor (the head MLP reads it)"""
        cap = geom.n_cap
        y = cur
        for n in range(1, 5):
            lvl = 4 - n
            d = self.act(f"{tag}.u{n}d", npass, cap, L[f"up{n}.0.net.0"].cout, f32=not lean)
            self._conv(L[f"up{n}.0.net.0"], geom.nbr_up[lvl], geom.d_n[lvl], cap, y, out=d, npass=npass)
            b, _ = self._res(L, f"up{n}.1.0", geom, lvl, d, skips[lvl], npass, f"{tag}.u{n}r1", lean=lean)
            g = gates[4 + n] if (gates is not None and n < 4) else None
            o, og = self._res(L, f"up{n}.1.1", geom, lvl, b, None, npass, f"{tag}.u{n}r2", gate=g, want_plain=(g is None), lean=lean,
                              out_f32=(n == 4))
            y = og if g is not None else o
        return y

    # ---- conditioning ------------------------------------------------------------------------------------
    def _prepare_uncond(self):
        """x_uncond = all-zero points -> one voxel at the origin with zero feature; its encoder output is
        a single 256-vector that depends on the weights only (App. D.2).  Gate rows for all steps."""
        dev = self.device
        g1 = Geometry(self.h, 16, with_up=False, use_pairs=False)
        coords = torch.zeros((16, 4), dtype=torch.float32, device=dev)
        g1.build(coords, 16)
        F0 = self.act("uenc.F0", 1, 16, 3)
        F0.f.zero_()
        skips, _ = self._encoder(self.enc, g1, F0, 1, "uenc")
        part_u = skips[4].f[0][:1].clone()                            # (1,256)
        A = self._part_A(part_u, 1, None, "u")
        self.table_u = []                                             # [g] -> (T, C_g)
        for g in range(8):
            t = torch.empty((self.T, self.lat_2[g].n_out), device=dev)
            for s in range(self.T):
                self._linear(A[g], self.lat_2[g], t[s:s + 1], prebias=self.bvec[g][s], pre_act=1)
            self.table_u.append(t)
        for k in [k for k in self._acts if k.startswith("uenc")]:
            del self._acts[k]

    def set_condition(self, scan: torch.Tensor):
        """scan (N,3): the conditioning point cloud (x_cond).  Runs MinkGlobalEnc once (App. D.2)."""
        dev, N = self.device, scan.shape[0]
        pts = scan.to(device=dev, dtype=torch.float32).contiguous()
        if self.geom_cond is None or self.geom_cond.n_cap != N:
            self._graphs.clear()
            self.geom_cond = Geometry(self.h, N, with_up=False, use_pairs=False)
            self._perm_lookup = ChainMap(self.geom.perm_of, self.geom_cond.perm_of)
            self._mask_lookup = ChainMap(self.geom.mask_of, self.geom_cond.mask_of)
            self._tile_order_lookup = ChainMap(self.geom.tile_order_of, self.geom_cond.tile_order_of)
        coords = self.buf("cond.coords", (N, 4))
        coords[:, 0] = 0
        self.h.quantize(pts, self.resolution, self.div_mode, self.buf("cond.q", (N, 3)))
        coords[:, 1:] = self._bufs["cond.q"]
        g = self.geom_cond
        g.build(coords, N)
        F0 = self.act("cond.F0", 1, N, 3)
        g.voxel_mean(pts, N, F0.f[0])
        skips, _ = self._encoder(self.enc, g, F0, 1, "cenc")
        self.part_F = skips[4].f[0]                                    # (N cap, 256), rows valid < d_n[4]
        self.part_C, self.part_dn, self.part_grid = g.C[4], g.d_n[4], g.grid[4]
        self.part_cap = N
        # box hierarchy over the scan's stride-16 voxels: built once per scan, into the same buffer (captured step graphs point at it)
        self.part_tree = self.h.nn_tree(self.part_C, self.part_dn, N, out=getattr(self, "part_tree", None))
        self.A_cond = self._part_A(self.part_F, N, self.part_dn, "c")

    # ---- one denoising step ----------------------------------------------------------------------------------
    def step(self, i: int, x_t, x_next, coords, coords_next, x_init, noise_i, x0_state, eps_out=None):
        h, N, g = self.h, self.N, self.geom
        self._conv_counter = 0
        nn = [None] * 5
        tabs_box = []

        def gate_tables():
            tabs_box.append(self._gate_tables(self.A_cond, self.part_cap, self.part_dn, i, "c"))

        # the gate tables depend on the step index only: third stream, from the start of the step
        if self.use_side_stream:
            self._side2.wait_stream(torch.cuda.current_stream())      # the previous step's readers of gate_* are enqueued
            with torch.cuda.stream(self._side2):
                gate_tables()
                self._side2_done.record(self._side2)
        else:
            gate_tables()

        def matches():
            # the NN matches need only the coordinate levels: they run on a side stream next to the kernel-map / row-order
            # construction (all of them small latency-bound kernels)
            for l in range(4, -1, -1):               # coarse to fine: a voxel's search starts from its parent voxel's answer
                ix = self.buf(f"nn{l}", (N,), torch.int32)
                # (the shared-memory-table variant lb2_nn_match_table measured slower: 2.1 vs 1.7 ms for the 5 levels)
                if self.nn_algo == "grid":
                    h.nn_match_grid(g.C[l], g.d_n[l], N, self.part_C, self.part_dn, self.part_cap, self.part_grid, 16, 4, ix)
                elif l == 4:
                    h.nn_match_tree(g.C[l], g.d_n[l], N, self.part_tree, self.part_cap, ix)
                else:
                    h.nn_match_tree(g.C[l], g.d_n[l], N, self.part_tree, self.part_cap, ix, self.part_C, g.inv[l + 1], nn[l + 1])
                nn[l] = ix

        def after_levels():
            if not self.use_side_stream:
                return matches()
            main = torch.cuda.current_stream()
            self._side.wait_stream(main)             # the levels are enqueued; the previous step's readers of nn* too
            with torch.cuda.stream(self._side):
                matches()
                self._side_done.record(self._side)

        def join_sides():                            # called by the encoder behind the stem, in front of the first gate multiply
            if self.use_side_stream:
                torch.cuda.current_stream().wait_event(self._side_done)
                torch.cuda.current_stream().wait_event(self._side2_done)

        def join_late_maps():                        # called by the encoder in front of stage 2 (first user of a late map)
            if self.late_maps:
                torch.cuda.current_stream().wait_event(self._side3_done)

        if self.late_maps:
            g.build(coords, N, after_levels, late_stream=self._side3, late_done=self._side3_done)
        else:
            g.build(coords, N, after_levels)
        if self.pair_hist is not None:
            if self.late_maps:
                torch.cuda.current_stream().wait_event(self._side3_done)
            g.pairs[13:18] = torch.cat(g.d_n).long()
            self.pair_hist[self._hist_row % self.pair_hist.shape[0]] = g.pairs
            self._hist_row += 1
        F0 = self.act("F0", 1, N, 3)
        g.voxel_mean(x_t, N, F0.f[0])
        tabs_c = tabs_box[0]
        gates = [[(tabs_c[k], nn[GATE_LEVEL[k]]), (self.table_u[k][i:i + 1], None)] for k in range(8)]
        skips, cur = self._encoder(self.diff, g, F0, 2, "d", gates, lean=self.lean, before_gates=join_sides, before_stage2=join_late_maps)
        y4 = self._decoder(self.diff, g, skips, cur, 2, "d", gates, lean=self.lean)
        eps = self.buf("eps_vox", (2, N, 3))
        self._head(y4.f, self.head, eps, 0, g.d_n[0])
        c = self.sched.coefficients(i)
        # diffusers: second order once one x0 prediction is stored (lower_order_nums >= 1), also at step 0 of a later scan
        second = self._have_x0 and not (i == self.T - 1 and self.T < 15)
        self._have_x0 = True
        cf = DpmCoef(c["c_sample"], c["c_x0"], c["c_noise"], c["sigma_s"], c["alpha_s"], c["inv_r0"] if second else 0.0,
                     self.w, self.resolution, 1 if second else 0, self.div_mode, 1)
        h.guidance_dpm_step(eps[0], eps[1], g.inv[0], x_t, x_init, noise_i, x0_state, N, cf, eps_out, x_next, coords_next)

    # ---- the loop (completion_loop, pipeline:155-169) -----------------------------------------------------------
    def start(self, x_init: torch.Tensor, x_feats: torch.Tensor, fresh: bool = True):
        """condition on the scan and load the noisy start; returns the loop state dict.  fresh=False keeps the multistep
        state (last x0 prediction) of the previous trajectory like the reference's never-reset scheduler does."""
        dev, N = self.device, self.N
        if fresh:
            self._have_x0 = False
        x_src = x_init.reshape(-1, 3)
        assert x_src.shape[0] == N, f"engine built for {N} points, got {x_src.shape[0]}"
        x_init = self.buf("x_init", (N, 3), torch.float64)               # persistent (captured step graphs point at it)
        x_init.copy_(x_src)
        self.set_condition(x_init)
        st = dict(x_init=x_init, xa=self.buf("x_a", (N, 3)), xb=self.buf("x_b", (N, 3)), ca=self.buf("c_a", (N, 4)),
                  cb=self.buf("c_b", (N, 4)), x0s=self.buf("x0_state", (N, 3), torch.float64), i=0)
        st["xa"].copy_(x_feats.reshape(-1, 3).to(device=dev, dtype=torch.float32))
        st["ca"][:, 0] = 0
        self.h.quantize(st["xa"], self.resolution, self.div_mode, self.buf("q0", (N, 3)))
        st["ca"][:, 1:] = self._bufs["q0"]
        return st

    def advance(self, st, noise_i, host_noise=None, host_out=None):
        """one denoising step on the loop state.  host_noise (pinned (N,3) fp32): copied H2D inside the step;
        host_out (pinned (N,3) fp32): the step's x_t is copied D2H (what a caller that visualises / logs every
        step pays).  After one eager step the work of a step is replayed from a CUDA graph (LB2_GRAPHS=0: always eager)."""
        i = st["i"] % self.T
        graphed = self.use_graphs and self.conv_events is None and self.layer_log is None and self.pair_hist is None
        if host_noise is not None or graphed:
            nbuf = self.buf("noise_in", (self.N, 3))
            nbuf.copy_(host_noise if host_noise is not None else noise_i, non_blocking=True)
            noise_i = nbuf
        if not graphed or self._eager_steps < 1:
            self.step(i, st["xa"], st["xb"], st["ca"], st["cb"], st["x_init"], noise_i, st["x0s"])
            self._eager_steps += 1
        else:
            second = self._have_x0 and not (i == self.T - 1 and self.T < 15)
            key = (i, st["xa"].data_ptr(), bool(second))
            ent = self._graphs.get(key)
            if ent is None:
                have = self._have_x0
                l0 = self.h.launch_count()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self.step(i, st["xa"], st["xb"], st["ca"], st["cb"], st["x_init"], noise_i, st["x0s"])
                ent = self._graphs[key] = (g, self.h.launch_count() - l0)
                self._captured_launches += ent[1]                      # counted by the library although capture executes nothing
                self._have_x0 = have                                   # capture does not execute: the replay below is this step
            ent[0].replay()
            self._have_x0 = True
            self.graph_replays += 1
            self.replayed_launches += ent[1]
        st["xa"], st["xb"], st["ca"], st["cb"] = st["xb"], st["xa"], st["cb"], st["ca"]
        st["i"] += 1
        if host_out is not None:
            host_out.copy_(st["xa"], non_blocking=True)

    def launches(self) -> int:
        """kernels launched on behalf of this engine's handle: eager launches counted by the library + graph-replayed ones"""
        return self.h.launch_count() - self._captured_launches + self.replayed_launches

    def run(self, x_init: torch.Tensor, x_feats: torch.Tensor, step_noise=None, n_steps=None, return_device=False, fresh=True):
        """x_init (1,N,3) fp64 conditioning scan, x_feats (1,N,3) noisy start.  Returns final x_t.F (N,3)."""
        dev, N = self.device, self.N
        st = self.start(x_init, x_feats, fresh=fresh)
        T = self.T if n_steps is None else n_steps
        if step_noise is not None:
            step_noise = step_noise.reshape(-1, N, 3).to(device=dev, dtype=torch.float32).contiguous()
        for i in range(T):
            # without injected noise: one fp32 draw per step, in the order diffusers' step() draws it (the operator path and the
            # reference consume the torch RNG stream identically); no (T, N, 3) tensor is materialised (2.2 GB at T = 1000)
            nz = step_noise[i] if step_noise is not None else torch.randn((1, N, 3), device=dev, dtype=torch.float32)[0]
            self.advance(st, nz)
        if return_device:
            return st["xa"]
        out = st["xa"].cpu().numpy()
        if self.h.read_status() & 1:
            raise RuntimeError("lidiff_b200: a coordinate left the supported key range during sampling")
        return out

    # ---- after the loop: postprocess_scan + refinement forward + 6x offsets (pipeline:107-138) ------------------------------
    def postprocess(self, completed: torch.Tensor, x_init: torch.Tensor) -> torch.Tensor:
        """postprocess_scan (pipeline:107-115) on the device: range filter and the z band of the input scan.  completed (N,3) fp32,
        x_init (N,3) fp64.  Same arithmetic as the reference's numpy expressions (fp32 squared norm summed left to right)."""
        x, y, z = completed[:, 0], completed[:, 1], completed[:, 2]
        dist = torch.sqrt((x * x + y * y) + z * z)
        zi = x_init.reshape(-1, 3)[:, 2]
        max_z = zi.max().item()
        min_z = (zi.mean() - 2 * zi.std()).item()
        keep = (dist < self.max_range) & (z < max_z) & (z > min_z)
        return completed[keep].contiguous()

    def refine_offsets(self, pts: torch.Tensor) -> torch.Tensor:
        """refine_forward (pipeline:134-138, MinkUNet.forward minkunet.py:596-619) on `pts` (n,3) fp32 device points, n <= N:
        voxelise, stem + 4 stages + 4 ups through the fused conv kernels (one pass), head on voxel rows, slice back to the points.
        Returns (n,18) fp32 offsets on the device."""
        if self.refine is None:
            raise RuntimeError("DenoiseEngine was built without the refinement network (sd_refine)")
        h, g, N = self.h, self.geom, self.N
        pts = pts.to(device=self.device, dtype=torch.float32).contiguous()
        n = pts.shape[0]
        if n > N:
            raise RuntimeError(f"refine_offsets: {n} points exceed the engine capacity {N}")
        if n == 0:
            return torch.zeros((0, 18), device=self.device)
        coords = self.buf("r.coords", (N, 4))
        q = self.buf("r.q", (N, 3))
        h.quantize(pts, self.resolution, self.div_mode, q[:n])
        coords[:n, 0] = 0
        coords[:n, 1:] = q[:n]
        g.build(coords, n)
        F0 = self.act("r.F0", 1, N, 3)
        g.voxel_mean(pts, n, F0.f[0])
        skips, cur = self._encoder(self.refine, g, F0, 1, "r", lean=self.lean)
        y4 = self._decoder(self.refine, g, skips, cur, 1, "r", None, lean=self.lean)
        off_v = self.buf("r.off_v", (1, N, 18))
        self._head(y4.f, self.refine_head, off_v, 2, g.d_n[0])
        off_v = off_v[0]
        out = torch.empty((n, 18), device=self.device)
        h.gather_rows(off_v, g.inv[0], n, 18, out)
        return out

    def complete(self, x_init: torch.Tensor, x_feats: torch.Tensor, step_noise=None, fresh=True):
        """complete_scan after preprocessing (pipeline:117-132), all on the device: T denoising steps, postprocess, refinement
        forward, 6 offsets per point.  Returns (refined (6n,3), post (n,3)) device tensors."""
        x_t = self.run(x_init, x_feats, step_noise, return_device=True, fresh=fresh)
        post = self.postprocess(x_t, x_init.reshape(-1, 3).to(self.device))
        off = self.refine_offsets(post).reshape(-1, 6, 3)
        refined = (post[:, None, :] + off).reshape(-1, 3)
        if self.h.read_status() & 1:
            raise RuntimeError("lidiff_b200: a coordinate left the supported key range during sampling")
        return refined, post

"""ctypes binding of include/lidiff_b200.h (the C-ABI CUDA library, sm_100a).

There is deliberately NO CPU fallback: importing works anywhere (so host logic can be tested), but
`get_lib()` raises if the shared object is missing and `Lib.handle(device)` raises if no B200 is
visible.  torch is used only for device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import torch

_SO = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_C", "liblidiff_b200.so")

ALGO_AUTO, ALGO_FFMA, ALGO_TC, ALGO_TC_TILE = 0, 1, 2, 3
OPT_TC_PAIR, OPT_TC_N256, OPT_TC_SMALL, OPT_TC_PERSISTENT, OPT_TC_FULL_LAG, OPT_TC_NSPLIT = range(6)


class Grid(C.Structure):
    _fields_ = [("keys", C.c_void_p), ("vals", C.c_void_p), ("cap_table", C.c_int32)]


class ConvIO(C.Structure):
    _fields_ = [("in1", C.c_void_p), ("in2", C.c_void_p), ("residual", C.c_void_p), ("out", C.c_void_p),
                ("gate_table", C.c_void_p), ("gate_idx", C.c_void_p), ("out_gated", C.c_void_p), ("pre_add", C.c_void_p),
                ("in1_h", C.c_void_p), ("in2_h", C.c_void_p), ("out_h", C.c_void_p), ("out_gated_h", C.c_void_p),
                ("residual_h", C.c_void_p)]


class ConvDesc(C.Structure):
    _fields_ = [("c1", C.c_int32), ("c2", C.c_int32), ("cout", C.c_int32), ("kvol", C.c_int32),
                ("weight", C.c_void_p), ("weight_packed", C.c_void_p),
                ("scale", C.c_void_p), ("shift", C.c_void_p), ("relu", C.c_int32),
                ("nbr", C.c_void_p), ("nbr_stride", C.c_int64),
                ("d_mout", C.c_void_p), ("mout_cap", C.c_int32), ("row_perm", C.c_void_p), ("row_mask", C.c_void_p),
                ("npass", C.c_int32),
                ("io", ConvIO * 2),
                ("tile_order128", C.c_void_p), ("tile_order256", C.c_void_p)]


class ScatterDesc(C.Structure):
    _fields_ = [("c1", C.c_int32), ("c2", C.c_int32), ("cout", C.c_int32), ("kvol", C.c_int32),
                ("weight_packed", C.c_void_p), ("pair_in", C.c_void_p), ("pair_out", C.c_void_p),
                ("koff", C.c_void_p), ("tile_off", C.c_void_p), ("npass", C.c_int32),
                ("in1", C.c_void_p * 2), ("in2", C.c_void_p * 2), ("in1_h", C.c_void_p * 2), ("in2_h", C.c_void_p * 2),
                ("out", C.c_void_p * 2),
                ("d_zero_rows", C.c_void_p), ("zero_rows_cap", C.c_int32)]


class VoxelHistResult(C.Structure):
    _fields_ = [("n_a", C.c_int64), ("n_b", C.c_int64), ("occ_a", C.c_int64), ("occ_b", C.c_int64), ("occ_ab", C.c_int64),
                ("jsd_3d", C.c_double), ("jsd_bev", C.c_double)]


class DpmCoef(C.Structure):
    _fields_ = [("c_sample", C.c_double), ("c_x0", C.c_double), ("c_noise", C.c_double),
                ("sigma_s", C.c_double), ("alpha_s", C.c_double), ("inv_r0", C.c_double),
                ("guidance_w", C.c_float), ("resolution", C.c_float),
                ("second_order", C.c_int32), ("div_mode", C.c_int32), ("f64_state", C.c_int32)]


EXPORTS = [
    "lb2_create", "lb2_destroy", "lb2_last_error", "lb2_version", "lb2_launch_count", "lb2_read_status",
    "lb2_set_option", "lb2_get_option", "lb2_tile_order", "lb2_tile_split",
    "lb2_quantize", "lb2_unique_scratch_bytes", "lb2_unique_build", "lb2_voxel_mean", "lb2_kernel_map",
    "lb2_spconv_forward", "lb2_packed_weight_bytes", "lb2_pack_weights", "lb2_nn_match", "lb2_linear",
    "lb2_gate_mul", "lb2_gather_rows", "lb2_head_mlp", "lb2_kernel_map_self", "lb2_guidance_dpm_step", "lb2_farthest_point_sample",
    "lb2_row_order", "lb2_row_order_scratch_bytes", "lb2_nn_match_grid",
    "lb2_nn_table_bytes", "lb2_nn_table_build", "lb2_nn_match_table",
    "lb2_nn_tree_bytes", "lb2_nn_tree_build", "lb2_nn_match_tree",
    "lb2_pair_list", "lb2_pair_list_scratch_bytes", "lb2_spconv_scatter", "lb2_spconv_scatter_supported",
    "lb2_cloud_nn_scratch_bytes", "lb2_cloud_nn_distance", "lb2_voxel_hist_scratch_bytes", "lb2_voxel_hist_compare",
    "lb2_threshold_counts",
]


def _ptr(t):
    if t is None:
        return None
    if isinstance(t, int):
        return t
    return t.data_ptr()


class Lib:
    """Loaded shared object + one handle per device."""

    def __init__(self, path: str = _SO):
        if not os.path.exists(path):
            raise RuntimeError(f"lidiff_b200: CUDA library not built ({path}); run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "or lidiff_b200/csrc/build.sh — there is no CPU fallback")
        self.path = path
        self.dll = C.CDLL(path)
        d = self.dll
        d.lb2_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        d.lb2_destroy.argtypes = [C.c_void_p]
        d.lb2_destroy.restype = None
        d.lb2_last_error.argtypes = [C.c_void_p]
        d.lb2_last_error.restype = C.c_char_p
        d.lb2_launch_count.argtypes = [C.c_void_p]
        d.lb2_launch_count.restype = C.c_int64
        d.lb2_read_status.argtypes = [C.c_void_p, C.c_void_p]
        d.lb2_set_option.argtypes = [C.c_void_p, C.c_int, C.c_int]
        d.lb2_get_option.argtypes = [C.c_void_p, C.c_int]
        d.lb2_unique_scratch_bytes.argtypes = [C.c_int64]
        d.lb2_unique_scratch_bytes.restype = C.c_size_t
        d.lb2_packed_weight_bytes.argtypes = [C.c_int32] * 3
        d.lb2_packed_weight_bytes.restype = C.c_size_t
        vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float
        d.lb2_quantize.argtypes = [vp, vp, vp, i64, f32, C.c_int, vp]
        d.lb2_unique_build.argtypes = [vp, vp, vp, vp, vp, i32, i32, Grid, vp, vp, vp, vp]
        d.lb2_voxel_mean.argtypes = [vp, vp, vp, vp, i32, i32, vp, i32, vp, vp]
        d.lb2_kernel_map.argtypes = [vp, vp, Grid, vp, vp, i32, i32, i32, vp, i64, vp, vp]
        d.lb2_kernel_map_self.argtypes = [vp, vp, Grid, vp, vp, i32, i32, vp, i64, vp, vp]
        d.lb2_row_order.argtypes = [vp, vp, vp, vp, i32, i32, vp, vp, vp, i32]
        d.lb2_tile_order.argtypes = [vp, vp, vp, vp, vp, i32, vp, vp, vp]
        d.lb2_tile_split.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, vp, vp]
        d.lb2_row_order_scratch_bytes.restype = C.c_size_t
        d.lb2_row_order_scratch_bytes.argtypes = [i32]
        d.lb2_spconv_forward.argtypes = [vp, vp, C.POINTER(ConvDesc), C.c_int]
        d.lb2_pack_weights.argtypes = [vp, vp, vp, i32, i32, i32, vp]
        d.lb2_nn_match.argtypes = [vp, vp, vp, vp, i32, vp, vp, i32, i32, vp]
        d.lb2_pair_list.argtypes = [vp, vp, vp, i64, vp, i32, i32, i32, vp, vp, vp, vp, vp, vp]
        d.lb2_pair_list_scratch_bytes.restype = C.c_size_t
        d.lb2_spconv_scatter.argtypes = [vp, vp, C.POINTER(ScatterDesc)]
        d.lb2_spconv_scatter_supported.argtypes = [i32, i32, i32, i32]
        d.lb2_nn_table_bytes.restype = C.c_size_t
        d.lb2_nn_tree_bytes.restype = C.c_size_t
        d.lb2_nn_tree_bytes.argtypes = [i32]
        d.lb2_nn_tree_build.argtypes = [vp, vp, vp, vp, i32, vp]
        d.lb2_nn_match_tree.argtypes = [vp, vp, vp, vp, i32, vp, i32, vp, vp, vp, vp]
        d.lb2_nn_table_build.argtypes = [vp, vp, vp, vp, i32, vp]
        d.lb2_nn_match_table.argtypes = [vp, vp, vp, vp, i32, vp, vp, i32, vp, i32, i32, vp]
        d.lb2_nn_match_grid.argtypes = [vp, vp, vp, vp, i32, vp, vp, i32, Grid, i32, i32, vp]
        d.lb2_linear.argtypes = [vp, vp, vp, i64, vp, vp, vp, i64, i32, vp, i32, i32, i32, vp, i64,
                                 vp, i32]
        d.lb2_gate_mul.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, vp, vp]
        d.lb2_gather_rows.argtypes = [vp, vp, vp, vp, i32, i32, vp]
        d.lb2_head_mlp.argtypes = [vp, vp, vp, i64, i64, vp, vp, vp, vp, i32, vp, i32, i32, i32, i32, i32, vp, i64, i64]
        d.lb2_guidance_dpm_step.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, DpmCoef, vp, vp, vp, vp]
        d.lb2_farthest_point_sample.argtypes = [vp, vp, vp, i32, i32, vp, vp]
        d.lb2_cloud_nn_scratch_bytes.argtypes = [i64, i64]
        d.lb2_cloud_nn_scratch_bytes.restype = C.c_size_t
        d.lb2_cloud_nn_distance.argtypes = [vp, vp, vp, i64, vp, i64, vp, vp]
        d.lb2_voxel_hist_scratch_bytes.argtypes = [i64, i64]
        d.lb2_voxel_hist_scratch_bytes.restype = C.c_size_t
        d.lb2_voxel_hist_compare.argtypes = [vp, vp, vp, i64, vp, i64, vp, i32, vp, vp]
        d.lb2_threshold_counts.argtypes = [vp, vp, vp, i64, vp, i32, vp]
        self._handles = {}
        self._lock = threading.Lock()

    def missing_symbols(self):
        return [s for s in EXPORTS if not hasattr(self.dll, s)]

    def handle(self, device) -> "Handle":
        dev = torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError("lidiff_b200 runs on CUDA (B200, sm_100a) only; no CPU fallback")
        idx = dev.index if dev.index is not None else torch.cuda.current_device()
        with self._lock:
            if idx not in self._handles:
                hp = C.c_void_p()
                rc = self.dll.lb2_create(idx, C.byref(hp))
                if rc != 0:
                    raise RuntimeError(f"lb2_create(device={idx}) failed with {rc} (needs an sm_100 GPU)")
                self._handles[idx] = Handle(self, hp, idx)
            return self._handles[idx]


class Handle:
    def __init__(self, lib: Lib, hp, device_index: int):
        self.lib, self.dll, self.hp, self.device_index = lib, lib.dll, hp, device_index
        self.device = torch.device("cuda", device_index)

    # -- plumbing ----------------------------------------------------------------------------------
    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _check(self, rc, what):
        if rc != 0:
            msg = self.dll.lb2_last_error(self.hp)
            raise RuntimeError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")

    def launch_count(self) -> int:
        return int(self.dll.lb2_launch_count(self.hp))

    def read_status(self) -> int:
        return int(self.dll.lb2_read_status(self.hp, self._stream()))

    def set_option(self, option: int, value: int):
        self._check(self.dll.lb2_set_option(self.hp, int(option), int(value)), "set_option")

    def get_option(self, option: int) -> int:
        return int(self.dll.lb2_get_option(self.hp, int(option)))

    # -- coordinate manager ------------------------------------------------------------------------
    def new_grid(self, n_cap: int):
        cap = 1 << max(4, (2 * n_cap - 1).bit_length())
        keys = torch.empty(cap, dtype=torch.int64, device=self.device)
        vals = torch.empty(2 * cap, dtype=torch.int32, device=self.device)
        return (keys, vals, cap)

    @staticmethod
    def _grid(g):
        return Grid(g[0].data_ptr(), g[1].data_ptr(), g[2])

    def unique_scratch(self, n_cap: int) -> torch.Tensor:
        nbytes = int(self.dll.lb2_unique_scratch_bytes(n_cap))
        return torch.empty(nbytes, dtype=torch.uint8, device=self.device)

    def quantize(self, x, resolution, div_mode, out):
        self._check(self.dll.lb2_quantize(self.hp, self._stream(), _ptr(x), x.numel(), float(resolution), int(div_mode), _ptr(out)), "lb2_quantize")

    def unique_build(self, in_f, in_i, d_nin, n_cap, ts_floor, grid, out_coords, inverse, d_nout, scratch):
        self._check(self.dll.lb2_unique_build(self.hp, self._stream(), _ptr(in_f), _ptr(in_i), _ptr(d_nin), int(n_cap), int(ts_floor),
                                              self._grid(grid), _ptr(out_coords), _ptr(inverse), _ptr(d_nout), _ptr(scratch)), "lb2_unique_build")

    def voxel_mean(self, feats, inverse, n, c, d_m, m_cap, out, counts):
        self._check(self.dll.lb2_voxel_mean(self.hp, self._stream(), _ptr(feats), _ptr(inverse), int(n), int(c), _ptr(d_m), int(m_cap),
                                            _ptr(out), _ptr(counts)), "lb2_voxel_mean")

    def kernel_map(self, grid_in, out_coords, d_nout, nout_cap, ks, step, nbr, nbr_stride, pair_count=None, row_mask=None):
        self._check(self.dll.lb2_kernel_map(self.hp, self._stream(), self._grid(grid_in), _ptr(out_coords), _ptr(d_nout), int(nout_cap),
                                            int(ks), int(step), _ptr(nbr), int(nbr_stride), _ptr(pair_count), _ptr(row_mask)), "lb2_kernel_map")

    def kernel_map_self(self, grid, coords, d_n, n_cap, step, nbr, nbr_stride, pair_count=None, row_mask=None):
        self._check(self.dll.lb2_kernel_map_self(self.hp, self._stream(), self._grid(grid), _ptr(coords), _ptr(d_n), int(n_cap), int(step),
                                                 _ptr(nbr), int(nbr_stride), _ptr(pair_count), _ptr(row_mask)), "lb2_kernel_map_self")

    def row_order_scratch_bytes(self, n_cap) -> int:
        return int(self.dll.lb2_row_order_scratch_bytes(int(n_cap)))

    def row_order(self, row_mask, d_n, n_cap, kvol, perm, scratch, coords=None, coord_shift=0):
        self._check(self.dll.lb2_row_order(self.hp, self._stream(), _ptr(row_mask), _ptr(d_n), int(n_cap), int(kvol), _ptr(perm), _ptr(scratch),
                                           _ptr(coords), int(coord_shift)), "lb2_row_order")

    def tile_order(self, row_mask, row_perm, d_n, n_cap, order128, order256, scratch):
        self._check(self.dll.lb2_tile_order(self.hp, self._stream(), _ptr(row_mask), _ptr(row_perm), _ptr(d_n), int(n_cap), _ptr(order128),
                                            _ptr(order256), _ptr(scratch)), "lb2_tile_order")

    def tile_split(self, row_mask, row_perm, d_n, n_cap, kvol, min_rows, dense_mask, res_mask):
        self._check(self.dll.lb2_tile_split(self.hp, self._stream(), _ptr(row_mask), _ptr(row_perm), _ptr(d_n), int(n_cap), int(kvol), int(min_rows),
                                            _ptr(dense_mask), _ptr(res_mask)), "lb2_tile_split")

    # -- conv ----------------------------------------------------------------------------------------
    def spconv(self, desc: ConvDesc, algo: int = ALGO_AUTO):
        self._check(self.dll.lb2_spconv_forward(self.hp, self._stream(), C.byref(desc), int(algo)), "lb2_spconv_forward")

    def pair_list(self, nbr, nbr_stride, d_nout, nout_cap, kvol, skip_k, pair_in, pair_out, koff, tile_off, scratch, row_mask=None):
        self._check(self.dll.lb2_pair_list(self.hp, self._stream(), _ptr(nbr), int(nbr_stride), _ptr(d_nout), int(nout_cap), int(kvol), int(skip_k),
                                           _ptr(pair_in), _ptr(pair_out), _ptr(koff), _ptr(tile_off), _ptr(scratch), _ptr(row_mask)), "lb2_pair_list")

    def scatter_supported(self, c1, c2, cout, kvol) -> bool:
        return bool(self.dll.lb2_spconv_scatter_supported(int(c1), int(c2), int(cout), int(kvol)))

    def spconv_scatter(self, desc: "ScatterDesc"):
        self._check(self.dll.lb2_spconv_scatter(self.hp, self._stream(), C.byref(desc)), "lb2_spconv_scatter")

    def packed_weight_bytes(self, kvol, cin, cout) -> int:
        return int(self.dll.lb2_packed_weight_bytes(kvol, cin, cout))

    def pack_weights(self, w: torch.Tensor):
        kvol, cin, cout = w.shape
        nbytes = self.packed_weight_bytes(kvol, cin, cout)
        if nbytes == 0:
            return None
        out = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        self._check(self.dll.lb2_pack_weights(self.hp, self._stream(), _ptr(w), kvol, cin, cout, _ptr(out)), "lb2_pack_weights")
        return out

    # -- misc ----------------------------------------------------------------------------------------
    def nn_match(self, q, d_nq, nq_cap, k, d_nk, nk_cap, batch_scale, idx):
        self._check(self.dll.lb2_nn_match(self.hp, self._stream(), _ptr(q), _ptr(d_nq), int(nq_cap), _ptr(k), _ptr(d_nk), int(nk_cap),
                                          int(batch_scale), _ptr(idx)), "lb2_nn_match")

    def nn_match_grid(self, q, d_nq, nq_cap, k, d_nk, nk_cap, key_grid, key_stride, max_ring, idx):
        self._check(self.dll.lb2_nn_match_grid(self.hp, self._stream(), _ptr(q), _ptr(d_nq), int(nq_cap), _ptr(k), _ptr(d_nk), int(nk_cap),
                                               self._grid(key_grid), int(key_stride), int(max_ring), _ptr(idx)), "lb2_nn_match_grid")

    def nn_table(self, k, d_nk, nk_cap):
        """compact hash table of the key voxels for nn_match_table (one per conditioning scan)"""
        t = torch.empty(int(self.dll.lb2_nn_table_bytes()), dtype=torch.uint8, device=self.device)
        self._check(self.dll.lb2_nn_table_build(self.hp, self._stream(), _ptr(k), _ptr(d_nk), int(nk_cap), _ptr(t)), "lb2_nn_table_build")
        return t

    def nn_tree(self, k, d_nk, nk_cap, out=None):
        """bounding-box hierarchy over the key voxels for nn_match_tree (one per conditioning scan); `out` re-uses a buffer"""
        nbytes = int(self.dll.lb2_nn_tree_bytes(int(nk_cap)))
        t = out if (out is not None and out.numel() == nbytes) else torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        self._check(self.dll.lb2_nn_tree_build(self.hp, self._stream(), _ptr(k), _ptr(d_nk), int(nk_cap), _ptr(t)), "lb2_nn_tree_build")
        return t

    def nn_match_tree(self, q, d_nq, nq_cap, tree, nk_cap, idx, k=None, hint_of=None, hint_idx=None):
        self._check(self.dll.lb2_nn_match_tree(self.hp, self._stream(), _ptr(q), _ptr(d_nq), int(nq_cap), _ptr(tree), int(nk_cap),
                                               _ptr(k), _ptr(hint_of), _ptr(hint_idx), _ptr(idx)), "lb2_nn_match_tree")

    def nn_match_table(self, q, d_nq, nq_cap, k, d_nk, nk_cap, table, key_stride, max_ring, idx):
        self._check(self.dll.lb2_nn_match_table(self.hp, self._stream(), _ptr(q), _ptr(d_nq), int(nq_cap), _ptr(k), _ptr(d_nk), int(nk_cap),
                                                _ptr(table), int(key_stride), int(max_ring), _ptr(idx)), "lb2_nn_match_table")

    def linear(self, x, ldx, w, b, addend, ld_add, m_cap, d_m, n_in, n_out, act, y, ldy, prebias=None, pre_act=0):
        self._check(self.dll.lb2_linear(self.hp, self._stream(), _ptr(x), int(ldx), _ptr(w), _ptr(b), _ptr(addend), int(ld_add), int(m_cap),
                                        _ptr(d_m), int(n_in), int(n_out), int(act), _ptr(y), int(ldy), _ptr(prebias), int(pre_act)), "lb2_linear")

    def head_mlp(self, x, ldx, x_pass_stride, w0, b0, w1, b1, m_cap, d_m, n_in, n_hid, n_out, out_act, npass, y, ldy, y_pass_stride):
        self._check(self.dll.lb2_head_mlp(self.hp, self._stream(), _ptr(x), int(ldx), int(x_pass_stride), _ptr(w0), _ptr(b0), _ptr(w1), _ptr(b1),
                                          int(m_cap), _ptr(d_m), int(n_in), int(n_hid), int(n_out), int(out_act), int(npass), _ptr(y), int(ldy),
                                          int(y_pass_stride)), "lb2_head_mlp")

    def gate_mul(self, x, table, idx, d_m, m_cap, c, out, out_h=None):
        self._check(self.dll.lb2_gate_mul(self.hp, self._stream(), _ptr(x), _ptr(table), _ptr(idx), _ptr(d_m), int(m_cap), int(c), _ptr(out),
                                          _ptr(out_h)), "lb2_gate_mul")

    def gather_rows(self, src, idx, n, c, out):
        self._check(self.dll.lb2_gather_rows(self.hp, self._stream(), _ptr(src), _ptr(idx), int(n), int(c), _ptr(out)), "lb2_gather_rows")

    def guidance_dpm_step(self, eps_c, eps_u, inverse, x_t, x_init, noise, x0_state, n_points, coef: DpmCoef,
                          eps_out, x_next, coord_next, batch_col=None):
        self._check(self.dll.lb2_guidance_dpm_step(self.hp, self._stream(), _ptr(eps_c), _ptr(eps_u), _ptr(inverse), _ptr(x_t), _ptr(x_init),
                                                   _ptr(noise), _ptr(x0_state), int(n_points), coef, _ptr(eps_out), _ptr(x_next),
                                                   _ptr(coord_next), _ptr(batch_col)), "lb2_guidance_dpm_step")

    def farthest_point_sample(self, pts, n, n_samples, out_idx, dist):
        self._check(self.dll.lb2_farthest_point_sample(self.hp, self._stream(), _ptr(pts), int(n), int(n_samples), _ptr(out_idx), _ptr(dist)),
                    "lb2_farthest_point_sample")

    # -- evaluation metrics ----------------------------------------------------------------------------
    def cloud_nn_scratch_bytes(self, nq, nr) -> int:
        return int(self.dll.lb2_cloud_nn_scratch_bytes(int(nq), int(nr)))

    def cloud_nn_distance(self, query, nq, ref, nr, scratch, dist):
        self._check(self.dll.lb2_cloud_nn_distance(self.hp, self._stream(), _ptr(query), int(nq), _ptr(ref), int(nr), _ptr(scratch),
                                                   _ptr(dist)), "lb2_cloud_nn_distance")

    def voxel_hist_scratch_bytes(self, na, nb) -> int:
        return int(self.dll.lb2_voxel_hist_scratch_bytes(int(na), int(nb)))

    def voxel_hist_compare(self, a, na, b, nb, edges, bins, scratch, out):
        """`out`: a device buffer of ctypes.sizeof(VoxelHistResult) bytes"""
        self._check(self.dll.lb2_voxel_hist_compare(self.hp, self._stream(), _ptr(a), int(na), _ptr(b), int(nb), _ptr(edges), int(bins),
                                                    _ptr(scratch), _ptr(out)), "lb2_voxel_hist_compare")

    def threshold_counts(self, d, n, thr, nthr, counts):
        self._check(self.dll.lb2_threshold_counts(self.hp, self._stream(), _ptr(d), int(n), _ptr(thr), int(nthr), _ptr(counts)),
                    "lb2_threshold_counts")


_LIB = None


def get_lib() -> Lib:
    global _LIB
    if _LIB is None:
        _LIB = Lib()
    return _LIB


def get_handle(device) -> Handle:
    return get_lib().handle(device)

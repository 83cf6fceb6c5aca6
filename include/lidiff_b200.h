/*
 * lidiff_b200 — C ABI of the B200-native (sm_100a) implementation of the LiDiff denoising hot path.
 *
 * The reference (PRBonn/LiDiff) reaches this path through three un-vendored Python packages, not
 * through a C interface (SURVEY.md 8b):
 *     import MinkowskiEngine as ME      lidiff/models/minkunet.py:6, tools/diff_completion_pipeline.py:2
 *     pykeops.torch.LazyTensor.argKmin  lidiff/models/minkunet.py:8,412-416
 *     diffusers.DPMSolverMultistepScheduler.step   tools/diff_completion_pipeline.py:6,163
 * Each entry point below names the reference call site(s) it stands behind.  The Python operator
 * surface that mirrors those packages lives in lidiff_b200/ and binds this library with ctypes
 * (INTEGRATION.md shows the stub).
 *
 * Conventions
 *   - every buffer is CALLER-OWNED device memory (a torch CUDA tensor); the library allocates nothing
 *     the caller can see and keeps no state besides the handle's error string;
 *   - all calls are asynchronous on the given `stream` (a cudaStream_t passed as void*), never
 *     synchronise, never allocate => capturable in a CUDA graph;
 *   - data-dependent row counts live in DEVICE int32 scalars (`d_n*`); buffers are sized by a host
 *     capacity (`*_cap`) and kernels read the count on the device;
 *   - return value: 0 = OK, negative = error; `lb2_last_error(h)` gives the message;
 *   - coordinates are int32 rows [b, x, y, z]; features are fp32 row-major (rows, channels);
 *   - no CPU fallback exists: without a CUDA device the calls fail with LB2_ERR_CUDA.
 */
#ifndef LIDIFF_B200_H_
#define LIDIFF_B200_H_

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LB2_OK            0
#define LB2_ERR_ARG      -1
#define LB2_ERR_CUDA     -2
#define LB2_ERR_UNSUP    -3

#define LB2_KEY_EMPTY 0xFFFFFFFFFFFFFFFFull

/* ---- handle ----------------------------------------------------------------------------------- */
int         lb2_create(int device, void** handle);
void        lb2_destroy(void* handle);
const char* lb2_last_error(void* handle);
int         lb2_version(void);
/* number of kernels this library has launched through `handle` since creation (bench gpu_launches) */
int64_t     lb2_launch_count(void* handle);
/* Kernel-selection options of a handle (development / A-B knobs; every setting computes the same results and is exercised by
 * the GPU tests).  Defaults come from the environment variable of the same name (LB2_TC_PAIR, ...) at lb2_create. */
#define LB2_OPT_TC_PAIR       0   /* CTA-pair cta_group::2 conv kernel: 0 off, 1 = Cout 256, 2 = Cout 256 and 128 (default 2) */
#define LB2_OPT_TC_N256       1   /* single-CTA register-total kernel for Cout 256 (default 1) */
#define LB2_OPT_TC_SMALL      2   /* two-drain-warpgroup kernel for Cout <= 128 (default 1) */
#define LB2_OPT_TC_PERSISTENT 3   /* persistent kernels for LB2_ALGO_TC (default 1; 0 = one CTA per tile) */
#define LB2_OPT_TC_FULL_LAG   4   /* generic persistent kernel: S-1 gather lookahead (default 0) */
#define LB2_OPT_TC_NSPLIT     5   /* per-tile kernel: split Cout 256 over two CTAs (default 0) */
#define LB2_OPT_COUNT         6
int         lb2_set_option(void* handle, int option, int value);
int         lb2_get_option(void* handle, int option);   /* value, or a negative LB2_ERR_* */
/* synchronising read-and-clear of the device status word; bit0 = a coordinate fell outside the key
 * range (10 bit batch, 18 bit signed axes) and was clamped.  Returns the word (>= 0) or an error. */
int         lb2_read_status(void* handle, void* stream);

/* ---- hash grid (coordinate manager)  — replaces ME's CoordinateManager -------------------------
 * One hash grid per coordinate level.  `keys` (uint64[cap_table]) and `vals` (int32[2*cap_table]:
 * [0,cap) scratch "first point index", [cap,2cap) row id) are caller-owned; cap_table is a power
 * of two >= 2 * max rows.  Key packing: 10 bit batch | 3 x 18 bit signed coordinate.
 */
typedef struct {
    uint64_t* keys;
    int32_t*  vals;
    int32_t   cap_table;
} lb2_grid;

/* coord = round_half_even(x / resolution) on every column of an (n,ncol) fp32 array.
 * Reference: tools/diff_completion_pipeline.py:71-72, utils/collations.py:8-12 (torch.round(x/res)).
 * div_mode 0: true fp32 division; 1: multiply by fp32(1/resolution) (PyTorch CUDA scalar division). */
int lb2_quantize(void* h, void* stream, const float* x, int64_t n_elem, float resolution, int div_mode,
                 float* out_coord);

/* ME.TensorField.sparse() coordinate part (pipeline:149, minkunet.py:135,597) and ME strided
 * coordinate maps (conv stride 2, minkunet.py:103,184...).
 * Input rows: either fp32 integer-valued coords (`in_f`, floor() is applied; TensorField) or int32
 * coords (`in_i`; a parent level).  If ts_floor > 0 the xyz columns are floored to multiples of
 * ts_floor (stride map).  Output: unique rows in FIRST-OCCURRENCE order, `inverse[i]` = output row of
 * input row i, `*d_nout` = number of unique rows.  `scratch` >= lb2_unique_scratch_bytes(n_cap). */
size_t lb2_unique_scratch_bytes(int64_t n_cap);
int lb2_unique_build(void* h, void* stream,
                     const float* in_f, const int32_t* in_i, const int32_t* d_nin, int32_t n_cap,
                     int32_t ts_floor, lb2_grid grid,
                     int32_t* out_coords, int32_t* inverse, int32_t* d_nout, void* scratch);

/* UNWEIGHTED_AVERAGE voxel features (ME.SparseTensorQuantizationMode, pipeline:77): mean of member
 * point features.  `counts` int32[m_cap] scratch. out (m_cap, c). */
int lb2_voxel_mean(void* h, void* stream, const float* feats, const int32_t* inverse, int32_t n,
                   int32_t c, const int32_t* d_m, int32_t m_cap, float* out, int32_t* counts);

/* Kernel map (ME kernel maps for MinkowskiConvolution / ConvolutionTranspose; minkunet.py:17-24,36-42).
 * Output-stationary neighbour table: nbr[k * nbr_stride + o] = input row at coords(o) + offset_k, or -1.
 *   ks=3: offset_d = (k_d - 1) * step      ks=2: offset_d = k_d * step   (step < 0: transposed map)
 *   k = kx + ks*ky + ks*ks*kz.
 * pair_count (device uint64, optional): += number of (in,out) pairs found (roofline accounting).
 * row_mask (uint32[nout_cap], optional): bit k of row_mask[o] set iff nbr[k][o] >= 0. */
int lb2_kernel_map(void* h, void* stream, lb2_grid grid_in, const int32_t* out_coords,
                   const int32_t* d_nout, int32_t nout_cap, int32_t ks, int32_t step,
                   int32_t* nbr, int64_t nbr_stride, uint64_t* pair_count, uint32_t* row_mask);

/* The 3^3 stride-1 map of a coordinate set onto itself (`grid` was built from exactly `coords`; step = the level's tensor stride):
 * same table and row masks as lb2_kernel_map(ks = 3), with half the hash probes (the pair set is symmetric: row j at offset k of row o
 * <=> o at offset 26 - k of j). */
int lb2_kernel_map_self(void* h, void* stream, lb2_grid grid, const int32_t* coords, const int32_t* d_n, int32_t n_cap,
                        int32_t step, int32_t* nbr, int64_t nbr_stride, uint64_t* pair_count, uint32_t* row_mask);

/* Execution order of the output rows for lb2_spconv_forward (no reference counterpart: scheduling only).
 * perm[0..n) = the rows 0..n-1 sorted by their neighbour mask (kvol 27: centre-only rows, rows with one neighbour grouped
 * by it, then the rest in mask order; kvol <= 8: by the 8-bit mask) so that 128-row tiles skip unpopulated kernel offsets.
 * Results do not depend on the order.  scratch >= lb2_row_order_scratch_bytes(n_cap).
 * coords (optional, kvol 27 only): the rows' int32 [b,x,y,z] coordinates; rows of equal mask are then ordered by the Morton code of
 * (x,y,z) >> coord_shift (coord_shift = log2 of the level's tensor stride), which makes the tiles of large mask groups spatially
 * compact (L2 locality of the gathers). */
size_t lb2_row_order_scratch_bytes(int32_t n_cap);
int lb2_row_order(void* h, void* stream, const uint32_t* row_mask, const int32_t* d_n, int32_t n_cap,
                  int32_t kvol, int32_t* perm, void* scratch, const int32_t* coords, int32_t coord_shift);

/* Cost order of the tiles of a map (scheduling only; results do not depend on it): order128[i] / order256[i] = index of the i-th most
 * expensive 128-row tile / 256-row super-tile of the row order `row_perm`, cost = number of kernel offsets the tile has to run (popcount of
 * the OR of its rows' masks); entries beyond the live tile count are -1.  The persistent convolution kernels deal tiles to their CTAs in
 * snake order over this sequence (lb2_conv_desc.tile_order128 / tile_order256), which balances a static assignment to within 1-3 %.
 * order128: cdiv(n_cap,128) ints, order256: cdiv(n_cap,256) ints, scratch: cdiv(n_cap,128) * 4 bytes. */
int lb2_tile_order(void* h, void* stream, const uint32_t* row_mask, const int32_t* row_perm, const int32_t* d_n, int32_t n_cap,
                   int32_t* order128, int32_t* order256, void* scratch);

/* Dense / residual split of a map's row masks for the CTA-pair convolution (scheduling only: the pair set is unchanged).  For every
 * 256-row super-tile of the row order `row_perm`, offset k is dense when at least min_rows of its rows have it (min_rows = 0: all offsets).
 * dense_mask[row] = row_mask[row] & dense offsets of its super-tile, res_mask[row] = row_mask[row] & ~those (uint32[n_cap] each).
 * The output-stationary kernel runs dense_mask (zero rows of sparse offsets are not multiplied); lb2_pair_list(row_mask = res_mask)
 * compacts the rest for lb2_spconv_scatter. */
int lb2_tile_split(void* h, void* stream, const uint32_t* row_mask, const int32_t* row_perm, const int32_t* d_n, int32_t n_cap,
                   int32_t kvol, int32_t min_rows, uint32_t* dense_mask, uint32_t* res_mask);

/* ---- sparse convolution  — replaces ME.MinkowskiConvolution(+Transpose) forward, with the
 * MinkowskiBatchNorm(eval)/MinkowskiReLU/residual-add/ME.cat/gate-multiply that follow it in
 * minkunet.py:13-80,431,464 fused as prologue/epilogue.
 *   out[o] = epi( sum_k [in1|in2][nbr[k][o]] @ W[k] )
 *   epi(y) = relu?( (y + pre_add[o])*scale + shift + residual[o] );  optional second output
 *   out_gated = epi(y) * gate_table[gate_idx[o]].
 * Up to two guidance passes (conditional/unconditional) share W and the map. */
typedef struct {
    const float*   in1;         /* (rows_in, c1) */
    const float*   in2;         /* (rows_in, c2) or NULL  (ME.cat as a second K segment) */
    const float*   residual;    /* (m, cout) or NULL */
    float*         out;         /* (m, cout) or NULL */
    const float*   gate_table;  /* (rows_g, cout) or NULL */
    const int32_t* gate_idx;    /* (m) or NULL (=> row 0 broadcast) */
    float*         out_gated;   /* (m, cout) or NULL */
    const float*   pre_add;     /* (m, cout) or NULL: added to the raw convolution sum before the affine
                                   (the off-centre part computed by lb2_spconv_scatter) */
    /* optional fp16 "split" companions (row = [C halfs hi | C halfs lo], x ~= hi + lo; same 4C bytes as fp32):
       inputs let the tensor-core kernels gather with cp.async instead of converting in registers,
       outputs are written by the epilogue next to the fp32 tensors. */
    const void*    in1_h;       /* (rows_in, 2*c1) fp16 or NULL */
    const void*    in2_h;       /* (rows_in, 2*c2) fp16 or NULL */
    void*          out_h;       /* (m, 2*cout) fp16 or NULL */
    void*          out_gated_h; /* (m, 2*cout) fp16 or NULL */
    /* An activation may exist as its companion only: in1/in2 may be NULL when in1_h/in2_h are given (tensor-core variants), out /
       out_gated may be NULL when out_h / out_gated_h are given, and the residual may be read from a companion (hi + lo): */
    const void*    residual_h;  /* (m, 2*cout) fp16 or NULL; used when residual == NULL */
} lb2_conv_io;

typedef struct {
    int32_t        c1, c2, cout, kvol;
    const float*   weight;      /* (kvol, c1+c2, cout) fp32 */
    const void*    weight_packed; /* tensor-core layout from lb2_pack_weights or NULL */
    const float*   scale;       /* (cout) or NULL */
    const float*   shift;       /* (cout) or NULL */
    int32_t        relu;
    const int32_t* nbr;         /* [kvol][nbr_stride] or NULL => identity map (1x1 conv) */
    int64_t        nbr_stride;
    const int32_t* d_mout;      /* device row count or NULL => mout_cap */
    int32_t        mout_cap;
    const int32_t* row_perm;    /* execution order from lb2_row_order or NULL (natural order) */
    const uint32_t* row_mask;   /* per output row: bit k set <=> nbr[k][row] >= 0 (lb2_kernel_map's row_mask) or NULL.
                                   Every variant (tensor-core and CUDA-core) convolves only the offsets whose bit is
                                   set, so a subset (lb2_tile_split's dense_mask) convolves that subset of pairs */
    int32_t        npass;       /* 1 or 2 */
    lb2_conv_io    io[2];
    const int32_t* tile_order128;  /* from lb2_tile_order or NULL (tiles in row-order sequence, heaviest-looking last) */
    const int32_t* tile_order256;
} lb2_conv_desc;

#define LB2_ALGO_AUTO  0
#define LB2_ALGO_FFMA  1    /* fp32 CUDA-core implicit GEMM */
#define LB2_ALGO_TC    2    /* tcgen05 FP16x3 split-precision implicit GEMM (needs weight_packed), persistent CTAs */
#define LB2_ALGO_TC_TILE 3  /* same math, one CTA per 128-row tile (non-persistent reference variant) */
int lb2_spconv_forward(void* h, void* stream, const lb2_conv_desc* d, int algo);

/* The same convolution in gather-GEMM-scatter form (what ME's GPU backend does per kernel offset) for levels
 * with few neighbours per voxel: lb2_pair_list compacts the (in,out) pairs of a kernel map per offset (optionally
 * skipping one offset, e.g. the centre 13 of a 3^3 kernel), lb2_spconv_scatter computes
 *     out[pair_out] += in[pair_in] @ W[k]        (tensor cores, FP16x3, fp32 red.add; order-dependent last bits)
 * into a buffer that lb2_spconv_forward then consumes as `pre_add` while it handles the skipped offset with
 * kvol = 1, or the dense offsets of lb2_tile_split.  Cout <= 256; W[k] stays in shared memory when it fits (Cout <= 128,
 * Cin <= 256), otherwise it streams per 64-channel K chunk.
 * lb2_pair_list's row_mask (optional): only the pairs (nbr[k][o], o) with bit k of row_mask[o] set. */
typedef struct {
    int32_t        c1, c2, cout, kvol;
    const void*    weight_packed;
    const int32_t* pair_in;        /* [pairs] input row  */
    const int32_t* pair_out;       /* [pairs] output row */
    const int32_t* koff;           /* [kvol+1] first pair of each offset */
    const int32_t* tile_off;       /* [kvol+1] first 128-pair tile of each offset */
    int32_t        npass;
    const float*   in1[2];
    const float*   in2[2];
    const void*    in1_h[2];       /* fp16 split companions of in1 / in2 (or NULL), see lb2_conv_io */
    const void*    in2_h[2];
    float*         out[2];         /* (m, cout) accumulation buffers */
    const int32_t* d_zero_rows;    /* rows to clear first: device count (or NULL => zero_rows_cap) */
    int32_t        zero_rows_cap;  /* 0 = caller already cleared `out` */
} lb2_scatter_desc;
size_t lb2_pair_list_scratch_bytes(void);
int lb2_pair_list(void* h, void* stream, const int32_t* nbr, int64_t nbr_stride, const int32_t* d_nout,
                  int32_t nout_cap, int32_t kvol, int32_t skip_k, int32_t* pair_in, int32_t* pair_out,
                  int32_t* koff, int32_t* tile_off, void* scratch, const uint32_t* row_mask);
int lb2_spconv_scatter_supported(int32_t c1, int32_t c2, int32_t cout, int32_t kvol);
int lb2_spconv_scatter(void* h, void* stream, const lb2_scatter_desc* d);

/* FP16 hi/lo split (power-of-two pre-scaled) + UMMA shared-memory image of a (kvol, cin, cout) fp32 weight
 * for LB2_ALGO_TC. */
size_t lb2_packed_weight_bytes(int32_t kvol, int32_t cin, int32_t cout);
int lb2_pack_weights(void* h, void* stream, const float* weight, int32_t kvol, int32_t cin, int32_t cout,
                     void* packed);

/* ---- nearest partial-scan voxel — replaces pykeops argKmin(1) in MinkUNetDiff.match_part_to_full
 * (minkunet.py:403-418): idx[q] = argmin_j |cq - ck_j|^2 over [b*2*max, x, y, z], ties -> lowest j. */
int lb2_nn_match(void* h, void* stream, const int32_t* q_coords, const int32_t* d_nq, int32_t nq_cap,
                 const int32_t* k_coords, const int32_t* d_nk, int32_t nk_cap, int32_t batch_scale,
                 int32_t* idx);

/* Same result as lb2_nn_match when the keys are the rows of a hash grid on a lattice of pitch key_stride
 * (the stride-16 partial-scan level): exact shell search around the query's lattice cell, exhaustive
 * fallback after max_ring shells.  Different-batch keys never match (lb2_nn_match batch_scale = 0). */
int lb2_nn_match_grid(void* h, void* stream, const int32_t* q_coords, const int32_t* d_nq, int32_t nq_cap,
                      const int32_t* k_coords, const int32_t* d_nk, int32_t nk_cap, lb2_grid key_grid,
                      int32_t key_stride, int32_t max_ring, int32_t* idx);

/* Variant with the key lattice in shared memory: lb2_nn_table_build re-hashes the (<= 8192) keys once per scan into
 * a compact table (`table`: lb2_nn_table_bytes() bytes), lb2_nn_match_table probes it from shared memory.  If the
 * keys do not fit the table is marked overflowing and every query takes the exhaustive path (still exact). */
size_t lb2_nn_table_bytes(void);
int lb2_nn_table_build(void* h, void* stream, const int32_t* k_coords, const int32_t* d_nk, int32_t nk_cap, void* table);
int lb2_nn_match_table(void* h, void* stream, const int32_t* q_coords, const int32_t* d_nq, int32_t nq_cap,
                       const int32_t* k_coords, const int32_t* d_nk, int32_t nk_cap, const void* table,
                       int32_t key_stride, int32_t max_ring, int32_t* idx);

/* Variant for keys that stay fixed over many calls (the conditioning scan): lb2_nn_tree_build sorts them along a
 * Morton curve and builds a bounding-box hierarchy once (`tree`: lb2_nn_tree_bytes(nk_cap) bytes); lb2_nn_match_tree
 * searches it exactly (same result as lb2_nn_match with batch_scale = 0, incl. lowest-row ties) in ~log(nk) box
 * tests per query, independent of how far the query is from the keys.  Optional hint: hint_idx[hint_of ? hint_of[q] : q]
 * names a key row that is probably close to query q (e.g. the answer of the coarser voxel containing it; needs
 * k_coords): the search starts from that key's distance as its bound; the result does not depend on the hint. */
size_t lb2_nn_tree_bytes(int32_t nk_cap);
int lb2_nn_tree_build(void* h, void* stream, const int32_t* k_coords, const int32_t* d_nk, int32_t nk_cap, void* tree);
int lb2_nn_match_tree(void* h, void* stream, const int32_t* q_coords, const int32_t* d_nq, int32_t nq_cap,
                      const void* tree, int32_t nk_cap, const int32_t* k_coords, const int32_t* hint_of,
                      const int32_t* hint_idx, int32_t* idx);

/* ---- small dense layers — torch.nn.Linear (+LeakyReLU) of the gate / head MLPs
 * (minkunet.py:165-181,376-380): y = act(x @ W^T + b [+ addend]); W is (n_out, n_in) torch layout.
 * act: 0 none, 1 LeakyReLU(0.1), 2 tanh.  rows read from d_m if non-NULL.
 * Optional input transform x' = pre_act(x + prebias[k]) (prebias (n_in) or NULL): evaluates the
 * hoisted gate MLP  latemp(cat(p,t)) = W2 . leaky(Wp.p + (Wt.t + b1)) + b2  (SURVEY.md App. D.1). */
int lb2_linear(void* h, void* stream, const float* x, int64_t ldx, const float* w, const float* b,
               const float* addend, int64_t ld_addend, int32_t m_cap, const int32_t* d_m,
               int32_t n_in, int32_t n_out, int32_t act, float* y, int64_t ldy,
               const float* prebias, int32_t pre_act);

/* The head of the U-Nets in one pass over the rows — `last` of MinkUNetDiff / MinkUNet (minkunet.py:376-380, :585-588):
 * y = out_act(W1 . LeakyReLU_0.1(W0 . x + b0) + b1), W0 (n_hid, n_in), W1 (n_out, n_hid) in torch layout; out_act as lb2_linear.
 * npass (1 or 2) row blocks x + p * x_pass_stride -> y + p * y_pass_stride (floats) share the weights and the launch.
 * n_in: multiple of 16, <= 128; n_hid <= 64; n_out <= 24; ldx a multiple of 4. */
int lb2_head_mlp(void* h, void* stream, const float* x, int64_t ldx, int64_t x_pass_stride, const float* w0, const float* b0,
                 const float* w1, const float* b1, int32_t m_cap, const int32_t* d_m, int32_t n_in, int32_t n_hid,
                 int32_t n_out, int32_t out_act, int32_t npass, float* y, int64_t ldy, int64_t y_pass_stride);

/* x * w row-gather multiply (`x0*w0`, minkunet.py:431...): out[r] = x[r] * table[idx ? idx[r] : 0];
 * out_h: optional fp16 split companion of out (see lb2_conv_io); out may be NULL when out_h is given. */
int lb2_gate_mul(void* h, void* stream, const float* x, const float* table, const int32_t* idx,
                 const int32_t* d_m, int32_t m_cap, int32_t c, float* out, void* out_h);

/* out[i] = src[idx[i]]  (SparseTensor.slice / x_part.F[match], minkunet.py:418,497) */
int lb2_gather_rows(void* h, void* stream, const float* src, const int32_t* idx, int32_t n, int32_t c,
                    float* out);

/* ---- fused tail — classifier-free guidance (pipeline:153) + DPM-Solver++(2M) SDE update
 * (pipeline:162-163; diffusers DPMSolverMultistepScheduler.step) + next TensorField features and
 * coordinates (pipeline:164 -> :68-84), one thread per point coordinate.
 *   eps      = eps_u[v] + w * (eps_c[v] - eps_u[v]),  v = inverse[point]   (voxel eps, (m,3) fp32)
 *   sample   = x_t - x_init;  x0 = (sample - sigma_s*eps)/alpha_s           (fp64 like the pipeline)
 *   prev     = c_sample*sample + c_x0*x0 [+ 0.5*c_x0*(x0 - x0_prev)/r0] + c_noise*noise
 *   x_next   = fp32(x_init + prev);  coord = round_half_even(x_next / resolution)
 * coord_next is (n,4) fp32 [b, x, y, z] ready for lb2_unique_build (b from batch_col or 0).
 * x0_state (n*3 fp64) is read when second_order != 0 and always overwritten with the new x0. */
typedef struct {
    double c_sample, c_x0, c_noise, sigma_s, alpha_s, inv_r0;
    float  guidance_w, resolution;
    int32_t second_order, div_mode, f64_state;
} lb2_dpm_coef;
int lb2_guidance_dpm_step(void* h, void* stream, const float* eps_c, const float* eps_u,
                          const int32_t* inverse, const float* x_t, const double* x_init,
                          const float* noise, double* x0_state, int64_t n_points, lb2_dpm_coef coef,
                          float* eps_out, float* x_next, float* coord_next /* (n,4) */,
                          const float* batch_col /* (n) or NULL */);

/* ---- farthest point sampling — open3d farthest_point_down_sample used by preprocess_scan
 * (pipeline:97-99): start at point 0, repeatedly take the first argmax of the running min squared
 * distance (fp64).  out_idx[n_samples] selection order; dist_scratch fp64[n]. */
int lb2_farthest_point_sample(void* h, void* stream, const double* pts, int32_t n, int32_t n_samples,
                              int32_t* out_idx, double* dist_scratch);

/* ---- evaluation metrics — lidiff/utils/metrics.py (RMSE, ChamferDistance, PrecisionRecall, CompletionIoU) and
 * lidiff/utils/histogram_metrics.py (compute_hist_metrics), which use open3d's KDTreeFlann and dense np.histogramdd grids.
 * Point clouds are fp64 (n, 3) row-major; n < 2^31.  Results stay on the device. */

/* dist[i] = min_j |query[i] - ref[j]|, exact in fp64: squared distances are evaluated as (dx*dx + dy*dy) + dz*dz without FMA
 * contraction and the square root is taken of the minimum, so dist equals numpy's np.sqrt(((q - r)**2).sum(1)) for the nearest r
 * bit for bit.  A bounding-box hierarchy over the Morton-sorted reference keeps the cost ~log(nr) per query however far the query
 * lies from the reference.  nq = 0 is a no-op; nr must be > 0.  scratch >= lb2_cloud_nn_scratch_bytes(nq, nr) (0 = bad sizes). */
size_t lb2_cloud_nn_scratch_bytes(int64_t nq, int64_t nr);
int lb2_cloud_nn_distance(void* h, void* stream, const double* query, int64_t nq, const double* ref, int64_t nr,
                          void* scratch, double* dist);

/* Two clouds on one voxel grid of bins^3 cells with per-axis edges `edges` (bins + 1 ascending fp64, np.linspace(-R, R, bins + 1)
 * in the reference), binned like np.histogramdd: bin = searchsorted(edges, x, 'right') - 1, x == edges[bins] goes in the last bin,
 * a point with a coordinate outside [edges[0], edges[bins]] is dropped.  The grid is never materialised (sorted bin keys).
 *   n_a, n_b        points of a / b inside the grid;  occ_a, occ_b, occ_ab  occupied cells of a, of b, of both
 *                   (CompletionIoU with a = ground truth: tp = occ_ab, fn = occ_a - tp, fp = occ_b - tp);
 *   jsd_3d          scipy.spatial.distance.jensenshannon (base e) of the two count histograms;
 *   jsd_bev         the same of the per-(x, y)-column numbers of occupied z cells (histogram_metrics.py with bev=True).
 * Deterministic (fixed-order fp64 reductions).  bins < 2^21 (keys 2 * bins^3 fit 64 bits).
 * scratch >= lb2_voxel_hist_scratch_bytes(na, nb); `out` is device memory. */
typedef struct {
    int64_t n_a, n_b;
    int64_t occ_a, occ_b, occ_ab;
    double  jsd_3d, jsd_bev;
} lb2_voxel_hist_result;
size_t lb2_voxel_hist_scratch_bytes(int64_t na, int64_t nb);
int lb2_voxel_hist_compare(void* h, void* stream, const double* a, int64_t na, const double* b, int64_t nb,
                           const double* edges, int32_t bins, void* scratch, lb2_voxel_hist_result* out);

/* counts[t] = #{i : d[i] < thr[t]} (strict, as np.where(d < t)) for nthr <= 8192 ascending thresholds; counts int64[nthr]. */
int lb2_threshold_counts(void* h, void* stream, const double* d, int64_t n, const double* thr, int32_t nthr, int64_t* counts);

#ifdef __cplusplus
}
#endif
#endif  /* LIDIFF_B200_H_ */

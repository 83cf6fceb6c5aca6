// K4 (variant B) — sparse convolution as an output-stationary implicit GEMM on the 5th-gen tensor
// cores (tcgen05.mma, accumulator in TMEM), split-precision FP16x3 so that 49 stacked layers stay
// inside the 1e-3 fp32 parity bar:
//     x = x_hi + x_lo (fp16 each),  w*2^k = w_hi + w_lo,   x.w ~= (x_hi.w_hi + x_lo.w_hi + x_hi.w_lo) * 2^-k
// (22 mantissa bits per operand; the dropped x_lo.w_lo term is ~2^-22 relative.  SURVEY.md App. B.4
// planned BF16x3; measured on the B200 it reached 1.3e-3 max-element error through the 49-layer U-Net,
// FP16x3 costs the same three kind::f16 MMAs and is ~100x more accurate.  Weights are pre-scaled by a
// power of two per layer so their low parts stay in fp16's normal range; activations saturate at
// +-65504.)
//
// One CTA owns 128 output rows x all Cout channels.  Warp roles (320 threads):
//   warps 0-3  A producers: gather the neighbour rows of kernel offset k / channel chunk c from the
//              fp32 feature matrix, split to fp16 hi/lo in registers, store into the UMMA K-major
//              SWIZZLE_128B shared-memory image.
//   warp 4     MMA issuer: one thread issues 3 x (chunk/16) tcgen05.mma per stage, tcgen05.commit
//              releases the stage / signals the drain warps.
//   warp 5     B producer: one thread streams the pre-packed weight image of (k, c) with one
//              cp.async.bulk (TMA bulk copy, mbarrier complete_tx) per stage.
//   warps 6-9  drain + epilogue: TWO-LEVEL ACCUMULATION.  The tensor core adds into TMEM with
//              truncation, so the error of a chained accumulation grows linearly with the number of MMA
//              steps (measured: ~1300 steps -> 8e-5 relative per layer, 1e-3 through the 49-layer
//              U-Net).  The MMA chain is therefore cut into groups of <= ~128 steps; after each group
//              these warps tcgen05.ld the partial sum, add it to a running fp32 total (round-to-nearest,
//              kept in a second TMEM region via tcgen05.st) and release the accumulator.  The last
//              group's drain is the epilogue: BN affine + residual + ReLU + gate -> global.
// Kernel offsets where none of the tile's 128 rows has a neighbour are skipped by every role.
//
// Stands behind ME.MinkowskiConvolution(+Transpose) forward, /root/reference/lidiff/models/minkunet.py:17-24,36-42,53-74.
#include "common.cuh"
#include <algorithm>
#include <stdlib.h>
#include "tc_common.cuh"

namespace tc {

constexpr int NUM_PRODUCER = 128;
constexpr int THREADS = 320;
constexpr int DRAIN_WARP0 = 6;        // warps 6..9
constexpr int STEP_BUDGET = 64;       // max chained MMA steps per TMEM accumulation group
constexpr int MAX_KVOL = 27;
constexpr int MAX_STAGES = 4;

struct Params {
    int c1, c2, cout, kvol;
    const unsigned char* wpacked;
    const float* scale;
    const float* shift;
    int relu;
    const int* nbr;
    long long nbr_stride;
    const int* d_mout;
    int mout_cap;
    const int* row_perm;
    const unsigned* row_mask;   // offsets to convolve per output row (NULL: all of the map)
    int stages, nchunks, tmem_cols, tot_col, group;     // tot_col: TMEM column of the running total; group: offsets per drain
    int nbuf, acc_stride;
    int ncta;                                           // output channels handled by one CTA (cout or cout/2): blockIdx.z picks the slice                               // ping-pong accumulators (2 when 3 regions fit in TMEM) and their column pitch
    lb2_conv_io io[2];
};

__global__ void __launch_bounds__(THREADS, 1) k_spconv_tc(const Params p) {
    extern __shared__ unsigned char smem_raw[];
    const int M = p.d_mout ? min(*p.d_mout, p.mout_cap) : p.mout_cap;
    const int m0 = blockIdx.x * BM;
    if (m0 >= M) return;
    const lb2_conv_io io = p.io[blockIdx.y];
    const int n0 = blockIdx.z * p.ncta;              // first output channel of this CTA
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ctot = p.c1 + p.c2;

    // ---- shared memory carve-up (tiles 1024-byte aligned for SWIZZLE_128B) -----------------------------
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    unsigned char* gen = smem_raw + (base - raw);
    const uint32_t b_tile = (uint32_t)p.ncta * 128u;                 // one fp16 B tile (hi or lo) of this CTA's channels
    const uint32_t b_full = (uint32_t)p.cout * 128u;                 // the same tile over all cout channels (packed layout)
    const float out_scale = __ldg(reinterpret_cast<const float*>(p.wpacked) + 1);     // 2^-k of the packed weights
    const uint32_t stage_bytes = 2u * A_TILE + 2u * b_tile;
    unsigned char* tail = gen + (size_t)p.stages * stage_bytes;
    int* idx_s = reinterpret_cast<int*>(tail);                       // [kvol][BM]
    uint64_t* bars = reinterpret_cast<uint64_t*>(tail + MAX_KVOL * BM * sizeof(int));
    uint32_t* misc = reinterpret_cast<uint32_t*>(bars + 3 * MAX_STAGES + 4);   // [0] tmem base, [1] offset mask
    int* row_s = reinterpret_cast<int*>(misc + 4);                             // [BM] output row of each tile slot
    const uint32_t bar0 = smem_u32(bars);
    auto full_a = [&](int s) { return bar0 + 8u * s; };
    auto full_b = [&](int s) { return bar0 + 8u * (MAX_STAGES + s); };
    auto empty = [&](int s) { return bar0 + 8u * (2 * MAX_STAGES + s); };
    auto acc_full = [&](int b) { return bar0 + 8u * (3 * MAX_STAGES + b); };        // MMA group complete -> drain warps
    auto acc_empty = [&](int b) { return bar0 + 8u * (3 * MAX_STAGES + 2 + b); };   // drain complete     -> MMA issuer

    if (threadIdx.x == 0) {
        for (int s = 0; s < p.stages; ++s) { mbar_init(full_a(s), NUM_PRODUCER); mbar_init(full_b(s), 1); mbar_init(empty(s), 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(acc_full(b), 1); mbar_init(acc_empty(b), 128); }
        misc[1] = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 4) {      // TMEM allocation (whole warp), result written to misc[0]
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&misc[0])), "r"((uint32_t)p.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    __syncthreads();
    // ---- neighbour indices of this tile + mask of non-empty kernel offsets -----------------------------
    if (threadIdx.x < BM) {
        const int slot = m0 + threadIdx.x;
        const int row = (slot < M) ? (p.row_perm ? __ldg(p.row_perm + slot) : slot) : -1;
        row_s[threadIdx.x] = row;
        const uint32_t rmask = (row >= 0 && p.row_mask) ? __ldg(p.row_mask + row) : 0xffffffffu;
        uint32_t mymask = 0;
        for (int k0 = 0; k0 < p.kvol; k0 += 9) {        // 9 independent loads in flight, then the votes
            int v[9];
#pragma unroll
            for (int q = 0; q < 9; ++q) {
                const int k = k0 + q;
                v[q] = -1;
                if (k < p.kvol && row >= 0 && ((rmask >> k) & 1u)) v[q] = p.nbr ? __ldg(p.nbr + (long long)k * p.nbr_stride + row) : row;
            }
#pragma unroll
            for (int q = 0; q < 9; ++q) {
                const int k = k0 + q;
                if (k < p.kvol) {
                    idx_s[k * BM + threadIdx.x] = v[q];
                    if (__any_sync(0xffffffffu, v[q] >= 0)) mymask |= 1u << k;
                }
            }
        }
        if (lane == 0 && mymask) atomicOr(&misc[1], mymask);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_d = misc[0];
    const uint32_t kmask = misc[1];
    const int n_off = __popc(kmask);
    const int n_groups = (n_off + p.group - 1) / p.group;

    if (warp < 4) {
        // =========================== A producers ===========================
        const int sub = threadIdx.x & 7;           // 8-channel group inside the 64-channel chunk
        const int rbase = threadIdx.x >> 3;        // 0..15
        const bool use_h = (io.in1_h != nullptr) && (p.c2 == 0 || io.in2_h != nullptr);   // fp16 split inputs: cp.async gather
        const int D = p.stages - 1;                // cp.async lookahead: stages still landing while the next is issued
        int it = 0, arrived = 0;
        for (uint32_t km = kmask; km; km &= km - 1) {
            const int k = __ffs(km) - 1;
            const int* idxk = idx_s + k * BM;
            int src[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) src[j] = idxk[rbase + 16 * j];
            for (int c = 0; c < p.nchunks; ++c, ++it) {
                const int s = it % p.stages;
                mbar_wait(empty(s), ((it / p.stages) & 1) ^ 1);
                unsigned char* a_hi = gen + (size_t)s * stage_bytes;
                const uint32_t a_hi_u = base + (uint32_t)s * stage_bytes;
                const int ch = c * KC + sub * 8;
                if (ch < ctot) {
                    const bool first = ch < p.c1;
                    const int cw = first ? p.c1 : p.c2;
                    const int co = first ? ch : ch - p.c1;
                    if (use_h) produce_a_split(reinterpret_cast<const __half*>(first ? io.in1_h : io.in2_h), cw, co, src, a_hi_u, a_hi_u + A_TILE, rbase, sub);
                    else produce_a_f32(first ? io.in1 : io.in2, cw, co, src, a_hi, a_hi + A_TILE, rbase, sub);
                }
                if (use_h) {
                    cp_async_commit();
                    if (it >= D) {                 // the copies of iteration it-D have landed
                        cp_async_wait_dyn(D);
                        fence_proxy_async();
                        mbar_arrive(full_a(arrived % p.stages));
                        ++arrived;
                    }
                } else {
                    fence_proxy_async();
                    mbar_arrive(full_a(s));
                }
            }
        }
        if (use_h) {
            cp_async_wait<0>();
            fence_proxy_async();
            for (; arrived < it; ++arrived) mbar_arrive(full_a(arrived % p.stages));
        }
    } else if (warp == 4) {
        // =========================== MMA issuer ===========================
        if (lane == 0) {
            const uint32_t idesc = make_idesc(p.ncta);
            int it = 0, in_group = 0, group_idx = 0, off_idx = 0;
            for (uint32_t km = kmask; km; km &= km - 1, ++off_idx) {
                const int buf = group_idx % p.nbuf;
                const uint32_t tmem_acc = tmem_d + (uint32_t)(buf * p.acc_stride);
                if (in_group == 0 && group_idx >= p.nbuf) {       // this accumulator's previous group must be drained first
                    mbar_wait(acc_empty(buf), ((group_idx / p.nbuf) - 1) & 1);
                    tc_fence_after();
                }
                for (int c = 0; c < p.nchunks; ++c, ++it) {
                    const int s = it % p.stages;
                    const uint32_t par = (it / p.stages) & 1;
                    mbar_wait(full_b(s), par);
                    mbar_wait(full_a(s), par);
                    tc_fence_after();
                    const uint32_t a_hi = base + (uint32_t)s * stage_bytes, a_lo = a_hi + A_TILE;
                    const uint32_t b_hi = a_lo + A_TILE, b_lo = b_hi + b_tile;
                    const int ksteps = min(KC, ctot - c * KC) >> 4;
                    for (int ks = 0; ks < ksteps; ++ks) {
                        const uint64_t dah = make_desc(a_hi + ks * 32), dal = make_desc(a_lo + ks * 32);
                        const uint64_t dbh = make_desc(b_hi + ks * 32), dbl = make_desc(b_lo + ks * 32);
                        umma(tmem_acc, dah, dbh, idesc, (in_group | c | ks) ? 1u : 0u);   // first MMA of a group overwrites
                        umma(tmem_acc, dal, dbh, idesc, 1);
                        umma(tmem_acc, dah, dbl, idesc, 1);
                    }
                    umma_commit(empty(s));            // frees the stage when these MMAs have read it
                }
                if (++in_group == p.group || off_idx == n_off - 1) {
                    umma_commit(acc_full(buf));       // partial sum of this group complete -> drain warps
                    in_group = 0;
                    ++group_idx;
                }
            }
        }
        __syncwarp();
    } else if (warp >= DRAIN_WARP0) {
        // =========================== drain + epilogue (two-level accumulation) ===========================
        const int q4 = warp & 3;                                   // TMEM lane quarter this warp may access
        const uint32_t lane_base = (uint32_t)(q4 * 32) << 16;
        float* stage_c = reinterpret_cast<float*>(gen);            // [BM][pitch] fp32, reuses the (then idle) stage ring
        const int pitch = p.ncta + 4;                              // +4 floats: conflict-free 16-byte row writes
        for (int g = 0; g < max(n_groups, 1); ++g) {
            const bool last = g >= n_groups - 1;
            const int buf = g % p.nbuf;
            const uint32_t acc_col = (uint32_t)(buf * p.acc_stride);
            if (n_groups > 0) {
                mbar_wait(acc_full(buf), (g / p.nbuf) & 1);
                tc_fence_after();
            }
            for (int c0 = 0; c0 < p.ncta; c0 += 32) {
                float acc[32];
                if (n_groups > 0) {
                    uint32_t r[32];
                    tmem_ld32(tmem_d + lane_base + acc_col + (uint32_t)c0, r);
                    if (g > 0) {
                        uint32_t t[32];
                        tmem_ld32(tmem_d + lane_base + (uint32_t)(p.tot_col + c0), t);
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 32; ++j) acc[j] = __fadd_rn(__uint_as_float(t[j]), __uint_as_float(r[j]));
                    } else {
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 32; ++j) acc[j] = __uint_as_float(r[j]);
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) acc[j] = 0.f;
                }
                if (!last) {                       // running total back to TMEM
                    uint32_t t[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) t[j] = __float_as_uint(acc[j]);
                    tmem_st32(tmem_d + lane_base + (uint32_t)(p.tot_col + c0), t);
                } else {                           // final sum -> shared-memory staging tile (the stage ring is idle now)
                    float* srow = stage_c + (size_t)(q4 * 32 + lane) * pitch + c0;
#pragma unroll
                    for (int q = 0; q < 8; ++q)
                        *reinterpret_cast<float4*>(srow + q * 4) = make_float4(acc[q * 4] * out_scale, acc[q * 4 + 1] * out_scale,
                                                                               acc[q * 4 + 2] * out_scale, acc[q * 4 + 3] * out_scale);
                }
            }
            if (!last) {
                asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                tc_fence_before();
                mbar_arrive(acc_empty(buf));       // this accumulator may be overwritten by its next group
            }
        }
        // ---- epilogue, coalesced: each drain warp owns 32 tile rows and walks their (row, 4-channel) elements with
        //      consecutive lanes on consecutive channels, so every global access is a contiguous row segment ----------
        asm volatile("bar.sync 1, 128;" ::: "memory");          // the 4 drain warps: staging tile complete
        const int nv = p.ncta >> 2;                              // float4 per row (this CTA's channels)
        for (int e = lane; e < 32 * nv; e += 32) {
            const int rr = q4 + 4 * (e / nv);
            const int lcol = (e % nv) * 4;
            const int col = n0 + lcol;
            const int orow = row_s[rr];
            if (orow < 0) continue;
            const long long ro = (long long)orow * p.cout;
            const float4 a4 = *reinterpret_cast<const float4*>(stage_c + (size_t)rr * pitch + lcol);
            float y[4] = {a4.x, a4.y, a4.z, a4.w};
            if (io.pre_add) {
                const float4 t4 = __ldg(reinterpret_cast<const float4*>(io.pre_add + ro + col));
                y[0] += t4.x; y[1] += t4.y; y[2] += t4.z; y[3] += t4.w;
            }
            if (p.scale) {
                const float4 s4 = __ldg(reinterpret_cast<const float4*>(p.scale + col));
                const float4 h4 = __ldg(reinterpret_cast<const float4*>(p.shift + col));
                y[0] = fmaf(y[0], s4.x, h4.x); y[1] = fmaf(y[1], s4.y, h4.y); y[2] = fmaf(y[2], s4.z, h4.z); y[3] = fmaf(y[3], s4.w, h4.w);
            }
            if (io.residual || io.residual_h) {
                const float4 t4 = load_residual4(io.residual, io.residual_h, orow, p.cout, col);
                y[0] += t4.x; y[1] += t4.y; y[2] += t4.z; y[3] += t4.w;
            }
            if (p.relu) {
#pragma unroll
                for (int j = 0; j < 4; ++j) y[j] = fmaxf(y[j], 0.f);
            }
            if (io.out) *reinterpret_cast<float4*>(io.out + ro + col) = make_float4(y[0], y[1], y[2], y[3]);
            if (io.out_h) store_split4(io.out_h, orow, p.cout, col, y);
            if (io.out_gated || io.out_gated_h) {
                if (io.gate_table) {
                    const long long g = io.gate_idx ? __ldg(io.gate_idx + orow) : 0;
                    const float4 g4 = __ldg(reinterpret_cast<const float4*>(io.gate_table + g * p.cout + col));
                    y[0] *= g4.x; y[1] *= g4.y; y[2] *= g4.z; y[3] *= g4.w;
                }
                if (io.out_gated) *reinterpret_cast<float4*>(io.out_gated + ro + col) = make_float4(y[0], y[1], y[2], y[3]);
                if (io.out_gated_h) store_split4(io.out_gated_h, orow, p.cout, col, y);
            }
        }
    } else if (warp == 5) {
        // =========================== B producer (weights) ===========================
        if (lane == 0) {
            int it = 0;
            for (uint32_t km = kmask; km; km &= km - 1) {
                const int k = __ffs(km) - 1;
                for (int c = 0; c < p.nchunks; ++c, ++it) {
                    const int s = it % p.stages;
                    mbar_wait(empty(s), ((it / p.stages) & 1) ^ 1);
                    const uint32_t dst = base + (uint32_t)s * stage_bytes + 2u * A_TILE;
                    const unsigned char* src = p.wpacked + PACK_HEADER + ((size_t)k * p.nchunks + c) * (2u * b_full) + (size_t)n0 * 128u;
                    mbar_expect_tx(full_b(s), 2u * b_tile);
                    bulk_g2s(dst, src, b_tile, full_b(s));                       // hi rows n0 .. n0+ncta
                    bulk_g2s(dst + b_tile, src + b_full, b_tile, full_b(s));     // lo rows
                }
            }
        }
        __syncwarp();
    }
    // ---- teardown --------------------------------------------------------------------------------------------
    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"((uint32_t)p.tmem_cols) : "memory");
    }
}

// ---- weight packing: (kvol, cin, cout) fp32 -> [256 B header][per (k, chunk): hi tile | lo tile], each tile cout rows
// x 128 B in the K-major SWIZZLE_128B image, channels beyond cin zero-filled.  Values are W * 2^k with k chosen so
// that max|W| * 2^k lies in [8192, 16384); header[1] = 2^-k is applied to the accumulator in the epilogue. ---------
__global__ void k_weight_absmax(const float* __restrict__ w, long long n, unsigned* __restrict__ header) {
    long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    float m = 0.f;
    for (; t < n; t += (long long)gridDim.x * blockDim.x) m = fmaxf(m, fabsf(w[t]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(header, __float_as_uint(m));      // non-negative floats order like uints
}

__device__ __forceinline__ float weight_scale(unsigned max_bits) {
    const float m = __uint_as_float(max_bits);
    if (!(m > 0.f) || !isfinite(m)) return 1.f;
    int e;
    frexpf(m, &e);                         // m = f * 2^e, f in [0.5, 1)
    return ldexpf(1.f, 14 - e);            // m * scale in [8192, 16384)
}

__global__ void k_pack_weights(const float* __restrict__ w, int kvol, int cin, int cout, int nchunks, unsigned char* __restrict__ out) {
    const long long total = (long long)kvol * nchunks * cout * KC;
    long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const float scale = weight_scale(*reinterpret_cast<const unsigned*>(out));
    if (t == 0) reinterpret_cast<float*>(out)[1] = 1.0f / scale;
    if (t >= total) return;
    const int kk = (int)(t % KC);
    const int n = (int)((t / KC) % cout);
    const int c = (int)((t / ((long long)KC * cout)) % nchunks);
    const int k = (int)(t / ((long long)KC * cout * nchunks));
    const int ch = c * KC + kk;
    const float v = ch < cin ? w[((long long)k * cin + ch) * cout + n] * scale : 0.f;
    const __half hi = __float2half_rn(v);
    const __half lo = __float2half_rn(v - __half2float(hi));
    const size_t tile = (size_t)cout * 128;
    unsigned char* blob = out + PACK_HEADER + ((size_t)k * nchunks + c) * 2 * tile;
    const uint32_t off = sw128(n, kk >> 3) + (uint32_t)(kk & 7) * 2u;
    *reinterpret_cast<__half*>(blob + off) = hi;
    *reinterpret_cast<__half*>(blob + tile + off) = lo;
}

static bool shape_ok(int c1, int c2, int cout, int kvol) {
    const int ctot = c1 + c2;
    if (kvol < 1 || kvol > MAX_KVOL) return false;
    if (ctot % 16 != 0 || ctot < 16) return false;
    if (c2 > 0 && (c1 % 8 != 0 || c2 % 8 != 0)) return false;
    if (cout % 32 != 0 || cout < 32 || cout > 256) return false;
    return true;
}

static size_t smem_bytes(int cout, int stages) {
    return 1024 + (size_t)stages * (2 * A_TILE + 2 * (size_t)cout * 128) + MAX_KVOL * BM * sizeof(int) + (3 * MAX_STAGES + 4) * 8 + 16 + BM * sizeof(int);
}

}  // namespace tc

bool lb2_spconv_tc_supported(const lb2_conv_desc* d) { return tc::shape_ok(d->c1, d->c2, d->cout, d->kvol); }

extern "C" size_t lb2_packed_weight_bytes(int32_t kvol, int32_t cin, int32_t cout) {
    if (!tc::shape_ok(cin, 0, cout, kvol)) return 0;
    const int nchunks = (cin + tc::KC - 1) / tc::KC;
    return tc::PACK_HEADER + (size_t)kvol * nchunks * 2 * (size_t)cout * 128;
}

extern "C" int lb2_pack_weights(void* handle, void* stream, const float* weight, int32_t kvol, int32_t cin, int32_t cout, void* packed) {
    Lb2Handle* h = (Lb2Handle*)handle;
    LB2_REQUIRE(h, h && weight && packed, "pack_weights null");
    if (!tc::shape_ok(cin, 0, cout, kvol)) return lb2_fail(h, LB2_ERR_UNSUP, "pack_weights: shape not supported by the tensor-core variant%s", "");
    const int nchunks = (cin + tc::KC - 1) / tc::KC;
    const long long total = (long long)kvol * nchunks * cout * tc::KC;
    const long long nw = (long long)kvol * cin * cout;
    if (cudaMemsetAsync(packed, 0, tc::PACK_HEADER, (cudaStream_t)stream) != cudaSuccess) return lb2_fail(h, LB2_ERR_CUDA, "pack_weights memset%s", "");
    tc::k_weight_absmax<<<(unsigned)std::min<long long>(cdiv(nw, 256), 1024), 256, 0, (cudaStream_t)stream>>>(weight, nw, (unsigned*)packed);
    LB2_POST_LAUNCH(h, "k_weight_absmax");
    tc::k_pack_weights<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(weight, kvol, cin, cout, nchunks, (unsigned char*)packed);
    LB2_POST_LAUNCH(h, "k_pack_weights");
    return LB2_OK;
}


int lb2_spconv_tc2_launch(Lb2Handle* h, cudaStream_t s, const lb2_conv_desc* d, int step_budget);

int lb2_spconv_tc_launch(Lb2Handle* h, cudaStream_t s, const lb2_conv_desc* d, bool persistent) {
    if (persistent && h->opt[LB2_OPT_TC_PERSISTENT]) return lb2_spconv_tc2_launch(h, s, d, tc::STEP_BUDGET);
    tc::Params p;
    p.c1 = d->c1; p.c2 = d->c2; p.cout = d->cout; p.kvol = d->kvol;
    p.wpacked = (const unsigned char*)d->weight_packed;
    p.scale = d->scale; p.shift = d->shift; p.relu = d->relu;
    p.nbr = d->nbr; p.nbr_stride = d->nbr_stride; p.d_mout = d->d_mout; p.mout_cap = d->mout_cap; p.row_perm = d->row_perm; p.row_mask = d->row_mask;
    p.nchunks = (d->c1 + d->c2 + tc::KC - 1) / tc::KC;
    const int nsplit = (d->cout == 256 && h->opt[LB2_OPT_TC_NSPLIT]) ? 2 : 1;   // measured slower (A gathered twice): off by default     // 256 channels: two CTAs of 128 (drain overlap, 3 stages)
    p.ncta = d->cout / nsplit;
    int stages = tc::MAX_STAGES;
    while (stages > 1 && tc::smem_bytes(p.ncta, stages) > 227 * 1024) --stages;
    p.stages = stages;
    const int half = p.ncta <= 32 ? 32 : p.ncta <= 64 ? 64 : p.ncta <= 128 ? 128 : 256;
    p.nbuf = half <= 128 ? 2 : 1;              // ping-pong accumulators when acc0 | acc1 | total fit in 512 columns
    p.acc_stride = half;
    p.tot_col = p.nbuf * half;                 // [b*half, +cout): MMA accumulators, [tot_col, +cout): running fp32 total
    { int need = (p.nbuf + 1) * half; p.tmem_cols = 32; while (p.tmem_cols < need) p.tmem_cols <<= 1; }
    const int steps_per_offset = 3 * ((d->c1 + d->c2 + 15) / 16);
    p.group = std::max(1, tc::STEP_BUDGET / steps_per_offset);
    p.io[0] = d->io[0]; p.io[1] = d->io[d->npass > 1 ? 1 : 0];
    const size_t smem = tc::smem_bytes(p.ncta, stages);
    {
        cudaError_t e = lb2_configure_smem(h, LB2_K_TC, tc::k_spconv_tc, (int)(227 * 1024));
        if (e != cudaSuccess) return lb2_fail(h, LB2_ERR_CUDA, "k_spconv_tc smem attribute: %s", cudaGetErrorString(e));
    }
    dim3 grid(cdiv(d->mout_cap, tc::BM), d->npass, nsplit);
    tc::k_spconv_tc<<<grid, tc::THREADS, smem, s>>>(p);
    LB2_POST_LAUNCH(h, "k_spconv_tc");
    return LB2_OK;
}

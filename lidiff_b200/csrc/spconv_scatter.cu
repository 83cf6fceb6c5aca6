// K4 (variant C) — sparse convolution in gather-GEMM-scatter form on the tensor cores, for the levels
// where a voxel has only a few neighbours (L0-L2: 1.1 - 4.8 of 27).  The output-stationary variant
// (spconv_tc.cu) pays a full 128-row MMA for every (tile, offset) that has at least one pair; here the
// (in,out) pairs of a kernel offset are compacted first, so every MMA row is a real pair:
//
//   for each offset k (except the centre, which the output-stationary kernel handles as a dense GEMM):
//       Y[pairs_k, Cout] = X[pair_in] @ W[k]          tcgen05, FP16x3 split, accumulator in TMEM
//       out[pair_out] += Y                             red.global.add.v4.f32
//
// Persistent, weight-stationary: one CTA per SM walks a contiguous range of 128-pair tiles (sorted by k), so
// the packed W[k] (all Cin chunks, <= 96 KB) is loaded into shared memory once per run of equal k and every
// MMA reads B from there; only the gathered A rows stream through the stage ring.  A W[k] that does not fit
// (Cout 256: 256-384 KB) streams instead, one 64-column K chunk per slot of a two-slot ring, next to the A rows.
//   warps 0-3 A producers (gather by pair_in, fp16 hi/lo split, SWIZZLE_128B image)     warp 4 MMA issuer
//   warp 5 weight loader (cp.async.bulk)     warps 6-9 scatter epilogue (tcgen05.ld -> red.add), ping-pong TMEM
// The scattered buffer is the `pre_add` input of the centre convolution, which applies BN/ReLU/residual/gate.
//
// Stands behind ME.MinkowskiConvolution forward (ME's own GPU algorithm is this gather-GEMM-scatter),
// /root/reference/lidiff/models/minkunet.py:17-24,53-66.
#include "common.cuh"
#include <algorithm>
#include "tc_common.cuh"

namespace sc {
using namespace tc;

constexpr int THREADS = 320;
constexpr int MAX_STAGES = 4;
constexpr int MAX_KVOL = 27;
constexpr int SLAB_PITCH = 36;
constexpr int SLAB_BYTES = BM * SLAB_PITCH * 4;
constexpr int NBAR = 2 * MAX_STAGES + 8;

struct Params {
    int c1, c2, cout, kvol, nchunks, stages, npass;
    const unsigned char* wpacked;
    const int* pair_in;
    const int* pair_out;
    const int* koff;        // [kvol+1]
    const int* tile_off;    // [kvol+1]
    const float* in1[2];
    const float* in2[2];
    const void* in1_h[2];
    const void* in2_h[2];
    float* out[2];
    int acc_stride, tmem_cols;
    int stream_w;           // 1: W[k] streams through a 2-slot ring of K chunks instead of staying resident
};

__global__ void __launch_bounds__(THREADS, 1) k_spconv_scatter(const Params p) {
    extern __shared__ unsigned char smem_raw[];
    __shared__ int s_koff[MAX_KVOL + 1];
    __shared__ int s_toff[MAX_KVOL + 1];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ctot = p.c1 + p.c2;
    if (threadIdx.x <= p.kvol) { s_koff[threadIdx.x] = p.koff[threadIdx.x]; s_toff[threadIdx.x] = p.tile_off[threadIdx.x]; }

    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    unsigned char* gen = smem_raw + (base - raw);
    const uint32_t b_tile = (uint32_t)p.cout * 128u;
    const uint32_t w_bytes = (uint32_t)(p.stream_w ? 2 : p.nchunks) * 2u * b_tile;   // resident W[k] or the 2-slot chunk ring
    const uint32_t a_stage = 2u * A_TILE;
    unsigned char* a_gen = gen + w_bytes;
    const uint32_t a_base = base + w_bytes;
    float* slab = reinterpret_cast<float*>(a_gen + (size_t)p.stages * a_stage);         // [4 warps][32][SLAB_PITCH] epilogue transpose
    uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<unsigned char*>(slab) + SLAB_BYTES);
    uint32_t* misc = reinterpret_cast<uint32_t*>(bars + NBAR);
    const uint32_t bar0 = smem_u32(bars);
    auto full_a = [&](int s) { return bar0 + 8u * s; };
    auto empty_a = [&](int s) { return bar0 + 8u * (MAX_STAGES + s); };
    auto w_full = [&](int s) { return bar0 + 8u * (2 * MAX_STAGES + s); };          // slot 0 only when W[k] is resident
    auto w_empty = [&](int s) { return bar0 + 8u * (2 * MAX_STAGES + 2 + s); };
    auto acc_full = [&](int b) { return bar0 + 8u * (2 * MAX_STAGES + 4 + b); };
    auto acc_empty = [&](int b) { return bar0 + 8u * (2 * MAX_STAGES + 6 + b); };

    if (threadIdx.x == 0) {
        for (int s = 0; s < p.stages; ++s) { mbar_init(full_a(s), 128); mbar_init(empty_a(s), 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(w_full(s), 1); mbar_init(w_empty(s), 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(acc_full(b), 1); mbar_init(acc_empty(b), 128); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 4) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&misc[0])), "r"((uint32_t)p.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_d = misc[0];

    // this CTA's contiguous range of (pass, tile) work items
    const int tiles_per_pass = s_toff[p.kvol];
    const long long total = (long long)tiles_per_pass * p.npass;
    const int t_begin = (int)(total * blockIdx.x / gridDim.x), t_end = (int)(total * (blockIdx.x + 1) / gridDim.x);

    // decode work item T -> (pass, k, first pair, pair count)
    auto decode = [&](int T, int& pass, int& k, int& pbase, int& cnt) {
        pass = T / tiles_per_pass;
        const int t = T - pass * tiles_per_pass;
        k = 0;
        while (k + 1 < p.kvol && s_toff[k + 1] <= t) ++k;
        pbase = s_koff[k] + (t - s_toff[k]) * BM;
        cnt = min(BM, s_koff[k + 1] - pbase);
    };

    if (warp < 4) {
        // =========================== A producers ===========================
        const int sub = threadIdx.x & 7, rbase = threadIdx.x >> 3;
        const int D = p.stages - 1;
        int it = 0, arrived = 0;
        bool any_h = false;
        for (int T = t_begin; T < t_end; ++T) {
            int pass, k, pbase, cnt;
            decode(T, pass, k, pbase, cnt);
            const bool use_h = (p.in1_h[pass] != nullptr) && (p.c2 == 0 || p.in2_h[pass] != nullptr);
            any_h |= use_h;
            int src[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) { const int r = rbase + 16 * j; src[j] = r < cnt ? __ldg(p.pair_in + pbase + r) : -1; }
            for (int c = 0; c < p.nchunks; ++c, ++it) {
                const int s = it % p.stages;
                mbar_wait(empty_a(s), ((it / p.stages) & 1) ^ 1);
                unsigned char* a_hi = a_gen + (size_t)s * a_stage;
                const uint32_t a_hi_u = a_base + (uint32_t)s * a_stage;
                const int ch = c * KC + sub * 8;
                if (ch < ctot) {
                    const bool first = ch < p.c1;
                    const int cw = first ? p.c1 : p.c2;
                    const int co = first ? ch : ch - p.c1;
                    if (use_h) produce_a_split(reinterpret_cast<const __half*>(first ? p.in1_h[pass] : p.in2_h[pass]), cw, co, src, a_hi_u, a_hi_u + A_TILE, rbase, sub);
                    else produce_a_f32(first ? p.in1[pass] : p.in2[pass], cw, co, src, a_hi, a_hi + A_TILE, rbase, sub);
                }
                // one protocol for both paths: a cp.async group per stage (empty for the fp32 path), arrive D stages later
                cp_async_commit();
                if (it >= D) {
                    cp_async_wait_dyn(D);
                    fence_proxy_async();
                    mbar_arrive(full_a(arrived % p.stages));
                    ++arrived;
                }
            }
        }
        cp_async_wait<0>();
        fence_proxy_async();
        for (; arrived < it; ++arrived) mbar_arrive(full_a(arrived % p.stages));
        (void)any_h;
    } else if (warp == 4) {
        // =========================== MMA issuer ===========================
        if (lane == 0) {
            const uint32_t idesc = make_idesc(p.cout);
            int it = 0, j = 0, wrun = -1, cur_k = -1, cur_pass = -1;
            for (int T = t_begin; T < t_end; ++T, ++j) {
                int pass, k, pbase, cnt;
                decode(T, pass, k, pbase, cnt);
                if (!p.stream_w && (k != cur_k || pass != cur_pass)) {    // new run of equal k: its weights must have landed
                    ++wrun; cur_k = k; cur_pass = pass;
                    mbar_wait(w_full(0), wrun & 1);
                    tc_fence_after();
                }
                const int buf = j & 1;
                if (j >= 2) { mbar_wait(acc_empty(buf), ((j >> 1) - 1) & 1); tc_fence_after(); }
                const uint32_t tmem_acc = tmem_d + (uint32_t)(buf * p.acc_stride);
                for (int c = 0; c < p.nchunks; ++c, ++it) {
                    const int s = it % p.stages;
                    mbar_wait(full_a(s), (it / p.stages) & 1);
                    tc_fence_after();
                    if (p.stream_w) { mbar_wait(w_full(it & 1), (it >> 1) & 1); tc_fence_after(); }
                    const uint32_t a_hi = a_base + (uint32_t)s * a_stage, a_lo = a_hi + A_TILE;
                    const uint32_t b_hi = base + (uint32_t)(p.stream_w ? (it & 1) : c) * 2u * b_tile, b_lo = b_hi + b_tile;
                    const int ksteps = min(KC, ctot - c * KC) >> 4;
                    for (int ks = 0; ks < ksteps; ++ks) {
                        const uint64_t dah = make_desc(a_hi + ks * 32), dal = make_desc(a_lo + ks * 32);
                        const uint64_t dbh = make_desc(b_hi + ks * 32), dbl = make_desc(b_lo + ks * 32);
                        umma(tmem_acc, dah, dbh, idesc, (c | ks) ? 1u : 0u);
                        umma(tmem_acc, dal, dbh, idesc, 1);
                        umma(tmem_acc, dah, dbl, idesc, 1);
                    }
                    umma_commit(empty_a(s));
                    if (p.stream_w) umma_commit(w_empty(it & 1));
                }
                umma_commit(acc_full(buf));
                if (p.stream_w) continue;
                // last tile of this run of equal k?  then the weights may be replaced once these MMAs are done
                bool run_ends = (T + 1 == t_end);
                if (!run_ends) {
                    int p2, k2, pb2, c2;
                    decode(T + 1, p2, k2, pb2, c2);
                    run_ends = (k2 != k) || (p2 != pass);
                }
                if (run_ends) umma_commit(w_empty(0));
            }
        }
        __syncwarp();
    } else if (warp == 5) {
        // =========================== weight loader ===========================
        if (lane == 0 && p.stream_w) {
            int it = 0;
            for (int T = t_begin; T < t_end; ++T) {
                int pass, k, pbase, cnt;
                decode(T, pass, k, pbase, cnt);
                const unsigned char* src = p.wpacked + PACK_HEADER + (size_t)k * p.nchunks * 2u * b_tile;
                for (int c = 0; c < p.nchunks; ++c, ++it) {
                    const int s = it & 1;
                    if (it >= 2) mbar_wait(w_empty(s), ((it >> 1) - 1) & 1);
                    mbar_expect_tx(w_full(s), 2u * b_tile);
                    bulk_g2s(base + (uint32_t)s * 2u * b_tile, src + (size_t)c * 2u * b_tile, 2u * b_tile, w_full(s));
                }
            }
        } else if (lane == 0) {
            int wrun = -1, cur_k = -1, cur_pass = -1;
            for (int T = t_begin; T < t_end; ++T) {
                int pass, k, pbase, cnt;
                decode(T, pass, k, pbase, cnt);
                if (k == cur_k && pass == cur_pass) continue;
                ++wrun; cur_k = k; cur_pass = pass;
                if (wrun >= 1) mbar_wait(w_empty(0), (wrun - 1) & 1);
                const unsigned char* src = p.wpacked + PACK_HEADER + (size_t)k * w_bytes;
                mbar_expect_tx(w_full(0), w_bytes);
                for (int c = 0; c < p.nchunks; ++c) bulk_g2s(base + (uint32_t)c * 2u * b_tile, src + (size_t)c * 2u * b_tile, 2u * b_tile, w_full(0));
            }
        }
        __syncwarp();
    } else {
        // =========================== scatter epilogue ===========================
        // per 32-column slab: TMEM -> registers -> the warp's smem slab (transpose) -> lanes along channels, so each
        // red.global.add.v4.f32 instruction covers 4 rows x 128 contiguous bytes (full sectors) instead of 32 rows x 16 B
        const int q4 = warp & 3;
        const float out_scale = __ldg(reinterpret_cast<const float*>(p.wpacked) + 1);
        const uint32_t lane_base = (uint32_t)(q4 * 32) << 16;
        float* myslab = slab + (size_t)q4 * 32 * SLAB_PITCH;
        int j = 0;
        for (int T = t_begin; T < t_end; ++T, ++j) {
            int pass, k, pbase, cnt;
            decode(T, pass, k, pbase, cnt);
            const int r = q4 * 32 + lane;
            const int orow = r < cnt ? __ldg(p.pair_out + pbase + r) : -1;
            const int buf = j & 1;
            mbar_wait(acc_full(buf), (j >> 1) & 1);
            tc_fence_after();
            for (int c0 = 0; c0 < p.cout; c0 += 32) {
                uint32_t v[32];
                tmem_ld32(tmem_d + lane_base + (uint32_t)(buf * p.acc_stride + c0), v);
                tmem_ld_wait();
                __syncwarp();
                float* srow = myslab + lane * SLAB_PITCH;
#pragma unroll
                for (int q = 0; q < 8; ++q)
                    *reinterpret_cast<float4*>(srow + q * 4) = make_float4(__uint_as_float(v[q * 4]) * out_scale, __uint_as_float(v[q * 4 + 1]) * out_scale,
                                                                           __uint_as_float(v[q * 4 + 2]) * out_scale, __uint_as_float(v[q * 4 + 3]) * out_scale);
                __syncwarp();
#pragma unroll
                for (int e = lane; e < 256; e += 32) {
                    const int rr = e >> 3, c4 = (e & 7) * 4;
                    const int dst_row = __shfl_sync(0xffffffffu, orow, rr);
                    if (dst_row >= 0) {
                        const float4 a4 = *reinterpret_cast<const float4*>(myslab + rr * SLAB_PITCH + c4);
                        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p.out[pass] + (long long)dst_row * p.cout + c0 + c4),
                                     "f"(a4.x), "f"(a4.y), "f"(a4.z), "f"(a4.w) : "memory");
                    }
                }
            }
            tc_fence_before();
            mbar_arrive(acc_empty(buf));
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_d), "r"((uint32_t)p.tmem_cols) : "memory");
}

// ---- pair lists of a kernel map, grouped by offset ------------------------------------------------------------------
// row_mask (optional): only the pairs whose bit is set in their output row's mask (a subset of the map's pairs)
__global__ void k_pair_count(const int* __restrict__ nbr, long long nbr_stride, const int* __restrict__ d_n, int n_cap, int skip_k,
                             const unsigned* __restrict__ row_mask, int* __restrict__ cnt) {
    const int k = blockIdx.y;
    if (k == skip_k) return;
    const int n = d_n ? min(*d_n, n_cap) : n_cap;
    const int o = blockIdx.x * blockDim.x + threadIdx.x;
    const bool hit = o < n && (!row_mask || ((row_mask[o] >> k) & 1u)) && nbr[(long long)k * nbr_stride + o] >= 0;   // as k_pair_fill
    const unsigned m = __ballot_sync(0xffffffffu, hit);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(cnt + k, __popc(m));
}

__global__ void k_pair_scan(const int* __restrict__ cnt, int kvol, int* __restrict__ koff, int* __restrict__ tile_off, int* __restrict__ cursor) {
    if (threadIdx.x == 0) {
        int a = 0, t = 0;
        for (int k = 0; k < kvol; ++k) { koff[k] = a; tile_off[k] = t; cursor[k] = 0; a += cnt[k]; t += (cnt[k] + tc::BM - 1) / tc::BM; }
        koff[kvol] = a; tile_off[kvol] = t;
    }
}

__global__ void k_pair_fill(const int* __restrict__ nbr, long long nbr_stride, const int* __restrict__ d_n, int n_cap, int skip_k,
                            const unsigned* __restrict__ row_mask, const int* __restrict__ koff, int* __restrict__ cursor,
                            int* __restrict__ pair_in, int* __restrict__ pair_out) {
    const int k = blockIdx.y;
    if (k == skip_k) return;
    const int n = d_n ? min(*d_n, n_cap) : n_cap;
    const int o = blockIdx.x * blockDim.x + threadIdx.x;
    const int v = (o < n && (!row_mask || ((row_mask[o] >> k) & 1u))) ? nbr[(long long)k * nbr_stride + o] : -1;
    const unsigned m = __ballot_sync(0xffffffffu, v >= 0);
    if (!m) return;
    const int lane = threadIdx.x & 31;
    int basep = 0;
    if (lane == __ffs(m) - 1) basep = atomicAdd(cursor + k, __popc(m));
    basep = __shfl_sync(0xffffffffu, basep, __ffs(m) - 1);
    if (v >= 0) {
        const int pos = koff[k] + basep + __popc(m & ((1u << lane) - 1));
        pair_in[pos] = v;
        pair_out[pos] = o;
    }
}

__global__ void k_zero_rows(float* __restrict__ buf, const int* __restrict__ d_n, int n_cap, int c) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int n = d_n ? min(*d_n, n_cap) : n_cap;
    if (t < (long long)n * c / 4) reinterpret_cast<float4*>(buf)[t] = make_float4(0.f, 0.f, 0.f, 0.f);
}

constexpr size_t SMEM_LIMIT = 227 * 1024 - 256;        // 224 B of static smem

// w_slots: K chunks of W[k] in shared memory (all of them: resident, 2: streamed)
static size_t smem_bytes(int w_slots, int cout, int stages) {
    return 1024 + (size_t)w_slots * 2 * cout * 128 + (size_t)stages * 2 * tc::A_TILE + SLAB_BYTES + NBAR * 8 + 64;
}

static int nchunks_of(int cin) { return (cin + tc::KC - 1) / tc::KC; }

static bool stream_w(int cin, int cout) { return smem_bytes(nchunks_of(cin), cout, 2) > SMEM_LIMIT; }

static bool shape_ok(int c1, int c2, int cout, int kvol) {
    const int ctot = c1 + c2;
    if (kvol < 1 || kvol > MAX_KVOL || ctot % 16 || ctot < 16) return false;
    if (c2 > 0 && (c1 % 8 || c2 % 8)) return false;
    if (cout % 32 || cout < 32 || cout > 256) return false;
    return smem_bytes(stream_w(ctot, cout) ? 2 : nchunks_of(ctot), cout, 2) <= SMEM_LIMIT;
}

}  // namespace sc

extern "C" size_t lb2_pair_list_scratch_bytes(void) { return 2 * 32 * sizeof(int); }

extern "C" int lb2_pair_list(void* handle, void* stream, const int32_t* nbr, int64_t nbr_stride, const int32_t* d_nout,
                             int32_t nout_cap, int32_t kvol, int32_t skip_k, int32_t* pair_in, int32_t* pair_out,
                             int32_t* koff, int32_t* tile_off, void* scratch, const uint32_t* row_mask) {
    Lb2Handle* h = (Lb2Handle*)handle;
    LB2_REQUIRE(h, h && nbr && pair_in && pair_out && koff && tile_off && scratch && nout_cap > 0 && kvol >= 1 && kvol <= sc::MAX_KVOL, "pair_list");
    cudaStream_t s = (cudaStream_t)stream;
    int* cnt = (int*)scratch;
    int* cursor = cnt + 32;
    if (cudaMemsetAsync(cnt, 0, 64 * sizeof(int), s) != cudaSuccess) return lb2_fail(h, LB2_ERR_CUDA, "pair_list memset%s", "");
    dim3 grid(cdiv(nout_cap, 256), kvol);
    sc::k_pair_count<<<grid, 256, 0, s>>>(nbr, nbr_stride, d_nout, nout_cap, skip_k, row_mask, cnt);
    LB2_POST_LAUNCH(h, "k_pair_count");
    sc::k_pair_scan<<<1, 32, 0, s>>>(cnt, kvol, koff, tile_off, cursor);
    LB2_POST_LAUNCH(h, "k_pair_scan");
    sc::k_pair_fill<<<grid, 256, 0, s>>>(nbr, nbr_stride, d_nout, nout_cap, skip_k, row_mask, koff, cursor, pair_in, pair_out);
    LB2_POST_LAUNCH(h, "k_pair_fill");
    return LB2_OK;
}

extern "C" int lb2_spconv_scatter_supported(int32_t c1, int32_t c2, int32_t cout, int32_t kvol) { return sc::shape_ok(c1, c2, cout, kvol) ? 1 : 0; }

extern "C" int lb2_spconv_scatter(void* handle, void* stream, const lb2_scatter_desc* d) {
    Lb2Handle* h = (Lb2Handle*)handle;
    LB2_REQUIRE(h, h && d && d->weight_packed && d->pair_in && d->pair_out && d->koff && d->tile_off, "spconv_scatter null");
    LB2_REQUIRE(h, d->npass == 1 || d->npass == 2, "npass");
    if (!sc::shape_ok(d->c1, d->c2, d->cout, d->kvol)) return lb2_fail(h, LB2_ERR_UNSUP, "spconv_scatter: shape not supported%s", "");
    cudaStream_t s = (cudaStream_t)stream;
    sc::Params p;
    p.c1 = d->c1; p.c2 = d->c2; p.cout = d->cout; p.kvol = d->kvol; p.npass = d->npass;
    p.nchunks = (d->c1 + d->c2 + tc::KC - 1) / tc::KC;
    p.wpacked = (const unsigned char*)d->weight_packed;
    p.pair_in = d->pair_in; p.pair_out = d->pair_out; p.koff = d->koff; p.tile_off = d->tile_off;
    for (int i = 0; i < 2; ++i) {
        const int j = d->npass > 1 ? i : 0;
        const bool has_h = d->in1_h[j] && (d->c2 == 0 || d->in2_h[j]);        // the producers read the companions when all are given
        const bool has_f = d->in1[j] && (d->c2 == 0 || d->in2[j]);
        LB2_REQUIRE(h, (has_h || has_f) && d->out[j] && (d->c2 > 0 || (!d->in2[j] && !d->in2_h[j])), "spconv_scatter io");
        p.in1[i] = d->in1[j]; p.in2[i] = d->in2[j]; p.out[i] = d->out[j];
        p.in1_h[i] = d->in1_h[j]; p.in2_h[i] = d->in2_h[j];
    }
    p.stream_w = sc::stream_w(d->c1 + d->c2, d->cout) ? 1 : 0;
    const int w_slots = p.stream_w ? 2 : p.nchunks;
    int stages = sc::MAX_STAGES;
    while (stages > 2 && sc::smem_bytes(w_slots, d->cout, stages) > sc::SMEM_LIMIT) --stages;
    p.stages = stages;
    const int half = d->cout <= 32 ? 32 : d->cout <= 64 ? 64 : d->cout <= 128 ? 128 : 256;
    p.acc_stride = half; p.tmem_cols = 2 * half;
    if (d->zero_rows_cap > 0) {        // clear the rows the scatter adds into
        for (int i = 0; i < d->npass; ++i) {
            sc::k_zero_rows<<<cdiv((long long)d->zero_rows_cap * d->cout / 4, 256), 256, 0, s>>>(d->out[i], d->d_zero_rows, d->zero_rows_cap, d->cout);
            LB2_POST_LAUNCH(h, "k_zero_rows");
        }
    }
    {
        cudaError_t e = lb2_configure_smem(h, LB2_K_SCATTER, sc::k_spconv_scatter, (int)sc::SMEM_LIMIT);
        if (e != cudaSuccess) return lb2_fail(h, LB2_ERR_CUDA, "k_spconv_scatter smem attribute: %s", cudaGetErrorString(e));
    }
    sc::k_spconv_scatter<<<h->num_sms, sc::THREADS, sc::smem_bytes(w_slots, d->cout, stages), s>>>(p);
    LB2_POST_LAUNCH(h, "k_spconv_scatter");
    return LB2_OK;
}

// K1/K2/K3 — GPU hash-grid coordinate manager: quantise, voxelise (unique rows in first-occurrence
// order), strided coordinate maps, kernel maps (neighbour tables).  Integer work, HBM/L2 bound:
// int4 coalesced coordinate loads, one 8-byte CAS per insert, open addressing in an L2-resident table.
//
// Stands behind ME.TensorField.sparse() / ME coordinate manager as used at
// /root/reference/lidiff/tools/diff_completion_pipeline.py:68-84,149 and lidiff/models/minkunet.py:17-24,36-42,135.
#include "common.cuh"
#include <stdlib.h>
#include <limits.h>
#include <algorithm>

// ---------------------------------------------------------------------------------------------------
// handle
// ---------------------------------------------------------------------------------------------------
extern "C" int lb2_version(void) { return 100; }

extern "C" int lb2_create(int device, void** handle) {
    if (!handle) return LB2_ERR_ARG;
    *handle = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) return LB2_ERR_CUDA;
    if (cudaSetDevice(device) != cudaSuccess) return LB2_ERR_CUDA;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return LB2_ERR_CUDA;
    if (prop.major != 10) return LB2_ERR_UNSUP;          // sm_100a binary only
    Lb2Handle* h = new Lb2Handle();
    h->device = device; h->num_sms = prop.multiProcessorCount; h->launches = 0; h->err[0] = 0; h->configured = 0;
    {
        auto env = [](const char* name, int dflt) { const char* e = getenv(name); return (e && e[0]) ? atoi(e) : dflt; };
        h->opt[LB2_OPT_TC_PAIR] = env("LB2_TC_PAIR", 2);
        h->opt[LB2_OPT_TC_N256] = env("LB2_TC_N256", 1);
        h->opt[LB2_OPT_TC_SMALL] = env("LB2_TC_SMALL", 1);
        h->opt[LB2_OPT_TC_PERSISTENT] = env("LB2_TC_PERSISTENT", 1);
        const char* lag = getenv("LB2_TC_LAG");
        h->opt[LB2_OPT_TC_FULL_LAG] = (lag && lag[0] == 'f') ? 1 : 0;
        h->opt[LB2_OPT_TC_NSPLIT] = env("LB2_TC_NSPLIT", 0);
    }
    if (cudaMalloc(&h->d_status, sizeof(int32_t)) != cudaSuccess) { delete h; return LB2_ERR_CUDA; }
    cudaMemset(h->d_status, 0, sizeof(int32_t));
    *handle = h;
    return LB2_OK;
}

extern "C" void lb2_destroy(void* handle) {
    Lb2Handle* h = (Lb2Handle*)handle;
    if (!h) return;
    cudaFree(h->d_status);
    delete h;
}

extern "C" int lb2_set_option(void* handle, int option, int value) {
    Lb2Handle* h = (Lb2Handle*)handle;
    LB2_REQUIRE(h, h && option >= 0 && option < LB2_OPT_COUNT, "set_option");
    h->opt[option] = value;
    return LB2_OK;
}

extern "C" int lb2_get_option(void* handle, int option) {
    Lb2Handle* h = (Lb2Handle*)handle;
    if (!h || option < 0 || option >= LB2_OPT_COUNT) return LB2_ERR_ARG;
    return h->opt[option];
}

extern "C" const char* lb2_last_error(void* handle) {
    return handle ? ((Lb2Handle*)handle)->err : "null handle";
}

extern "C" int64_t lb2_launch_count(void* handle) { return handle ? ((Lb2Handle*)handle)->launches : -1; }

// synchronising read-and-clear of the device status word (bit0: coordinate outside the key range)
extern "C" int lb2_read_status(void* handle, void* stream) {
    Lb2Handle* h = (Lb2Handle*)handle;
    if (!h) return LB2_ERR_ARG;
    int32_t v = 0;
    cudaStream_t s = (cudaStream_t)stream;
    if (cudaMemcpyAsync(&v, h->d_status, sizeof(v), cudaMemcpyDeviceToHost, s) != cudaSuccess) return LB2_ERR_CUDA;
    if (cudaMemsetAsync(h->d_status, 0, sizeof(v), s) != cudaSuccess) return LB2_ERR_CUDA;
    if (cudaStreamSynchronize(s) != cudaSuccess) return LB2_ERR_CUDA;
    return v;
}

// ---------------------------------------------------------------------------------------------------
// quantise: coord = rint(x / res)   (round-half-even == torch.round)
// ---------------------------------------------------------------------------------------------------
__global__ void k_quantize(const float* __restrict__ x, long long n, float res, float inv_res, int div_mode,
                           float* __restrict__ out) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float v = x[i];
    float q = div_mode == 0 ? __fdiv_rn(v, res) : __fmul_rn(v, inv_res);
    out[i] = rintf(q);
}

extern "C" int lb2_quantize(void* handle, void* stream, const float* x, int64_t n_elem, float resolution,
                            int div_mode, float* out_coord) {
    Lb2Handle* h = (Lb2Handle*)handle;
    LB2_REQUIRE(h, h && x && out_coord && resolution > 0.f, "quantize");
    if (n_elem == 0) return LB2_OK;
    float inv = 1.0f / resolution;       // fp32 reciprocal, as PyTorch's CUDA scalar-divide does
    k_quantize<<<cdiv(n_elem, 256), 256, 0, (cudaStream_t)stream>>>(x, n_elem, resolution, inv, div_mode, out_coord);
    LB2_POST_LAUNCH(h, "k_quantize");
    return LB2_OK;
}

// ---------------------------------------------------------------------------------------------------
// unique rows in first-occurrence order
// ---------------------------------------------------------------------------------------------------
#define SCAN_THREADS 512
#define SCAN_ITEMS   4
#define SCAN_TILE    (SCAN_THREADS * SCAN_ITEMS)

struct UniqueScratch {     // carved out of the caller's scratch buffer
    int* slot_of;          // [n_cap]
    int* rank;             // [n_cap]
    int* bsum;             // [SCAN_TILE]
};

extern "C" size_t lb2_unique_scratch_bytes(int64_t n_cap) {
    size_t a = ((size_t)n_cap * sizeof(int) + 255) / 256 * 256;
    return 2 * a + SCAN_TILE * sizeof(int) + 256;
}

static UniqueScratch carve(void* scratch, int64_t n_cap) {
    size_t a = ((size_t)n_cap * sizeof(int) + 255) / 256 * 256;
    char* p = (char*)scratch;
    UniqueScratch s;
    s.slot_of = (int*)p; s.rank = (int*)(p + a); s.bsum = (int*)(p + 2 * a);
    return s;
}

__global__ void k_grid_clear(unsigned long long* keys, int* vals, int cap) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < cap) { keys[i] = LB2_KEY_EMPTY; vals[i] = INT_MAX; vals[cap + i] = -1; }
}

__device__ __forceinline__ int4 load_row(const float* __restrict__ in_f, const int* __restrict__ in_i, int i, int ts) {
    int4 c;
    if (in_f) {
        float4 f = __ldg(reinterpret_cast<const float4*>(in_f) + i);
        c = make_int4((int)floorf(f.x), (int)floorf(f.y), (int)floorf(f.z), (int)floorf(f.w));
    } else {
        c = __ldg(reinterpret_cast<const int4*>(in_i) + i);
    }
    if (ts > 0) { c.y = floor_to_multiple(c.y, ts); c.z = floor_to_multiple(c.z, ts); c.w = floor_to_multiple(c.w, ts); }
    return c;
}

__global__ void k_grid_insert(const float* __restrict__ in_f, const int* __restrict__ in_i,
                              const int* __restrict__ d_n, int n_cap, int ts,
                              unsigned long long* keys, int* vals, unsigned mask,
                              int* __restrict__ slot_of, int* status) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int n = d_n ? min(*d_n, n_cap) : n_cap;
    if (i >= n) return;
    int4 c = load_row(in_f, in_i, i, ts);
    unsigned long long key;
    if (!lb2_pack_key(c.x, c.y, c.z, c.w, key)) atomicOr(status, 1);
    unsigned slot = lb2_hash(key) & mask;
    while (true) {
        unsigned long long prev = atomicCAS(keys + slot, (unsigned long long)LB2_KEY_EMPTY, key);
        if (prev == LB2_KEY_EMPTY || prev == key) break;
        slot = (slot + 1) & mask;
    }
    atomicMin(vals + slot, i);          // first occurrence wins
    slot_of[i] = (int)slot;
}

// block-level exclusive scan of the "is first occurrence" flags
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_local(const int* __restrict__ slot_of, const int* __restrict__ vals,
                                                             const int* __restrict__ d_n, int n_cap,
                                                             int* __restrict__ rank, int* __restrict__ bsum) {
    __shared__ int warp_tot[SCAN_THREADS / 32];
    int n = d_n ? min(*d_n, n_cap) : n_cap;
    int base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
    int f[SCAN_ITEMS], tsum = 0;
#pragma unroll
    for (int j = 0; j < SCAN_ITEMS; ++j) {
        int i = base + j;
        f[j] = (i < n) ? (vals[slot_of[i]] == i) : 0;
        tsum += f[j];
    }
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int incl = tsum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { int v = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += v; }
    if (lane == 31) warp_tot[w] = incl;
    __syncthreads();
    if (w == 0) {
        int v = (lane < SCAN_THREADS / 32) ? warp_tot[lane] : 0, inc2 = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { int u = __shfl_up_sync(0xffffffffu, inc2, d); if (lane >= d) inc2 += u; }
        if (lane < SCAN_THREADS / 32) warp_tot[lane] = inc2 - v;      // exclusive warp offsets
        if (lane == SCAN_THREADS / 32 - 1) bsum[blockIdx.x] = inc2;   // block total
    }
    __syncthreads();
    int excl = warp_tot[w] + incl - tsum;
#pragma unroll
    for (int j = 0; j < SCAN_ITEMS; ++j) {
        int i = base + j;
        if (i < n) rank[i] = f[j] ? excl : -1;     // -1: not a first occurrence
        excl += f[j];
    }
}

// single block: exclusive scan of up to SCAN_TILE block totals; writes the grand total
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_bsum(int* __restrict__ bsum, int nblocks, int* __restrict__ d_total) {
    __shared__ int warp_tot[SCAN_THREADS / 32];
    int base = threadIdx.x * SCAN_ITEMS;
    int v[SCAN_ITEMS], tsum = 0;
#pragma unroll
    for (int j = 0; j < SCAN_ITEMS; ++j) { v[j] = (base + j < nblocks) ? bsum[base + j] : 0; tsum += v[j]; }
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int incl = tsum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { int u = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += u; }
    if (lane == 31) warp_tot[w] = incl;
    __syncthreads();
    if (w == 0) {
        int x = (lane < SCAN_THREADS / 32) ? warp_tot[lane] : 0, inc2 = x;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { int u = __shfl_up_sync(0xffffffffu, inc2, d); if (lane >= d) inc2 += u; }
        if (lane < SCAN_THREADS / 32) warp_tot[lane] = inc2 - x;
        if (lane == SCAN_THREADS / 32 - 1) *d_total = inc2;
    }
    __syncthreads();
    int excl = warp_tot[w] + incl - tsum;
#pragma unroll
    for (int j = 0; j < SCAN_ITEMS; ++j) { if (base + j < nblocks) bsum[base + j] = excl; excl += v[j]; }
}

// winners publish their row id and coordinates
__global__ void k_unique_emit(const float* __restrict__ in_f, const int* __restrict__ in_i,
                              const int* __restrict__ d_n, int n_cap, int ts,
                              const int* __restrict__ slot_of, const int* __restrict__ rank,
                              const int* __restrict__ bsum, int* __restrict__ vals, int cap,
                              int4* __restrict__ out_coords) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int n = d_n ? min(*d_n, n_cap) : n_cap;
    if (i >= n) return;
    int r = rank[i];
    if (r < 0) return;
    r += bsum[i / SCAN_TILE];
    vals[cap + slot_of[i]] = r;
    out_coords[r] = load_row(in_f, in_i, i, ts);
}

__global__ void k_unique_inverse(const int* __restrict__ d_n, int n_cap, const int* __restrict__ slot_of,
                                 const int* __restrict__ vals, int cap, int* __restrict__ inverse) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int n = d_n ? min(*d_n, n_cap) : n_cap;
    if (i < n) inverse[i] = vals[cap + slot_of[i]];
}

extern "C" int lb2_unique_build(void* handle, void* stream, const float* in_f, const int32_t* in_i,
                                const int32_t* d_nin, int32_t n_cap, int32_t ts_floor, lb2_grid grid,
                                int32_t* out_coords, int32_t* inverse, int32_t* d_nout, void* scratch) {
    Lb2Handle* h = (Lb2Handle*)handle;
    LB2_REQUIRE(h, h != nullptr, "handle");
    LB2_REQUIRE(h, (in_f != nullptr) != (in_i != nullptr), "exactly one of in_f / in_i");
    LB2_REQUIRE(h, grid.keys && grid.vals && out_coords && d_nout && scratch, "null buffer");
    LB2_REQUIRE(h, n_cap > 0 && n_cap <= SCAN_TILE * SCAN_TILE, "n_cap out of range (max 4M rows)");
    LB2_REQUIRE(h, grid.cap_table >= 2 && (grid.cap_table & (grid.cap_table - 1)) == 0, "cap_table must be a power of two");
    LB2_REQUIRE(h, (long long)grid.cap_table >= 2LL * n_cap, "cap_table must be >= 2 * n_cap");
    LB2_REQUIRE(h, ts_floor >= 0, "ts_floor");
    cudaStream_t s = (cudaStream_t)stream;
    UniqueScratch sc = carve(scratch, n_cap);
    unsigned long long* keys = (unsigned long long*)grid.keys;
    int cap = grid.cap_table;
    unsigned mask = (unsigned)cap - 1u;
    int nblk = (int)cdiv(n_cap, SCAN_TILE);

    k_grid_clear<<<cdiv(cap, 256), 256, 0, s>>>(keys, grid.vals, cap);
    LB2_POST_LAUNCH(h, "k_grid_clear");
    k_grid_insert<<<cdiv(n_cap, 256), 256, 0, s>>>(in_f, in_i, d_nin, n_cap, ts_floor, keys, grid.vals, mask, sc.slot_of, h->d_status);
    LB2_POST_LAUNCH(h, "k_grid_insert");
    k_scan_local<<<nblk, SCAN_THREADS, 0, s>>>(sc.slot_of, grid.vals, d_nin, n_cap, sc.rank, sc.bsum);
    LB2_POST_LAUNCH(h, "k_scan_local");
    k_scan_bsum<<<1, SCAN_THREADS, 0, s>>>(sc.bsum, nblk, d_nout);
    LB2_POST_LAUNCH(h, "k_scan_bsum");
    k_unique_emit<<<cdiv(n_cap, 256), 256, 0, s>>>(in_f, in_i, d_nin, n_cap, ts_floor, sc.slot_of, sc.rank, sc.bsum,
                                                  grid.vals, cap, (int4*)out_coords);
    LB2_POST_LAUNCH(h, "k_unique_emit");
    if (inverse) {
        k_unique_inverse<<<cdiv(n_cap, 256), 256, 0, s>>>(d_nin, n_cap, sc.slot_of, grid.vals, cap, inverse);
        LB2_POST_LAUNCH(h, "k_unique_inverse");
    }
    return LB2_OK;
}

// ---------------------------------------------------------------------------------------------------
// voxel mean features
// ---------------------------------------------------------------------------------------------------
__global__ void k_voxel_accum(const float* __restrict__ feats, const int* __restrict__ inverse, int n, int c,
                              float* __restrict__ out, int* __restrict__ counts) {
    long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)n * c) return;
    int i = (int)(t / c), j = (int)(t % c);
    int r = inverse[i];
    atomicAdd(out + (long long)r * c + j, feats[t]);
    if (j == 0) atomicAdd(counts + r, 1);
}

__global__ void k_voxel_div(float* __restrict__ out, const int* __restrict__ counts, const int* __restrict__ d_m,
                            int m_cap, int c) {
    long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int m = d_m ? min(*d_m, m_cap) : m_cap;
    if (t >= (long long)m * c) return;
    out[t] = __fdiv_rn(out[t], (float)counts[t / c]);
}

extern "C" int lb2_voxel_mean(void* handle, void* stream, const float* feats, const int32_t* inverse, int32_t n,
                              int32_t c, const int32_t* d_m, int32_t m_cap, float* out, int32_t* counts) {
    Lb2Handle* h = (Lb2Handle*)handle;
    LB2_REQUIRE(h, h && feats && inverse && out && counts && n > 0 && c > 0 && m_cap > 0, "voxel_mean");
    cudaStream_t s = (cudaStream_t)stream;
    if (cudaMemsetAsync(out, 0, (size_t)m_cap * c * sizeof(float), s) != cudaSuccess ||
        cudaMemsetAsync(counts, 0, (size_t)m_cap * sizeof(int), s) != cudaSuccess)
        return lb2_fail(h, LB2_ERR_CUDA, "voxel_mean memset%s", "");
    k_voxel_accum<<<cdiv((long long)n * c, 256), 256, 0, s>>>(feats, inverse, n, c, out, counts);
    LB2_POST_LAUNCH(h, "k_voxel_accum");
    k_voxel_div<<<cdiv((long long)m_cap * c, 256), 256, 0, s>>>(out, counts, d_m, m_cap, c);
    LB2_POST_LAUNCH(h, "k_voxel_div");
    return LB2_OK;
}

// ---------------------------------------------------------------------------------------------------
// kernel map: neighbour table nbr[k][o]
// ---------------------------------------------------------------------------------------------------
// one thread per output row walks the K offsets: the row's coordinate is read once, its neighbour mask is built in a
// register, the K table writes stay coalesced across the warp for each k, and the K hash probes of a thread are
// independent loads in flight together
template <int KS>
__global__ void __launch_bounds__(128) k_kernel_map(const unsigned long long* __restrict__ keys, const int* __restrict__ rows, unsigned mask,
                                                    const int4* __restrict__ out_coords, const int* __restrict__ d_n, int n_cap,
                                                    int step, int* __restrict__ nbr, long long nbr_stride,
                                                    unsigned long long* __restrict__ pair_count, unsigned* __restrict__ row_mask) {
    constexpr int KV = KS * KS * KS;
    const int o = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = d_n ? min(*d_n, n_cap) : n_cap;
    unsigned found = 0;
    if (o < n) {
        const int4 c = __ldg(out_coords + o);
        constexpr int cen = (KS & 1) ? KS / 2 : 0;
        int res[KV];
        unsigned long long key[KV], got[KV];
        unsigned slot[KV];
#pragma unroll
        for (int k = 0; k < KV; ++k) {                                  // first probe of every offset: KV independent loads
            const int kx = k % KS, ky = (k / KS) % KS, kz = k / (KS * KS);
            const int x = c.y + (kx - cen) * step, y = c.z + (ky - cen) * step, z = c.w + (kz - cen) * step;
            const bool ok = lb2_pack_key(c.x, x, y, z, key[k]);
            slot[k] = ok ? (lb2_hash(key[k]) & mask) : 0u;
            got[k] = ok ? __ldg(keys + slot[k]) : LB2_KEY_EMPTY;
            if (!ok) key[k] = ~LB2_KEY_EMPTY;                           // differs from the EMPTY it "read": a miss below
        }
#pragma unroll
        for (int k = 0; k < KV; ++k) {
            if (got[k] == key[k]) res[k] = __ldg(rows + slot[k]);
            else if (got[k] == LB2_KEY_EMPTY) res[k] = -1;
            else {                                                      // collision on the first slot: continue the linear probe
                unsigned sl = (slot[k] + 1) & mask;
                res[k] = -1;
                while (true) {
                    const unsigned long long kk = __ldg(keys + sl);
                    if (kk == key[k]) { res[k] = __ldg(rows + sl); break; }
                    if (kk == LB2_KEY_EMPTY) break;
                    sl = (sl + 1) & mask;
                }
            }
        }
#pragma unroll
        for (int k = 0; k < KV; ++k) {
            nbr[(long long)k * nbr_stride + o] = res[k];
            if (res[k] >= 0) found |= 1u << k;
        }
    } else if (o < n_cap) {
#pragma unroll
        for (int k = 0; k < KV; ++k) nbr[(long long)k * nbr_stride + o] = -1;
    }
    if (row_mask && o < n_cap) row_mask[o] = found;
    if (pair_count) {        // algorithmic work counter for the roofline: one atomic per warp
        int cnt = __popc(found);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, d);
        if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(pair_count, (unsigned long long)cnt);
    }
}

extern "C" int lb2_kernel_map(void* handle, void* stream, lb2_grid grid_in, const int32_t* out_coords,
                              const int32_t* d_nout, int32_t nout_cap, int32_t ks, int32_t step,
                              int32_t* nbr, int64_t nbr_stride, uint64_t* pair_count, uint32_t* row_mask) {
    Lb2Handle* h = (Lb2Handle*)handle;
    LB2_REQUIRE(h, h && grid_in.keys && grid_in.vals && out_coords && nbr, "kernel_map null");
    LB2_REQUIRE(h, ks >= 1 && ks <= 3 && step != 0 && nout_cap > 0 && nbr_stride >= nout_cap, "kernel_map args");
    const unsigned long long* gk = (const unsigned long long*)grid_in.keys;
    const int* gr = grid_in.vals + grid_in.cap_table;
    const unsigned gm = (unsigned)grid_in.cap_table - 1u;
    const unsigned blocks = cdiv(nout_cap, 128);
    cudaStream_t s = (cudaStream_t)stream;
    if (ks == 3) k_kernel_map<3><<<blocks, 128, 0, s>>>(gk, gr, gm, (const int4*)out_coords, d_nout, nout_cap, step, nbr, nbr_stride, (unsigned long long*)pair_count, row_mask);
    else if (ks == 2) k_kernel_map<2><<<blocks, 128, 0, s>>>(gk, gr, gm, (const int4*)out_coords, d_nout, nout_cap, step, nbr, nbr_stride, (unsigned long long*)pair_count, row_mask);
    else k_kernel_map<1><<<blocks, 128, 0, s>>>(gk, gr, gm, (const int4*)out_coords, d_nout, nout_cap, step, nbr, nbr_stride, (unsigned long long*)pair_count, row_mask);
    LB2_POST_LAUNCH(h, "k_kernel_map");
    return LB2_OK;
}

// ---------------------------------------------------------------------------------------------------
// 3^3 map of a coordinate set onto itself (stride-1 convolutions: most of the maps of a U-Net pass).  The pair set is symmetric — row j
// sits at offset k of row o exactly when o sits at offset 26 - k of j — so every thread probes the 13 offsets below the centre only and
// writes both directions; the centre is the row itself.  Half the hash probes of k_kernel_map<3>, same table bit for bit.
// The offsets above the centre and the row masks are pre-set (-1 / 0) by the launcher.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_kernel_map_self(const unsigned long long* __restrict__ keys, const int* __restrict__ rows, unsigned mask,
                                                         const int4* __restrict__ coords, const int* __restrict__ d_n, int n_cap, int step,
                                                         int* __restrict__ nbr, long long nbr_stride,
                                                         unsigned long long* __restrict__ pair_count, unsigned* __restrict__ row_mask) {
    constexpr int HALF = 13;
    const int o = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = d_n ? min(*d_n, n_cap) : n_cap;
    unsigned found = 0;
    if (o < n) {
        const int4 c = __ldg(coords + o);
        int res[HALF];
        unsigned long long key[HALF], got[HALF];
        unsigned slot[HALF];
#pragma unroll
        for (int k = 0; k < HALF; ++k) {                                // first probe of every offset: independent loads
            const int kx = k % 3, ky = (k / 3) % 3, kz = k / 9;
            const int x = c.y + (kx - 1) * step, y = c.z + (ky - 1) * step, z = c.w + (kz - 1) * step;
            const bool ok = lb2_pack_key(c.x, x, y, z, key[k]);
            slot[k] = ok ? (lb2_hash(key[k]) & mask) : 0u;
            got[k] = ok ? __ldg(keys + slot[k]) : LB2_KEY_EMPTY;
            if (!ok) key[k] = ~LB2_KEY_EMPTY;
        }
#pragma unroll
        for (int k = 0; k < HALF; ++k) {
            if (got[k] == key[k]) res[k] = __ldg(rows + slot[k]);
            else if (got[k] == LB2_KEY_EMPTY) res[k] = -1;
            else {                                                      // collision on the first slot: continue the linear probe
                unsigned sl = (slot[k] + 1) & mask;
                res[k] = -1;
                while (true) {
                    const unsigned long long kk = __ldg(keys + sl);
                    if (kk == key[k]) { res[k] = __ldg(rows + sl); break; }
                    if (kk == LB2_KEY_EMPTY) break;
                    sl = (sl + 1) & mask;
                }
            }
        }
#pragma unroll
        for (int k = 0; k < HALF; ++k) {
            nbr[(long long)k * nbr_stride + o] = res[k];
            if (res[k] >= 0) {
                found |= 1u << k;
                nbr[(long long)(26 - k) * nbr_stride + res[k]] = o;     // the mirrored pair: nobody else writes this entry
                if (row_mask) atomicOr(row_mask + res[k], 1u << (26 - k));
            }
        }
        nbr[(long long)HALF * nbr_stride + o] = o;
        if (row_mask) atomicOr(row_mask + o, found | (1u << HALF));
    } else if (o < n_cap) {
#pragma unroll
        for (int k = 0; k <= HALF; ++k) nbr[(long long)k * nbr_stride + o] = -1;
    }
    if (pair_count) {        // algorithmic work counter for the roofline: one atomic per warp
        int cnt = (o < n) ? 2 * __popc(found) + 1 : 0;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, d);
        if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(pair_count, (unsigned long long)cnt);
    }
}

extern "C" int lb2_kernel_map_self(void* handle, void* stream, lb2_grid grid, const int32_t* coords, const int32_t* d_n, int32_t n_cap,
                                   int32_t step, int32_t* nbr, int64_t nbr_stride, uint64_t* pair_count, uint32_t* row_mask) {
    Lb2Handle* h = (Lb2Handle*)handle;
    LB2_REQUIRE(h, h && grid.keys && grid.vals && coords && nbr, "kernel_map_self null");
    LB2_REQUIRE(h, step > 0 && n_cap > 0 && nbr_stride >= n_cap, "kernel_map_self args");
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(nbr + 14 * nbr_stride, 0xff, (size_t)13 * nbr_stride * sizeof(int32_t), s);
    if (e == cudaSuccess && row_mask) e = cudaMemsetAsync(row_mask, 0, (size_t)n_cap * sizeof(uint32_t), s);
    if (e != cudaSuccess) return lb2_fail(h, LB2_ERR_CUDA, "kernel_map_self memset: %s", cudaGetErrorString(e));
    k_kernel_map_self<<<cdiv(n_cap, 128), 128, 0, s>>>((const unsigned long long*)grid.keys, grid.vals + grid.cap_table, (unsigned)grid.cap_table - 1u,
                                                       (const int4*)coords, d_n, n_cap, step, nbr, nbr_stride, (unsigned long long*)pair_count, row_mask);
    LB2_POST_LAUNCH(h, "k_kernel_map_self");
    return LB2_OK;
}

// ---------------------------------------------------------------------------------------------------
// row order: sort of the output rows by their neighbour mask, so that the 128-row tiles of the convolution
// kernels are (nearly) homogeneous in which kernel offsets are populated and skip the rest.
//   kvol <= 8 : one counting-sort pass on the 8-bit mask itself.
//   kvol == 27: stable LSD radix sort (3 passes of 9 bits) on the 27-bit key
//                  [ 2 or more off-centre neighbours ? 1 : 0 | mask without the (always set) centre bit ]
//               i.e. centre-only rows first, then the rows with exactly one neighbour grouped by it (tiles that need
//               two offsets), then everything else in mask order.  Measured on the bench trajectory the issued
//               (tile, offset) slots drop by 10-30 % on the levels with 3-14 neighbours per row against the
//               previous 55-class bucketing (profiles/r01_row_order_waste.txt).
// The order inside a group of equal keys is irrelevant for the results (each output row is computed independently).
// ---------------------------------------------------------------------------------------------------
#define RO_BINS 256
#define RS_BITS 9
#define RS_BINS (1 << RS_BITS)
#define RS_CHUNK 2048                       // rows per block and pass
#define RS_WARPS 8                          // 256 consecutive rows per warp

__device__ __forceinline__ unsigned ro_key27(unsigned mask) {
    const unsigned extras = mask & ~(1u << 13);
    const unsigned k26 = ((mask >> 14) << 13) | (mask & 0x1fffu);
    return ((__popc(extras) >= 2) ? (1u << 26) : 0u) | k26;
}

// 27-bit Morton code of a row's voxel coordinate (9 bits per axis of coord >> shift; wraps beyond 512 cells: locality hint only)
__device__ __forceinline__ unsigned ro_part9(unsigned v) {           // 9 bits -> every third bit
    v &= 0x1ffu;
    v = (v | (v << 16)) & 0x030000ffu;
    v = (v | (v << 8)) & 0x0300f00fu;
    v = (v | (v << 4)) & 0x030c30c3u;
    v = (v | (v << 2)) & 0x09249249u;
    return v;
}
__device__ __forceinline__ unsigned ro_morton(const int4 c, int shift) {
    return ro_part9((unsigned)(c.y >> shift)) | (ro_part9((unsigned)(c.z >> shift)) << 1) | (ro_part9((unsigned)(c.w >> shift)) << 2);
}

// where a pass takes its sort key from
struct RsSrc {
    const unsigned* keys;        // mode 0: keys[i] (ping-pong buffer of the previous pass)
    const unsigned* mask;        // mode 1: ro_key27(mask[i])            (first pass of a mask-only sort, value = i)
                                 // mode 3: ro_key27(mask[vals_in[i]])   (first mask pass behind the Morton passes)
    const int4* coords;          // mode 2: ro_morton(coords[i])          (first Morton pass, value = i)
    const int* vals;             // values of the previous pass or NULL (value = i)
    const unsigned long long* keys64;   // mode 4: keys64[vals ? vals[i] : i] >> key_shift   (64-bit keys, lb2_sort_keys64)
    int mode, coord_shift, key_shift;
};
__device__ __forceinline__ unsigned rs_key(const RsSrc& s, int i) {
    switch (s.mode) {
        case 0: return s.keys[i];
        case 1: return ro_key27(s.mask[i]);
        case 2: return ro_morton(s.coords[i], s.coord_shift);
        case 4: return (unsigned)(s.keys64[s.vals ? s.vals[i] : i] >> s.key_shift);
        default: return ro_key27(s.mask[s.vals[i]]);
    }
}

__global__ void __launch_bounds__(256) k_rs_hist(const RsSrc src, const int* __restrict__ d_n, int n_cap, int shift, int* __restrict__ hist,
                                                 int* __restrict__ total) {
    __shared__ int sh[RS_BINS];
    for (int i = threadIdx.x; i < RS_BINS; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    const int n = d_n ? min(*d_n, n_cap) : n_cap;
    const int lo = blockIdx.x * RS_CHUNK, hi = min(lo + RS_CHUNK, n);
    for (int i = lo + threadIdx.x; i < hi; i += blockDim.x) atomicAdd(&sh[(rs_key(src, i) >> shift) & (RS_BINS - 1)], 1);
    __syncthreads();
    for (int i = threadIdx.x; i < RS_BINS; i += blockDim.x) {
        hist[blockIdx.x * RS_BINS + i] = sh[i];                                                        // block-major: coalesced both ways
        if (sh[i]) atomicAdd(total + i, sh[i]);
    }
}

// stable scatter: warp w of block b owns rows [b*2048 + w*256, +256) and walks them in order, 32 at a time
__global__ void __launch_bounds__(32 * RS_WARPS) k_rs_scatter(const RsSrc src, const int* __restrict__ d_n, int n_cap,
                                                              int shift, const int* __restrict__ hist, const int* __restrict__ total,
                                                              unsigned* __restrict__ keys_out, int* __restrict__ vals_out) {
    const int* __restrict__ vals_in = src.vals;
    __shared__ int cnt[RS_WARPS][RS_BINS];
    __shared__ int first[RS_BINS];                 // global position of the first row of (bin, this block)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < RS_WARPS * RS_BINS; i += blockDim.x) (&cnt[0][0])[i] = 0;
    {   // exclusive scan of the bin totals (2 bins per thread) + the rows of the same bin in the blocks before this one
        const int t = threadIdx.x;
        const int t0 = total[2 * t], t1 = total[2 * t + 1];
        first[t] = t0 + t1;                        // pair sums, scanned in place over the first 256 entries
        __syncthreads();
        for (int d = 1; d < RS_BINS / 2; d <<= 1) {
            const int u = (t >= d) ? first[t - d] : 0;
            __syncthreads();
            first[t] += u;
            __syncthreads();
        }
        const int excl = first[t] - (t0 + t1);
        int p0 = 0, p1 = 0;
#pragma unroll 8
        for (int b = 0; b < (int)blockIdx.x; ++b) {
            const int2 v = *reinterpret_cast<const int2*>(hist + b * RS_BINS + 2 * t);
            p0 += v.x; p1 += v.y;
        }
        __syncthreads();
        first[2 * t] = excl + p0;
        first[2 * t + 1] = excl + t0 + p1;
    }
    __syncthreads();
    const int n = d_n ? min(*d_n, n_cap) : n_cap;
    const int w0 = blockIdx.x * RS_CHUNK + warp * (RS_CHUNK / RS_WARPS);
    for (int g = 0; g < RS_CHUNK / RS_WARPS / 32; ++g) {                       // this warp's digit histogram
        const int i = w0 + g * 32 + lane;
        if (i < n) atomicAdd(&cnt[warp][(rs_key(src, i) >> shift) & (RS_BINS - 1)], 1);
    }
    __syncthreads();
    for (int bin = threadIdx.x; bin < RS_BINS; bin += blockDim.x) {            // -> first position of (bin, warp)
        int run = first[bin];
        for (int w = 0; w < RS_WARPS; ++w) { const int v = cnt[w][bin]; cnt[w][bin] = run; run += v; }
    }
    __syncthreads();
    for (int g = 0; g < RS_CHUNK / RS_WARPS / 32; ++g) {
        const int i = w0 + g * 32 + lane;
        const bool ok = i < n;
        const unsigned active = __ballot_sync(0xffffffffu, ok);
        if (ok) {
            const unsigned key = rs_key(src, i);
            const int val = vals_in ? vals_in[i] : i;
            const int d = (key >> shift) & (RS_BINS - 1);
            const unsigned peers = __match_any_sync(active, d);
            const int rank = __popc(peers & ((1u << lane) - 1u));
            const int pos = cnt[warp][d] + rank;
            __syncwarp(active);
            if (rank == 0) cnt[warp][d] += __popc(peers);
            __syncwarp(active);
            if (keys_out) keys_out[pos] = key;
            vals_out[pos] = val;
        }
    }
}

__device__ __forceinline__ int ro_bucket(unsigned mask, int kvol) {
    (void)kvol;
    return (int)(mask & 0xffu);
}

__global__ void k_ro_hist(const unsigned* __restrict__ mask, const int* __restrict__ d_n, int n_cap, int kvol, int* __restrict__ bins) {
    __shared__ int sh[RO_BINS];
    for (int i = threadIdx.x; i < RO_BINS; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    const int n = d_n ? min(*d_n, n_cap) : n_cap;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) atomicAdd(&sh[ro_bucket(mask[i], kvol)], 1);
    __syncthreads();
    for (int i = threadIdx.x; i < RO_BINS; i += blockDim.x) if (sh[i]) atomicAdd(&bins[i], sh[i]);
}

__global__ void k_ro_scan(int* __restrict__ bins) {        // 1 block of RO_BINS threads: exclusive scan in place
    __shared__ int sh[RO_BINS];
    const int t = threadIdx.x;
    const int v = bins[t];
    sh[t] = v;
    __syncthreads();
    for (int d = 1; d < RO_BINS; d <<= 1) {
        const int u = (t >= d) ? sh[t - d] : 0;
        __syncthreads();
        sh[t] += u;
        __syncthreads();
    }
    bins[t] = sh[t] - v;
}

__global__ void k_ro_scatter(const unsigned* __restrict__ mask, const int* __restrict__ d_n, int n_cap, int kvol,
                             int* __restrict__ cursor, int* __restrict__ perm) {
    __shared__ int cnt[RO_BINS];
    __shared__ int base[RO_BINS];
    for (int i = threadIdx.x; i < RO_BINS; i += blockDim.x) cnt[i] = 0;
    __syncthreads();
    const int n = d_n ? min(*d_n, n_cap) : n_cap;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    int b = -1, local = 0;
    if (i < n) { b = ro_bucket(mask[i], kvol); local = atomicAdd(&cnt[b], 1); }
    __syncthreads();
    for (int j = threadIdx.x; j < RO_BINS; j += blockDim.x) if (cnt[j]) base[j] = atomicAdd(&cursor[j], cnt[j]);
    __syncthreads();
    if (i < n) perm[base[b] + local] = i;
}

static int rs_blocks(int n_cap) { return cdiv(n_cap, RS_CHUNK); }

// scratch layout: [nblk][RS_BINS] histogram, [6][RS_BINS] per-pass bin totals, then keys A, keys B, vals A (n_cap each);
// kvol <= 8 uses the first RO_BINS ints only
extern "C" size_t lb2_row_order_scratch_bytes(int32_t n_cap) {
    return ((size_t)RS_BINS * (rs_blocks(n_cap) + 6) + 3 * (size_t)n_cap) * sizeof(int);
}

extern "C" int lb2_row_order(void* handle, void* stream, const uint32_t* row_mask, const int32_t* d_n, int32_t n_cap,
                             int32_t kvol, int32_t* perm, void* scratch, const int32_t* coords, int32_t coord_shift) {
    Lb2Handle* h = (Lb2Handle*)handle;
    LB2_REQUIRE(h, h && row_mask && perm && scratch && n_cap > 0 && (kvol == 27 || (kvol >= 1 && kvol <= 8)), "row_order");
    LB2_REQUIRE(h, coord_shift >= 0 && coord_shift < 24, "row_order coord_shift");
    cudaStream_t s = (cudaStream_t)stream;
    if (kvol == 27) {
        const int nblk = rs_blocks(n_cap);
        int* hist = (int*)scratch;
        int* total = hist + (size_t)RS_BINS * nblk;
        unsigned* keys_a = (unsigned*)(total + 6 * RS_BINS);
        if (cudaMemsetAsync(total, 0, 6 * RS_BINS * sizeof(int), s) != cudaSuccess) return lb2_fail(h, LB2_ERR_CUDA, "row_order memset%s", "");
        unsigned* keys_b = keys_a + n_cap;
        int* vals_a = (int*)(keys_b + n_cap);
        // LSD radix sort, 9 bits per pass.  Without coordinates: 3 passes on the mask key, values perm -> vals_a -> perm.
        // With coordinates: 3 passes on the rows' Morton code first (values vals_a -> perm -> vals_a), then the 3 mask passes
        // (perm -> vals_a -> perm): rows of equal mask end up in Morton order, i.e. a 128-row tile of a large mask group covers a
        // compact block of voxels whose gathers re-hit the same input rows in L2.
        const int npass = coords ? 6 : 3;
        for (int pass = 0; pass < npass; ++pass) {
            const int mp = coords ? pass - 3 : pass;                    // index among the mask passes (< 0: Morton pass)
            const bool to_perm = coords ? (pass & 1) : !(pass & 1);
            RsSrc src;
            src.mask = row_mask; src.coords = (const int4*)coords; src.coord_shift = coord_shift;
            src.keys = (pass & 1) ? keys_a : keys_b;
            src.vals = (pass == 0) ? nullptr : (to_perm ? vals_a : perm);
            src.mode = (pass == 0) ? (coords ? 2 : 1) : ((coords && pass == 3) ? 3 : 0);
            unsigned* kout = (pass == npass - 1 || (coords && pass == 2)) ? nullptr : ((pass & 1) ? keys_b : keys_a);
            int* vout = to_perm ? perm : vals_a;
            const int shift = (mp >= 0 ? mp : pass) * RS_BITS;
            k_rs_hist<<<nblk, 256, 0, s>>>(src, d_n, n_cap, shift, hist, total + pass * RS_BINS);
            LB2_POST_LAUNCH(h, "k_rs_hist");
            k_rs_scatter<<<nblk, 32 * RS_WARPS, 0, s>>>(src, d_n, n_cap, shift, hist, total + pass * RS_BINS, kout, vout);
            LB2_POST_LAUNCH(h, "k_rs_scatter");
        }
        return LB2_OK;
    }
    int* bins = (int*)scratch;
    if (cudaMemsetAsync(bins, 0, RO_BINS * sizeof(int), s) != cudaSuccess) return lb2_fail(h, LB2_ERR_CUDA, "row_order memset%s", "");
    k_ro_hist<<<std::min<unsigned>(cdiv(n_cap, 256), 1024u), 256, 0, s>>>(row_mask, d_n, n_cap, kvol, bins);
    LB2_POST_LAUNCH(h, "k_ro_hist");
    k_ro_scan<<<1, RO_BINS, 0, s>>>(bins);
    LB2_POST_LAUNCH(h, "k_ro_scan");
    k_ro_scatter<<<cdiv(n_cap, 256), 256, 0, s>>>(row_mask, d_n, n_cap, kvol, bins, perm);
    LB2_POST_LAUNCH(h, "k_ro_scatter");
    return LB2_OK;
}

// Stable LSD sort of 64-bit keys to a permutation (evaluation metrics, metrics.cu): perm[i] = index of the i-th smallest of the
// low key_bits bits of keys[0..n).  Each pass reads its 9-bit digit of keys[previous permutation], so the keys are never moved.
// scratch: [nblk][RS_BINS] histogram, [8][RS_BINS] per-pass totals, one int[n] ping-pong buffer.
size_t lb2_sort_keys64_scratch_bytes(int n) {
    return ((size_t)RS_BINS * (rs_blocks(n) + 8) + (size_t)n) * sizeof(int);
}

int lb2_sort_keys64(Lb2Handle* h, cudaStream_t s, const unsigned long long* keys, int n, int key_bits, int* perm, void* scratch) {
    if (n <= 0) return LB2_OK;
    const int nblk = rs_blocks(n);
    const int npass = key_bits <= RS_BITS ? 1 : (key_bits + RS_BITS - 1) / RS_BITS;
    int* hist = (int*)scratch;
    int* total = hist + (size_t)RS_BINS * nblk;
    int* tmp = total + 8 * RS_BINS;
    if (cudaMemsetAsync(total, 0, (size_t)npass * RS_BINS * sizeof(int), s) != cudaSuccess) return lb2_fail(h, LB2_ERR_CUDA, "sort_keys64 memset%s", "");
    const int* vin = nullptr;
    for (int pass = 0; pass < npass; ++pass) {
        int* vout = ((npass - 1 - pass) & 1) ? tmp : perm;                  // the last pass writes perm
        RsSrc src;
        src.keys = nullptr; src.mask = nullptr; src.coords = nullptr; src.vals = vin; src.keys64 = keys;
        src.mode = 4; src.coord_shift = 0; src.key_shift = pass * RS_BITS;
        k_rs_hist<<<nblk, 256, 0, s>>>(src, nullptr, n, 0, hist, total + pass * RS_BINS);
        LB2_POST_LAUNCH(h, "k_rs_hist");
        k_rs_scatter<<<nblk, 32 * RS_WARPS, 0, s>>>(src, nullptr, n, 0, hist, total + pass * RS_BINS, nullptr, vout);
        LB2_POST_LAUNCH(h, "k_rs_scatter");
        vin = vout;
    }
    return LB2_OK;
}

// ---------------------------------------------------------------------------------------------------
// nn tree: a bounding-volume hierarchy over the Morton-sorted keys of lb2_nn_match (built once per scan, the keys
// are the conditioning scan's stride-16 voxels).  Complete binary tree in heap order over leaves of NT_LEAF
// consecutive sorted keys; every node holds the integer bounding box (and batch range) of its keys.  The exact
// search of k_nn_match_tree (dense.cu) prunes with box distances, so its cost is ~O(log nk) per query however far the
// query is from the keys (the shell search of lb2_nn_match_grid grows with the cube of that distance).
// Buffer layout (ints): [0..15] header {min x,y,z; max x,y,z; shift; nleaf; nk_cap} | nodes [2*nleaf][8] |
// sorted keys int4[nleaf*NT_LEAF] (x, y, z, original row; -1 past the last key) | batch[nleaf*NT_LEAF] | sort scratch.
// ---------------------------------------------------------------------------------------------------
#define NT_LEAF 4
#define NT_HDR 16

static int nt_nleaf(int nk_cap) { int n = 1; while (n * NT_LEAF < nk_cap) n <<= 1; return n; }
static size_t nt_sort_ints(int nk_cap) { return (size_t)RS_BINS * (rs_blocks(nk_cap) + 3) + 4 * (size_t)nk_cap; }

extern "C" size_t lb2_nn_tree_bytes(int32_t nk_cap) {
    return (NT_HDR + (size_t)2 * nt_nleaf(nk_cap) * 8 + 5 * (size_t)nt_nleaf(nk_cap) * NT_LEAF + nt_sort_ints(nk_cap)) * sizeof(int) + 64;
}

__global__ void k_nt_init(int* __restrict__ hdr, int nleaf, int nk_cap) {
    if (threadIdx.x < 3) { hdr[threadIdx.x] = 0x7fffffff; hdr[3 + threadIdx.x] = (int)0x80000000; }
    if (threadIdx.x == 0) { hdr[6] = 0; hdr[7] = nleaf; hdr[8] = nk_cap; }
}

__global__ void k_nt_minmax(const int4* __restrict__ keys, const int* __restrict__ d_nk, int nk_cap, int* __restrict__ hdr) {
    const int nk = d_nk ? min(*d_nk, nk_cap) : nk_cap;
    int lo[3] = {0x7fffffff, 0x7fffffff, 0x7fffffff}, hi[3] = {(int)0x80000000, (int)0x80000000, (int)0x80000000};
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nk; i += gridDim.x * blockDim.x) {
        const int4 c = __ldg(keys + i);
        lo[0] = min(lo[0], c.y); lo[1] = min(lo[1], c.z); lo[2] = min(lo[2], c.w);
        hi[0] = max(hi[0], c.y); hi[1] = max(hi[1], c.z); hi[2] = max(hi[2], c.w);
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { lo[a] = min(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o)); hi[a] = max(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o)); }
        if ((threadIdx.x & 31) == 0) { atomicMin(hdr + a, lo[a]); atomicMax(hdr + 3 + a, hi[a]); }
    }
}

__device__ __forceinline__ unsigned nt_spread9(unsigned v) {        // 9 bits -> every third bit
    unsigned r = 0;
#pragma unroll
    for (int b = 0; b < 9; ++b) r |= ((v >> b) & 1u) << (3 * b);
    return r;
}

__global__ void k_nt_morton(const int4* __restrict__ keys, const int* __restrict__ d_nk, int nk_cap, const int* __restrict__ hdr,
                            unsigned* __restrict__ codes) {
    const int nk = d_nk ? min(*d_nk, nk_cap) : nk_cap;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nk) return;
    long long ext = 0;
#pragma unroll
    for (int a = 0; a < 3; ++a) ext = max(ext, (long long)hdr[3 + a] - (long long)hdr[a]);
    int shift = 0;
    while ((ext >> shift) > 511) ++shift;                             // 9 bits per axis after the shift
    const int4 c = __ldg(keys + i);
    const unsigned x = (unsigned)(((long long)c.y - hdr[0]) >> shift), y = (unsigned)(((long long)c.z - hdr[1]) >> shift),
                   z = (unsigned)(((long long)c.w - hdr[2]) >> shift);
    codes[i] = nt_spread9(x) | (nt_spread9(y) << 1) | (nt_spread9(z) << 2);
}

__global__ void k_nt_gather(const int4* __restrict__ keys, const int* __restrict__ d_nk, int nk_cap, const int* __restrict__ order,
                            int slots, int4* __restrict__ skeys, int* __restrict__ sbatch) {
    const int nk = d_nk ? min(*d_nk, nk_cap) : nk_cap;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= slots) return;
    if (i >= nk) { skeys[i] = make_int4(0, 0, 0, -1); sbatch[i] = 0; return; }
    const int j = order[i];
    const int4 c = __ldg(keys + j);
    skeys[i] = make_int4(c.y, c.z, c.w, j);
    sbatch[i] = c.x;
}

// node = {lo x,y,z, hi x,y,z, batch lo, batch hi}; an empty node has lo > hi
__global__ void k_nt_leaves(const int4* __restrict__ skeys, const int* __restrict__ sbatch, const int* __restrict__ d_nk, int nk_cap,
                            int nleaf, int* __restrict__ nodes) {
    const int nk = d_nk ? min(*d_nk, nk_cap) : nk_cap;
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= nleaf) return;
    int v[8] = {0x7fffffff, 0x7fffffff, 0x7fffffff, (int)0x80000000, (int)0x80000000, (int)0x80000000, 0x7fffffff, (int)0x80000000};
    for (int t = 0; t < NT_LEAF; ++t) {
        const int i = l * NT_LEAF + t;
        if (i >= nk) break;
        const int4 c = skeys[i];
        const int b = sbatch[i];
        v[0] = min(v[0], c.x); v[1] = min(v[1], c.y); v[2] = min(v[2], c.z);
        v[3] = max(v[3], c.x); v[4] = max(v[4], c.y); v[5] = max(v[5], c.z);
        v[6] = min(v[6], b); v[7] = max(v[7], b);
    }
    int* n = nodes + (size_t)(nleaf + l) * 8;
#pragma unroll
    for (int a = 0; a < 8; ++a) n[a] = v[a];
}

__global__ void __launch_bounds__(1024) k_nt_internal(int nleaf, int* __restrict__ nodes) {       // one block, level by level bottom-up
    for (int first = nleaf >> 1; first >= 1; first >>= 1) {
        for (int i = first + threadIdx.x; i < 2 * first; i += blockDim.x) {
            const int* a = nodes + (size_t)(2 * i) * 8;
            const int* b = a + 8;
            int* n = nodes + (size_t)i * 8;
#pragma unroll
            for (int c = 0; c < 3; ++c) { n[c] = min(a[c], b[c]); n[3 + c] = max(a[3 + c], b[3 + c]); }
            n[6] = min(a[6], b[6]); n[7] = max(a[7], b[7]);
        }
        __syncthreads();
    }
}

extern "C" int lb2_nn_tree_build(void* handle, void* stream, const int32_t* k_coords, const int32_t* d_nk, int32_t nk_cap, void* tree) {
    Lb2Handle* h = (Lb2Handle*)handle;
    LB2_REQUIRE(h, h && k_coords && tree && nk_cap > 0, "nn_tree_build");
    cudaStream_t s = (cudaStream_t)stream;
    const int nleaf = nt_nleaf(nk_cap);
    int* hdr = (int*)tree;
    int* nodes = hdr + NT_HDR;
    int4* skeys = (int4*)(nodes + (size_t)2 * nleaf * 8);
    const int slots = nleaf * NT_LEAF;
    int* sbatch = (int*)(skeys + slots);
    int* hist = sbatch + slots;
    const int nblk = rs_blocks(nk_cap);
    int* total = hist + (size_t)RS_BINS * nblk;
    unsigned* codes = (unsigned*)(total + 3 * RS_BINS);
    unsigned* keys_b = codes + nk_cap;
    int* vals_a = (int*)(keys_b + nk_cap);
    int* vals_b = vals_a + nk_cap;
    k_nt_init<<<1, 32, 0, s>>>(hdr, nleaf, nk_cap);
    LB2_POST_LAUNCH(h, "k_nt_init");
    k_nt_minmax<<<std::min<unsigned>(cdiv(nk_cap, 256), 256u), 256, 0, s>>>((const int4*)k_coords, d_nk, nk_cap, hdr);
    LB2_POST_LAUNCH(h, "k_nt_minmax");
    k_nt_morton<<<cdiv(nk_cap, 256), 256, 0, s>>>((const int4*)k_coords, d_nk, nk_cap, hdr, codes);
    LB2_POST_LAUNCH(h, "k_nt_morton");
    if (cudaMemsetAsync(total, 0, 3 * RS_BINS * sizeof(int), s) != cudaSuccess) return lb2_fail(h, LB2_ERR_CUDA, "nn_tree memset%s", "");
    //   0: codes -> keys_b, vals_a        1: keys_b, vals_a -> codes, vals_b        2: codes, vals_b -> vals_a
    const unsigned* kin[3] = {codes, keys_b, codes};
    const int* vin[3] = {nullptr, vals_a, vals_b};
    unsigned* kout[3] = {keys_b, codes, nullptr};
    int* vout[3] = {vals_a, vals_b, vals_a};
    for (int pass = 0; pass < 3; ++pass) {
        RsSrc src;
        src.keys = kin[pass]; src.mask = nullptr; src.coords = nullptr; src.vals = vin[pass]; src.mode = 0; src.coord_shift = 0;
        k_rs_hist<<<nblk, 256, 0, s>>>(src, d_nk, nk_cap, pass * RS_BITS, hist, total + pass * RS_BINS);
        LB2_POST_LAUNCH(h, "k_rs_hist");
        k_rs_scatter<<<nblk, 32 * RS_WARPS, 0, s>>>(src, d_nk, nk_cap, pass * RS_BITS, hist, total + pass * RS_BINS, kout[pass], vout[pass]);
        LB2_POST_LAUNCH(h, "k_rs_scatter");
    }
    k_nt_gather<<<cdiv(slots, 256), 256, 0, s>>>((const int4*)k_coords, d_nk, nk_cap, vals_a, slots, skeys, sbatch);
    LB2_POST_LAUNCH(h, "k_nt_gather");
    k_nt_leaves<<<cdiv(nleaf, 256), 256, 0, s>>>(skeys, sbatch, d_nk, nk_cap, nleaf, nodes);
    LB2_POST_LAUNCH(h, "k_nt_leaves");
    k_nt_internal<<<1, 1024, 0, s>>>(nleaf, nodes);
    LB2_POST_LAUNCH(h, "k_nt_internal");
    return LB2_OK;
}

// ---------------------------------------------------------------------------------------------------
// tile order: the persistent convolution kernels assign tiles to CTAs statically (snake order).  That is balanced only if the tiles
// are sorted by cost.  The cost of a tile is the number of kernel offsets it has to run = popcount of the OR of its rows' masks;
// the mask-sorted row order is not monotone in it.  k_tile_masks ORs the masks of every 128-row tile (one warp per tile),
// k_tile_sort counting-sorts the 128-row tiles and the 256-row super-tiles (CTA pairs) by descending cost.
//   order128[i] / order256[i] = index of the i-th most expensive tile; entries beyond the live tile count are -1.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_tile_masks(const unsigned* __restrict__ mask, const int* __restrict__ perm, const int* __restrict__ d_n,
                                                    int n_cap, unsigned* __restrict__ tmask) {
    const int n = d_n ? min(*d_n, n_cap) : n_cap;
    const int nt = (n + 127) >> 7;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= nt) return;
    unsigned m = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int slot = warp * 128 + q * 32 + lane;
        if (slot < n) m |= __ldg(mask + (perm ? __ldg(perm + slot) : slot));
    }
    m = __reduce_or_sync(0xffffffffu, m);
    if (lane == 0) tmask[warp] = m;
}

__global__ void __launch_bounds__(1024) k_tile_sort(const unsigned* __restrict__ tmask, const int* __restrict__ d_n, int n_cap,
                                                    int* __restrict__ order128, int* __restrict__ order256) {
    __shared__ int bins[2][33];
    const int n = d_n ? min(*d_n, n_cap) : n_cap;
    const int nt128 = (n + 127) >> 7, nt256 = (n + 255) >> 8;
    const int cap128 = (n_cap + 127) >> 7, cap256 = (n_cap + 255) >> 8;
    if (threadIdx.x < 66) (&bins[0][0])[threadIdx.x] = 0;
    __syncthreads();
    // histogram of costs (0..32), descending order: bin b holds cost 32 - b
    for (int t = threadIdx.x; t < nt128; t += blockDim.x) atomicAdd(&bins[0][32 - __popc(tmask[t])], 1);
    for (int u = threadIdx.x; u < nt256; u += blockDim.x) {
        const unsigned m = tmask[2 * u] | ((2 * u + 1 < nt128) ? tmask[2 * u + 1] : 0u);
        atomicAdd(&bins[1][32 - __popc(m)], 1);
    }
    __syncthreads();
    if (threadIdx.x < 2) {                                   // exclusive scan of 33 bins
        int run = 0;
        for (int b = 0; b < 33; ++b) { const int v = bins[threadIdx.x][b]; bins[threadIdx.x][b] = run; run += v; }
    }
    __syncthreads();
    for (int t = threadIdx.x; t < nt128; t += blockDim.x) order128[atomicAdd(&bins[0][32 - __popc(tmask[t])], 1)] = t;
    for (int u = threadIdx.x; u < nt256; u += blockDim.x) {
        const unsigned m = tmask[2 * u] | ((2 * u + 1 < nt128) ? tmask[2 * u + 1] : 0u);
        order256[atomicAdd(&bins[1][32 - __popc(m)], 1)] = u;
    }
    for (int t = nt128 + threadIdx.x; t < cap128; t += blockDim.x) order128[t] = -1;
    for (int u = nt256 + threadIdx.x; u < cap256; u += blockDim.x) order256[u] = -1;
}

// dense / residual split of the row masks per 256-row super-tile (the work item of k_spconv_tc_pair): an offset stays in the
// output-stationary work when at least min_rows rows of the super-tile have it; otherwise the pairs of that offset go to the
// residual mask, whose pairs lb2_pair_list compacts for the gather-GEMM-scatter kernel.  Every pair lands in exactly one of the two.
__global__ void __launch_bounds__(256) k_tile_split(const unsigned* __restrict__ mask, const int* __restrict__ perm, const int* __restrict__ d_n,
                                                    int n_cap, int kvol, int min_rows, unsigned* __restrict__ dense, unsigned* __restrict__ res) {
    const int n = d_n ? min(*d_n, n_cap) : n_cap;
    if (blockIdx.x * 256 >= n) return;                                 // uniform over the block
    const int slot = blockIdx.x * 256 + threadIdx.x;
    const int row = slot < n ? (perm ? __ldg(perm + slot) : slot) : -1;
    const unsigned m = row >= 0 ? __ldg(mask + row) : 0u;
    unsigned keep = 0;
    for (int k = 0; k < kvol; ++k)
        if (__syncthreads_count((m >> k) & 1u) >= min_rows) keep |= 1u << k;
    if (row >= 0) { dense[row] = m & keep; res[row] = m & ~keep; }
}

extern "C" int lb2_tile_split(void* handle, void* stream, const uint32_t* row_mask, const int32_t* row_perm, const int32_t* d_n, int32_t n_cap,
                              int32_t kvol, int32_t min_rows, uint32_t* dense_mask, uint32_t* res_mask) {
    Lb2Handle* h = (Lb2Handle*)handle;
    LB2_REQUIRE(h, h && row_mask && dense_mask && res_mask && n_cap > 0 && kvol >= 1 && kvol <= 32 && min_rows >= 0 && min_rows <= 256,
                "tile_split");
    cudaStream_t s = (cudaStream_t)stream;
    k_tile_split<<<cdiv(n_cap, 256), 256, 0, s>>>(row_mask, row_perm, d_n, n_cap, kvol, min_rows, dense_mask, res_mask);
    LB2_POST_LAUNCH(h, "k_tile_split");
    return LB2_OK;
}

extern "C" int lb2_tile_order(void* handle, void* stream, const uint32_t* row_mask, const int32_t* row_perm, const int32_t* d_n, int32_t n_cap,
                              int32_t* order128, int32_t* order256, void* scratch) {
    Lb2Handle* h = (Lb2Handle*)handle;
    LB2_REQUIRE(h, h && row_mask && order128 && order256 && scratch && n_cap > 0, "tile_order");
    cudaStream_t s = (cudaStream_t)stream;
    const int cap128 = cdiv(n_cap, 128);
    k_tile_masks<<<cdiv(cap128, 8), 256, 0, s>>>(row_mask, row_perm, d_n, n_cap, (unsigned*)scratch);
    LB2_POST_LAUNCH(h, "k_tile_masks");
    k_tile_sort<<<1, 1024, 0, s>>>((const unsigned*)scratch, d_n, n_cap, order128, order256);
    LB2_POST_LAUNCH(h, "k_tile_sort");
    return LB2_OK;
}

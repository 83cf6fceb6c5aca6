// Evaluation metrics of completed scans — what lidiff/utils/metrics.py and histogram_metrics.py compute with open3d's k-d tree and
// dense np.histogramdd grids:
//   * exact fp64 cloud-to-cloud nearest distance (RMSE, Chamfer distance, precision / recall) over a bounding-box hierarchy;
//   * two-cloud voxel histograms on np.histogramdd's binning without materialising the grid (CompletionIoU, JSD 3D / BEV);
//   * threshold counts #{i : d[i] < thr[t]} (the precision / recall curve).
// The fp64 sums are reduced in a fixed order (per-block partials, then one block): two runs on the same input give the same bits.
#include "common.cuh"
#include <math.h>
#include <algorithm>

#define CN_LEAF 8            // points per leaf of the nearest-distance hierarchy
#define CN_STACK 32          // traversal stack; the tree depth is log2(nleaf) <= 28 for n < 2^31
#define RED_BLOCKS 256       // blocks of the partial reductions (a function of nothing but this constant)
#define THR_MAX 8192         // thresholds of lb2_threshold_counts (shared-memory histogram)

static inline size_t al256(size_t b) { return (b + 255) / 256 * 256; }
static inline unsigned red_blocks(long long n) { return std::max(1u, std::min<unsigned>(cdiv(n, 256), RED_BLOCKS)); }

// ---------------------------------------------------------------------------------------------------
// nearest distance: Morton-sorted bounding-box hierarchy over the reference cloud
//   nodes: heap order (root 1, children 2i / 2i+1, leaves nleaf..2nleaf-1), {lo x,y,z, hi x,y,z} fp64 computed from the leaf's
//   points, so a box distance is a true lower bound of the point distances below it (rounding is monotone); an empty box has
//   lo = +inf, hi = -inf and distance +inf.  Leaf slots past the last point hold +inf coordinates.
// ---------------------------------------------------------------------------------------------------
static int cn_nleaf(int n) { int l = 1; while ((long long)l * CN_LEAF < n) l <<= 1; return l; }

__global__ void __launch_bounds__(256) k_cn_bbox_partial(const double* __restrict__ p, int n, double* __restrict__ part) {
    __shared__ double sh[6][8];
    double v[6] = {INFINITY, INFINITY, INFINITY, -INFINITY, -INFINITY, -INFINITY};
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
#pragma unroll
        for (int a = 0; a < 3; ++a) { const double x = __ldg(p + 3 * (size_t)i + a); v[a] = fmin(v[a], x); v[3 + a] = fmax(v[3 + a], x); }
    }
#pragma unroll
    for (int a = 0; a < 6; ++a) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double u = __shfl_xor_sync(0xffffffffu, v[a], o);
            v[a] = a < 3 ? fmin(v[a], u) : fmax(v[a], u);
        }
        if ((threadIdx.x & 31) == 0) sh[a][threadIdx.x >> 5] = v[a];
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        const int a = threadIdx.x;
        double r = sh[a][0];
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) r = a < 3 ? fmin(r, sh[a][w]) : fmax(r, sh[a][w]);
        part[blockIdx.x * 6 + a] = r;
    }
}

__global__ void k_cn_bbox_final(const double* __restrict__ part, int nblk, double* __restrict__ box) {
    if (threadIdx.x >= 6) return;
    const int a = threadIdx.x;
    double r = part[a];
    for (int b = 1; b < nblk; ++b) r = a < 3 ? fmin(r, part[b * 6 + a]) : fmax(r, part[b * 6 + a]);
    box[a] = r;
}

__device__ __forceinline__ unsigned long long cn_spread10(unsigned v) {      // 10 bits -> every third bit
    unsigned long long x = v & 0x3ffu;
    x = (x | (x << 16)) & 0x030000ffull;
    x = (x | (x << 8)) & 0x0300f00full;
    x = (x | (x << 4)) & 0x030c30c3ull;
    x = (x | (x << 2)) & 0x09249249ull;
    return x;
}

// 30-bit Morton code of the point in the cloud's bounding box (cubic cells, 1024 per axis of the longest extent): ordering only
__global__ void k_cn_morton(const double* __restrict__ p, int n, const double* __restrict__ box, unsigned long long* __restrict__ code) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double ext = fmax(fmax(box[3] - box[0], box[4] - box[1]), box[5] - box[2]);
    const double s = ext > 0.0 ? 1023.0 / ext : 0.0;
    unsigned c[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const double t = (__ldg(p + 3 * (size_t)i + a) - box[a]) * s;
        c[a] = t >= 0.0 ? (unsigned)fmin(t, 1023.0) : 0u;                          // NaN -> 0
    }
    code[i] = cn_spread10(c[0]) | (cn_spread10(c[1]) << 1) | (cn_spread10(c[2]) << 2);
}

__global__ void k_cn_gather(const double* __restrict__ p, int n, const int* __restrict__ perm, int slots, double* __restrict__ sp) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= slots) return;
    if (i >= n) { sp[3 * (size_t)i] = INFINITY; sp[3 * (size_t)i + 1] = INFINITY; sp[3 * (size_t)i + 2] = INFINITY; return; }
    const size_t j = (size_t)__ldg(perm + i);
#pragma unroll
    for (int a = 0; a < 3; ++a) sp[3 * (size_t)i + a] = __ldg(p + 3 * j + a);
}

__global__ void k_cn_leaves(const double* __restrict__ sp, int n, int nleaf, double* __restrict__ nodes) {
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= nleaf) return;
    double v[6] = {INFINITY, INFINITY, INFINITY, -INFINITY, -INFINITY, -INFINITY};
    for (int t = 0; t < CN_LEAF; ++t) {
        const int i = l * CN_LEAF + t;
        if (i >= n) break;
#pragma unroll
        for (int a = 0; a < 3; ++a) { const double x = sp[3 * (size_t)i + a]; v[a] = fmin(v[a], x); v[3 + a] = fmax(v[3 + a], x); }
    }
    double* nd = nodes + (size_t)(nleaf + l) * 6;
#pragma unroll
    for (int a = 0; a < 6; ++a) nd[a] = v[a];
}

__device__ __forceinline__ void cn_merge(double* __restrict__ nodes, int i) {
    const double* a = nodes + (size_t)(2 * i) * 6;
    const double* b = a + 6;
    double* nd = nodes + (size_t)i * 6;
#pragma unroll
    for (int c = 0; c < 3; ++c) { nd[c] = fmin(a[c], b[c]); nd[3 + c] = fmax(a[3 + c], b[3 + c]); }
}

__global__ void k_cn_level(double* __restrict__ nodes, int first) {            // nodes [first, 2*first) of one level
    const int i = first + blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 2 * first) cn_merge(nodes, i);
}

__global__ void __launch_bounds__(1024) k_cn_top(double* __restrict__ nodes, int first) {   // levels first, first/2, ..., 1 in one block
    for (; first >= 1; first >>= 1) {
        for (int i = first + threadIdx.x; i < 2 * first; i += blockDim.x) cn_merge(nodes, i);
        __syncthreads();
    }
}

// squared distance in numpy's order, without FMA contraction: (dx*dx + dy*dy) + dz*dz
__device__ __forceinline__ double cn_d2(double dx, double dy, double dz) {
    return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

__device__ __forceinline__ double cn_box_d2(const double* __restrict__ nd, double qx, double qy, double qz) {
    const double gx = fmax(fmax(__dsub_rn(__ldg(nd + 0), qx), __dsub_rn(qx, __ldg(nd + 3))), 0.0);
    const double gy = fmax(fmax(__dsub_rn(__ldg(nd + 1), qy), __dsub_rn(qy, __ldg(nd + 4))), 0.0);
    const double gz = fmax(fmax(__dsub_rn(__ldg(nd + 2), qz), __dsub_rn(qz, __ldg(nd + 5))), 0.0);
    return cn_d2(gx, gy, gz);
}

// one thread per query, queries taken in the Morton order of the query cloud (neighbouring lanes walk the same branches);
// depth-first, nearer child first, subtrees whose box is not strictly closer than the best distance so far are skipped
__global__ void __launch_bounds__(128) k_cn_search(const double* __restrict__ q, const int* __restrict__ qperm, int nq,
                                                   const double* __restrict__ nodes, const double* __restrict__ sp, int nleaf,
                                                   double* __restrict__ dist) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nq) return;
    const size_t j = (size_t)__ldg(qperm + i);
    const double qx = __ldg(q + 3 * j), qy = __ldg(q + 3 * j + 1), qz = __ldg(q + 3 * j + 2);
    double best = INFINITY;
    int stack[CN_STACK];
    double bound[CN_STACK];
    int sp_top = 0, node = 1;
    while (true) {
        if (node >= nleaf) {
            const double* p = sp + (size_t)(node - nleaf) * CN_LEAF * 3;
#pragma unroll
            for (int t = 0; t < CN_LEAF; ++t) {
                const double d = cn_d2(__dsub_rn(qx, __ldg(p + 3 * t)), __dsub_rn(qy, __ldg(p + 3 * t + 1)), __dsub_rn(qz, __ldg(p + 3 * t + 2)));
                best = d < best ? d : best;
            }
        } else {
            int near = 2 * node, far = near + 1;
            double bn = cn_box_d2(nodes + (size_t)near * 6, qx, qy, qz), bf = cn_box_d2(nodes + (size_t)far * 6, qx, qy, qz);
            if (bf < bn) { const int t = near; near = far; far = t; const double u = bn; bn = bf; bf = u; }
            if (bf < best) { stack[sp_top] = far; bound[sp_top] = bf; ++sp_top; }
            if (bn < best) { node = near; continue; }
        }
        bool found = false;
        while (sp_top > 0) {
            --sp_top;
            if (bound[sp_top] < best) { node = stack[sp_top]; found = true; break; }
        }
        if (!found) break;
    }
    dist[j] = sqrt(best);
}

struct CnScratch {
    double *part, *rbox, *qbox, *nodes, *sp;
    unsigned long long* code;
    int *rperm, *qperm;
    void* sort;
};

static size_t cn_carve(int64_t nq, int64_t nr, char* base, CnScratch* c) {
    const int nmax = (int)std::max<int64_t>(std::max<int64_t>(nq, nr), 1);
    const int nleaf = cn_nleaf((int)std::max<int64_t>(nr, 1));
    size_t off = 0;
    auto take = [&](size_t bytes) { char* p = base ? base + off : nullptr; off += al256(bytes); return (void*)p; };
    CnScratch t;
    t.part = (double*)take(RED_BLOCKS * 6 * sizeof(double));
    t.rbox = (double*)take(6 * sizeof(double));
    t.qbox = (double*)take(6 * sizeof(double));
    t.code = (unsigned long long*)take((size_t)nmax * 8);
    t.rperm = (int*)take((size_t)std::max<int64_t>(nr, 1) * 4);
    t.qperm = (int*)take((size_t)std::max<int64_t>(nq, 1) * 4);
    t.nodes = (double*)take((size_t)2 * nleaf * 6 * sizeof(double));
    t.sp = (double*)take((size_t)nleaf * CN_LEAF * 3 * sizeof(double));
    t.sort = take(lb2_sort_keys64_scratch_bytes(nmax));
    if (c) *c = t;
    return off + 256;
}

extern "C" size_t lb2_cloud_nn_scratch_bytes(int64_t nq, int64_t nr) {
    if (nq < 0 || nr < 0 || nq >= (1ll << 31) || nr >= (1ll << 31)) return 0;
    return cn_carve(nq, nr, nullptr, nullptr);
}

// bounding box + Morton order of a cloud: box (6 doubles), perm (n ints)
static int cn_order(Lb2Handle* h, cudaStream_t s, const double* p, int n, CnScratch& c, double* box, int* perm) {
    const unsigned nb = red_blocks(n);
    k_cn_bbox_partial<<<nb, 256, 0, s>>>(p, n, c.part);
    LB2_POST_LAUNCH(h, "k_cn_bbox_partial");
    k_cn_bbox_final<<<1, 32, 0, s>>>(c.part, (int)nb, box);
    LB2_POST_LAUNCH(h, "k_cn_bbox_final");
    k_cn_morton<<<cdiv(n, 256), 256, 0, s>>>(p, n, box, c.code);
    LB2_POST_LAUNCH(h, "k_cn_morton");
    return lb2_sort_keys64(h, s, c.code, n, 30, perm, c.sort);
}

extern "C" int lb2_cloud_nn_distance(void* handle, void* stream, const double* query, int64_t nq, const double* ref, int64_t nr,
                                     void* scratch, double* dist) {
    Lb2Handle* h = (Lb2Handle*)handle;
    LB2_REQUIRE(h, h && nq >= 0 && nq < (1ll << 31) && nr >= 0 && nr < (1ll << 31), "cloud_nn_distance sizes (0 <= n < 2^31)");
    if (nq == 0) return LB2_OK;
    LB2_REQUIRE(h, query && ref && scratch && dist && nr > 0, "cloud_nn_distance (pointers; non-empty reference cloud)");
    cudaStream_t s = (cudaStream_t)stream;
    char* base = (char*)(((uintptr_t)scratch + 255) & ~(uintptr_t)255);
    CnScratch c;
    cn_carve(nq, nr, base, &c);
    const int n = (int)nr, m = (int)nq;
    const int nleaf = cn_nleaf(n), slots = nleaf * CN_LEAF;
    int rc = cn_order(h, s, ref, n, c, c.rbox, c.rperm);
    if (rc) return rc;
    k_cn_gather<<<cdiv(slots, 256), 256, 0, s>>>(ref, n, c.rperm, slots, c.sp);
    LB2_POST_LAUNCH(h, "k_cn_gather");
    k_cn_leaves<<<cdiv(nleaf, 256), 256, 0, s>>>(c.sp, n, nleaf, c.nodes);
    LB2_POST_LAUNCH(h, "k_cn_leaves");
    int first = nleaf >> 1;
    for (; first >= 2048; first >>= 1) {
        k_cn_level<<<cdiv(first, 256), 256, 0, s>>>(c.nodes, first);
        LB2_POST_LAUNCH(h, "k_cn_level");
    }
    if (first >= 1) {
        k_cn_top<<<1, 1024, 0, s>>>(c.nodes, first);
        LB2_POST_LAUNCH(h, "k_cn_top");
    }
    rc = cn_order(h, s, query, m, c, c.qbox, c.qperm);
    if (rc) return rc;
    k_cn_search<<<cdiv(m, 128), 128, 0, s>>>(query, c.qperm, m, c.nodes, c.sp, nleaf, dist);
    LB2_POST_LAUNCH(h, "k_cn_search");
    return LB2_OK;
}

// ---------------------------------------------------------------------------------------------------
// two-cloud voxel histogram.  Bin of a coordinate = searchsorted(edges, x, 'right') - 1, a coordinate equal to edges[bins] goes in
// the last bin, anything outside [edges[0], edges[bins]] (or NaN) drops the point: np.histogramdd's rule.  Key of a point =
// ((ix*bins + iy)*bins + iz)*2 + cloud (dropped points: 2*bins^3, sorted last); after the sort an occupied bin is a run of equal
// key >> 1 (cloud a first) and a BEV column a run of equal (key >> 1) / bins.  One thread per run head walks its run.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ int vh_bin(const double* __restrict__ edges, int bins, double x) {
    int lo = 0, hi = bins + 1;                          // number of edges <= x
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(edges + mid) <= x) lo = mid + 1; else hi = mid;
    }
    if (x == __ldg(edges + bins)) --lo;
    return (lo >= 1 && lo <= bins) ? lo - 1 : -1;
}

__global__ void k_vh_keys(const double* __restrict__ a, int na, const double* __restrict__ b, int nb, const double* __restrict__ edges,
                          int bins, unsigned long long* __restrict__ keys) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= na + nb) return;
    const int cloud = i >= na;
    const double* p = cloud ? b + 3 * (size_t)(i - na) : a + 3 * (size_t)i;
    const unsigned long long B = (unsigned long long)bins;
    const int ix = vh_bin(edges, bins, __ldg(p)), iy = vh_bin(edges, bins, __ldg(p + 1)), iz = vh_bin(edges, bins, __ldg(p + 2));
    keys[i] = (ix < 0 || iy < 0 || iz < 0) ? 2ull * B * B * B : ((((unsigned long long)ix * B + iy) * B + iz) << 1) | (unsigned long long)cloud;
}

__global__ void k_vh_sorted(const unsigned long long* __restrict__ keys, const int* __restrict__ perm, int n, unsigned long long* __restrict__ sk) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) sk[i] = __ldg(keys + __ldg(perm + i));
}

// pass 1: in-range points and occupied bins of each cloud (integer counts: atomics are exact)
__global__ void __launch_bounds__(256) k_vh_count(const unsigned long long* __restrict__ sk, int n, unsigned long long drop,
                                                  lb2_voxel_hist_result* __restrict__ out) {
    long long c[5] = {0, 0, 0, 0, 0};                    // n_a, n_b, occ_a, occ_b, occ_ab
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const unsigned long long k = sk[i];
        if (k == drop) break;                            // dropped points sort last
        if (i > 0 && (sk[i - 1] >> 1) == (k >> 1)) continue;
        long long ca = 0, cb = 0;
        for (int j = i; j < n && (sk[j] >> 1) == (k >> 1) && sk[j] != drop; ++j) { if (sk[j] & 1ull) ++cb; else ++ca; }
        c[0] += ca; c[1] += cb; c[2] += ca > 0; c[3] += cb > 0; c[4] += (ca > 0 && cb > 0);
    }
    __shared__ long long sh[5];
    if (threadIdx.x < 5) sh[threadIdx.x] = 0;
    __syncthreads();
#pragma unroll
    for (int t = 0; t < 5; ++t) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c[t] += __shfl_xor_sync(0xffffffffu, c[t], o);
        if ((threadIdx.x & 31) == 0 && c[t]) atomicAdd((unsigned long long*)&sh[t], (unsigned long long)c[t]);
    }
    __syncthreads();
    if (threadIdx.x < 5 && sh[threadIdx.x]) {
        int64_t* dst = threadIdx.x == 0 ? &out->n_a : threadIdx.x == 1 ? &out->n_b : threadIdx.x == 2 ? &out->occ_a : threadIdx.x == 3 ? &out->occ_b : &out->occ_ab;
        atomicAdd((unsigned long long*)dst, (unsigned long long)sh[threadIdx.x]);
    }
}

// scipy.special.rel_entr(x, y) for x >= 0, y > 0 where x > 0
__device__ __forceinline__ double vh_rel_entr(double x, double y) { return x > 0.0 ? x * log(x / y) : 0.0; }

// pass 2: the Jensen-Shannon terms, p = count_a / sum_a, q = count_b / sum_b, m = (p + q) / 2:
//   [0] sum rel_entr(p, m), [1] sum rel_entr(q, m) over the 3-D bins; [2], [3] the same over the BEV columns, whose counts are the
//   numbers of occupied z bins.  Per-thread sums in grid-stride order, per-block tree reduction -> part[block][4].
__global__ void __launch_bounds__(256) k_vh_terms(const unsigned long long* __restrict__ sk, int n, unsigned long long drop,
                                                  unsigned long long bins, const lb2_voxel_hist_result* __restrict__ cnt,
                                                  double* __restrict__ part) {
    const double na = (double)cnt->n_a, nb = (double)cnt->n_b, oa = (double)cnt->occ_a, ob = (double)cnt->occ_b;
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const unsigned long long k = sk[i];
        if (k == drop) break;
        const unsigned long long v = k >> 1;
        const unsigned long long prev = i > 0 ? (sk[i - 1] >> 1) : ~0ull;
        if (prev == v) continue;
        long long ca = 0, cb = 0;
        for (int j = i; j < n && (sk[j] >> 1) == v && sk[j] != drop; ++j) { if (sk[j] & 1ull) ++cb; else ++ca; }
        {
            const double p = ca / na, q = cb / nb, m = (p + q) / 2.0;
            acc[0] += vh_rel_entr(p, m);
            acc[1] += vh_rel_entr(q, m);
        }
        if (i == 0 || prev / bins != v / bins) {                 // head of a BEV column: count its occupied bins per cloud
            long long za = 0, zb = 0;
            unsigned long long last = ~0ull;
            bool has_a = false, has_b = false;
            for (int j = i; j < n && sk[j] != drop && (sk[j] >> 1) / bins == v / bins; ++j) {
                const unsigned long long w = sk[j] >> 1;
                if (w != last) { za += has_a; zb += has_b; has_a = has_b = false; last = w; }
                if (sk[j] & 1ull) has_b = true; else has_a = true;
            }
            za += has_a; zb += has_b;
            const double p = za / oa, q = zb / ob, m = (p + q) / 2.0;
            acc[2] += vh_rel_entr(p, m);
            acc[3] += vh_rel_entr(q, m);
        }
    }
    __shared__ double sh[4][256];
#pragma unroll
    for (int t = 0; t < 4; ++t) sh[t][threadIdx.x] = acc[t];
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) {
#pragma unroll
            for (int t = 0; t < 4; ++t) sh[t][threadIdx.x] += sh[t][threadIdx.x + w];
        }
        __syncthreads();
    }
    if (threadIdx.x < 4) part[blockIdx.x * 4 + threadIdx.x] = sh[threadIdx.x][0];
}

__global__ void k_vh_final(const double* __restrict__ part, int nblk, lb2_voxel_hist_result* __restrict__ out) {
    if (threadIdx.x != 0) return;
    double s[4] = {0.0, 0.0, 0.0, 0.0};
    for (int b = 0; b < nblk; ++b)
        for (int t = 0; t < 4; ++t) s[t] += part[b * 4 + t];
    out->jsd_3d = sqrt((s[0] + s[1]) / 2.0);
    out->jsd_bev = sqrt((s[2] + s[3]) / 2.0);
}

static size_t vh_carve(int64_t n, char* base, unsigned long long** keys, unsigned long long** sk, int** perm, double** part, void** sort) {
    const int nn = (int)std::max<int64_t>(n, 1);
    size_t off = 0;
    auto take = [&](size_t bytes) { char* p = base ? base + off : nullptr; off += al256(bytes); return (void*)p; };
    void* k = take((size_t)nn * 8);
    void* s = take((size_t)nn * 8);
    void* p = take((size_t)nn * 4);
    void* r = take(RED_BLOCKS * 4 * sizeof(double));
    void* t = take(lb2_sort_keys64_scratch_bytes(nn));
    if (keys) { *keys = (unsigned long long*)k; *sk = (unsigned long long*)s; *perm = (int*)p; *part = (double*)r; *sort = t; }
    return off + 256;
}

extern "C" size_t lb2_voxel_hist_scratch_bytes(int64_t na, int64_t nb) {
    if (na < 0 || nb < 0 || na + nb >= (1ll << 31)) return 0;
    return vh_carve(na + nb, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
}

extern "C" int lb2_voxel_hist_compare(void* handle, void* stream, const double* a, int64_t na, const double* b, int64_t nb,
                                      const double* edges, int32_t bins, void* scratch, lb2_voxel_hist_result* out) {
    Lb2Handle* h = (Lb2Handle*)handle;
    LB2_REQUIRE(h, h && na >= 0 && nb >= 0 && na + nb < (1ll << 31), "voxel_hist_compare sizes (0 <= na + nb < 2^31)");
    // keys up to 2*bins^3 must fit 64 bits: bins < 2^21
    LB2_REQUIRE(h, bins >= 1 && bins < (1 << 21), "voxel_hist_compare bins (1 <= bins < 2^21: bin keys must fit 64 bits)");
    LB2_REQUIRE(h, edges && scratch && out && (na == 0 || a) && (nb == 0 || b), "voxel_hist_compare pointers");
    cudaStream_t s = (cudaStream_t)stream;
    if (cudaMemsetAsync(out, 0, sizeof(lb2_voxel_hist_result), s) != cudaSuccess) return lb2_fail(h, LB2_ERR_CUDA, "voxel_hist memset%s", "");
    const int n = (int)(na + nb);
    if (n == 0) return LB2_OK;
    char* base = (char*)(((uintptr_t)scratch + 255) & ~(uintptr_t)255);
    unsigned long long *keys, *sk;
    int* perm;
    double* part;
    void* sort;
    vh_carve(n, base, &keys, &sk, &perm, &part, &sort);
    const unsigned long long B = (unsigned long long)bins, drop = 2ull * B * B * B;
    int key_bits = 1;
    while (key_bits < 64 && (drop >> key_bits) != 0) ++key_bits;
    k_vh_keys<<<cdiv(n, 256), 256, 0, s>>>(a, (int)na, b, (int)nb, edges, bins, keys);
    LB2_POST_LAUNCH(h, "k_vh_keys");
    int rc = lb2_sort_keys64(h, s, keys, n, key_bits, perm, sort);
    if (rc) return rc;
    k_vh_sorted<<<cdiv(n, 256), 256, 0, s>>>(keys, perm, n, sk);
    LB2_POST_LAUNCH(h, "k_vh_sorted");
    const unsigned nblk = red_blocks(n);
    k_vh_count<<<nblk, 256, 0, s>>>(sk, n, drop, out);
    LB2_POST_LAUNCH(h, "k_vh_count");
    k_vh_terms<<<nblk, 256, 0, s>>>(sk, n, drop, B, out, part);
    LB2_POST_LAUNCH(h, "k_vh_terms");
    k_vh_final<<<1, 32, 0, s>>>(part, (int)nblk, out);
    LB2_POST_LAUNCH(h, "k_vh_final");
    return LB2_OK;
}

// ---------------------------------------------------------------------------------------------------
// threshold counts: counts[t] = #{i : d[i] < thr[t]} for ascending thr.  j(d) = number of thresholds <= d (NaN: all of them);
// d is counted for t >= j(d): integer histogram of j, then an inclusive scan.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_thr_hist(const double* __restrict__ d, int n, const double* __restrict__ thr, int nthr,
                                                  unsigned long long* __restrict__ counts) {
    extern __shared__ unsigned sh_thr[];
    for (int t = threadIdx.x; t < nthr; t += blockDim.x) sh_thr[t] = 0;
    __syncthreads();
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const double x = __ldg(d + i);
        int lo = 0, hi = nthr;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (__ldg(thr + mid) <= x) lo = mid + 1; else hi = mid;
        }
        if (x != x) lo = nthr;
        if (lo < nthr) atomicAdd(&sh_thr[lo], 1u);
    }
    __syncthreads();
    for (int t = threadIdx.x; t < nthr; t += blockDim.x)
        if (sh_thr[t]) atomicAdd(counts + t, (unsigned long long)sh_thr[t]);
}

__global__ void k_thr_scan(unsigned long long* __restrict__ counts, int nthr) {
    if (threadIdx.x != 0) return;
    unsigned long long run = 0;
    for (int t = 0; t < nthr; ++t) { run += counts[t]; counts[t] = run; }
}

extern "C" int lb2_threshold_counts(void* handle, void* stream, const double* d, int64_t n, const double* thr, int32_t nthr, int64_t* counts) {
    Lb2Handle* h = (Lb2Handle*)handle;
    LB2_REQUIRE(h, h && n >= 0 && n < (1ll << 31), "threshold_counts n (0 <= n < 2^31)");
    LB2_REQUIRE(h, nthr >= 0 && nthr <= THR_MAX, "threshold_counts nthr (0 <= nthr <= 8192)");
    if (nthr == 0) return LB2_OK;
    LB2_REQUIRE(h, thr && counts && (n == 0 || d), "threshold_counts pointers");
    cudaStream_t s = (cudaStream_t)stream;
    if (cudaMemsetAsync(counts, 0, (size_t)nthr * sizeof(int64_t), s) != cudaSuccess) return lb2_fail(h, LB2_ERR_CUDA, "threshold_counts memset%s", "");
    if (n == 0) return LB2_OK;
    k_thr_hist<<<std::min<unsigned>(cdiv(n, 256), 2 * (unsigned)h->num_sms), 256, (size_t)nthr * sizeof(unsigned), s>>>(
        d, (int)n, thr, nthr, (unsigned long long*)counts);
    LB2_POST_LAUNCH(h, "k_thr_hist");
    k_thr_scan<<<1, 32, 0, s>>>((unsigned long long*)counts, nthr);
    LB2_POST_LAUNCH(h, "k_thr_scan");
    return LB2_OK;
}

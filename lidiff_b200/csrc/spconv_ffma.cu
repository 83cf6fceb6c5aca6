// K4 (variant A) — sparse convolution as an output-stationary implicit GEMM on the fp32 CUDA cores.
//
// Used for layers the tensor-core variant does not take (Cin = 3 stem, odd channel counts) and as
// the in-library fp32 baseline the tcgen05 variant is validated against.  One CTA owns a tile of
// 64 output rows x 64 output channels, walks the kernel offsets k (skipping offsets where none of
// its 64 rows has a neighbour), gathers the neighbour rows of the current Cin chunk into shared
// memory and accumulates in registers (4x4 micro-tile per thread).  The epilogue fuses what follows
// the convolution in the reference network: MinkowskiBatchNorm(eval) as a per-channel affine,
// residual add, MinkowskiReLU, and the conditioning gate multiply.
//
// Stands behind ME.MinkowskiConvolution / MinkowskiConvolutionTranspose forward
// (/root/reference/lidiff/models/minkunet.py:17-24,36-42,53-74) — semantics SURVEY.md App. A.4/A.5.
#include "common.cuh"
#include "tc_common.cuh"

#define FF_BM 64
#define FF_BN 64
#define FF_BK 16
#define FF_THREADS 256

struct FfmaParams {
    int c1, c2, cout, kvol;
    const float* W;
    const float* scale;
    const float* shift;
    int relu;
    const int* nbr;
    long long nbr_stride;
    const int* d_mout;
    int mout_cap;
    const int* row_perm;
    const unsigned* row_mask;   // offsets to convolve per output row (NULL: all of the map)
    lb2_conv_io io[2];
};

__global__ void __launch_bounds__(FF_THREADS) k_spconv_ffma(const FfmaParams p) {
    __shared__ int   idx_s[FF_BM];
    __shared__ int   row_s[FF_BM];
    __shared__ unsigned mask_s[FF_BM];
    __shared__ float As[FF_BK][FF_BM + 4];
    __shared__ float Bs[FF_BK][FF_BN + 4];

    const int M = p.d_mout ? min(*p.d_mout, p.mout_cap) : p.mout_cap;
    const int m0 = blockIdx.x * FF_BM;
    if (m0 >= M) return;
    const int n0 = blockIdx.y * FF_BN;
    const lb2_conv_io io = p.io[blockIdx.z];
    const int ctot = p.c1 + p.c2;
    const int t = threadIdx.x;
    const int ty = t >> 4, tx = t & 15;           // compute mapping: rows ty*4.., cols tx*4..
    const int ar = t >> 2, ac = (t & 3) * 4;      // A load mapping: row ar, channels ac..ac+3
    const int bk = t >> 4, bn = (t & 15) * 4;     // B load mapping: k row bk, cols bn..bn+3
    const bool vecA1 = (p.c1 % 4 == 0), vecA2 = (p.c2 % 4 == 0);
    const bool vecB = (p.cout % 4 == 0);

    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    if (t < FF_BM) {
        const int row = (m0 + t < M) ? (p.row_perm ? __ldg(p.row_perm + m0 + t) : m0 + t) : -1;
        row_s[t] = row;
        mask_s[t] = (row >= 0 && p.row_mask) ? __ldg(p.row_mask + row) : 0xffffffffu;
    }
    __syncthreads();
    for (int k = 0; k < p.kvol; ++k) {
        int my = -1;
        if (t < FF_BM) {
            const int row = row_s[t];
            if (row >= 0 && ((mask_s[t] >> k) & 1u)) my = p.nbr ? __ldg(p.nbr + (long long)k * p.nbr_stride + row) : row;
            idx_s[t] = my;
        }
        if (!__syncthreads_or(my >= 0)) continue;      // nobody in this tile has a neighbour at offset k
        const float* Wk = p.W + (long long)k * ctot * p.cout;

        for (int c0 = 0; c0 < ctot; c0 += FF_BK) {
            // ---- gather A chunk: rows idx_s[.] , channels c0 .. c0+15 -------------------------------
            {
                const int src = idx_s[ar];
                const int c = c0 + ac;
                float v[4] = {0.f, 0.f, 0.f, 0.f};
                if (src >= 0) {
                    if (c < p.c1) {
                        const float* rp = io.in1 + (long long)src * p.c1;
                        if (vecA1 && c + 3 < p.c1) {
                            float4 f = __ldg(reinterpret_cast<const float4*>(rp + c));
                            v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
                        } else {
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                int cj = c + j;
                                if (cj < p.c1) v[j] = __ldg(rp + cj);
                                else if (cj < ctot) v[j] = __ldg(io.in2 + (long long)src * p.c2 + (cj - p.c1));
                            }
                        }
                    } else if (c < ctot) {
                        const float* rp = io.in2 + (long long)src * p.c2;
                        const int cc = c - p.c1;
                        if (vecA2 && cc + 3 < p.c2) {
                            float4 f = __ldg(reinterpret_cast<const float4*>(rp + cc));
                            v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
                        } else {
#pragma unroll
                            for (int j = 0; j < 4; ++j) if (cc + j < p.c2) v[j] = __ldg(rp + cc + j);
                        }
                    }
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) As[ac + j][ar] = v[j];
            }
            // ---- B chunk: W[k][c0 + bk][n0 + bn ..] ---------------------------------------------------
            {
                const int c = c0 + bk, n = n0 + bn;
                float v[4] = {0.f, 0.f, 0.f, 0.f};
                if (c < ctot) {
                    const float* wp = Wk + (long long)c * p.cout + n;
                    if (vecB && n + 3 < p.cout) {
                        float4 f = __ldg(reinterpret_cast<const float4*>(wp));
                        v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
                    } else {
#pragma unroll
                        for (int j = 0; j < 4; ++j) if (n + j < p.cout) v[j] = __ldg(wp + j);
                    }
                }
                *reinterpret_cast<float4*>(&Bs[bk][bn]) = make_float4(v[0], v[1], v[2], v[3]);
            }
            __syncthreads();
#pragma unroll
            for (int kk = 0; kk < FF_BK; ++kk) {
                const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
                const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
                const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
            }
            __syncthreads();
        }
    }

    // ---- epilogue -------------------------------------------------------------------------------------
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int row = row_s[ty * 4 + i];
        if (row < 0) continue;
        const long long ro = (long long)row * p.cout;
        const float* gate_row = nullptr;
        if (io.gate_table) gate_row = io.gate_table + (long long)(io.gate_idx ? __ldg(io.gate_idx + row) : 0) * p.cout;
        float yv[4] = {0.f, 0.f, 0.f, 0.f}, gv[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int col = n0 + tx * 4 + j;
            if (col >= p.cout) continue;
            float y = acc[i][j];
            if (io.pre_add) y += __ldg(io.pre_add + ro + col);
            if (p.scale) y = fmaf(y, __ldg(p.scale + col), __ldg(p.shift + col));
            if (io.residual) y += __ldg(io.residual + ro + col);
            else if (io.residual_h) {
                const __half* rp = reinterpret_cast<const __half*>(io.residual_h) + 2 * ro + col;
                y += __half2float(__ldg(rp)) + __half2float(__ldg(rp + p.cout));
            }
            if (p.relu) y = fmaxf(y, 0.f);
            yv[j] = y;
            gv[j] = gate_row ? y * __ldg(gate_row + col) : y;
            if (io.out) io.out[ro + col] = y;
            if (io.out_gated) io.out_gated[ro + col] = gv[j];
        }
        if (n0 + tx * 4 + 3 < p.cout) {         // fp16 split companions (only for cout % 4 == 0 layers)
            if (io.out_h) tc::store_split4(io.out_h, row, p.cout, n0 + tx * 4, yv);
            if (io.out_gated_h) tc::store_split4(io.out_gated_h, row, p.cout, n0 + tx * 4, gv);
        }
    }
}

int lb2_spconv_ffma_launch(Lb2Handle* h, cudaStream_t s, const lb2_conv_desc* d) {
    FfmaParams p;
    p.c1 = d->c1; p.c2 = d->c2; p.cout = d->cout; p.kvol = d->kvol;
    p.W = d->weight; p.scale = d->scale; p.shift = d->shift; p.relu = d->relu;
    p.nbr = d->nbr; p.nbr_stride = d->nbr_stride; p.d_mout = d->d_mout; p.mout_cap = d->mout_cap; p.row_perm = d->row_perm; p.row_mask = d->row_mask;
    p.io[0] = d->io[0]; p.io[1] = d->io[d->npass > 1 ? 1 : 0];
    dim3 grid(cdiv(d->mout_cap, FF_BM), cdiv(d->cout, FF_BN), d->npass);
    k_spconv_ffma<<<grid, FF_THREADS, 0, s>>>(p);
    LB2_POST_LAUNCH(h, "k_spconv_ffma");
    return LB2_OK;
}

// Shared device/host helpers for the lidiff_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include "../../include/lidiff_b200.h"

struct Lb2Handle {
    int      device;
    int      num_sms;
    int64_t  launches;
    int32_t* d_status;      // device status word (bit0: coordinate out of key range)
    int      opt[LB2_OPT_COUNT];   // kernel-selection options (lb2_set_option)
    uint32_t configured;    // bit per kernel whose max-dynamic-shared-memory attribute has been set on this handle's device
    char     err[512];
};

// kernels that need more than 48 KB of dynamic shared memory: the attribute is per-device state, the handle is per device
enum { LB2_K_TC = 0, LB2_K_TC2, LB2_K_TC3, LB2_K_TC4, LB2_K_TC5_256, LB2_K_TC5_128, LB2_K_SCATTER, LB2_K_NN_TABLE };
template <class K>
static inline cudaError_t lb2_configure_smem(Lb2Handle* h, int bit, K kernel, int bytes) {
    if (h->configured & (1u << bit)) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess) h->configured |= 1u << bit;
    return e;
}

static inline int lb2_fail(Lb2Handle* h, int code, const char* fmt, const char* a = "", const char* b = "") {
    if (h) snprintf(h->err, sizeof(h->err), fmt, a, b);
    return code;
}

// after every launch: count it and surface launch-configuration errors (never synchronises)
#define LB2_POST_LAUNCH(h, name)                                                              \
    do {                                                                                      \
        (h)->launches++;                                                                      \
        cudaError_t e__ = cudaGetLastError();                                                 \
        if (e__ != cudaSuccess) return lb2_fail((h), LB2_ERR_CUDA, "%s: %s", name, cudaGetErrorString(e__)); \
    } while (0)

#define LB2_REQUIRE(h, cond, msg)                                                             \
    do { if (!(cond)) return lb2_fail((h), LB2_ERR_ARG, "bad argument: %s", msg); } while (0)

static inline unsigned cdiv(long long a, long long b) { return (unsigned)((a + b - 1) / b); }

// ---------------------------------------------------------------------------------------------------
// coordinate keys: 10 bit batch | 3 x 18 bit biased coordinate  (same packing as oracle/me_cpu.py)
// ---------------------------------------------------------------------------------------------------
#define LB2_AXIS_BITS 18
#define LB2_AXIS_OFF  (1 << (LB2_AXIS_BITS - 1))

__device__ __forceinline__ bool lb2_pack_key(int b, int x, int y, int z, unsigned long long& key) {
    unsigned ux = (unsigned)(x + LB2_AXIS_OFF), uy = (unsigned)(y + LB2_AXIS_OFF), uz = (unsigned)(z + LB2_AXIS_OFF);
    const unsigned lim = 1u << LB2_AXIS_BITS;
    bool ok = ((unsigned)b < 1024u) && ux < lim && uy < lim && uz < lim;
    if (!ok) {   // keep memory-safe: clamp; caller raises the status bit
        b = min(max(b, 0), 1023);
        ux = min(ux, lim - 1); uy = min(uy, lim - 1); uz = min(uz, lim - 1);
        if (x < -LB2_AXIS_OFF) ux = 0;
        if (y < -LB2_AXIS_OFF) uy = 0;
        if (z < -LB2_AXIS_OFF) uz = 0;
    }
    key = ((unsigned long long)b << (3 * LB2_AXIS_BITS)) | ((unsigned long long)ux << (2 * LB2_AXIS_BITS))
        | ((unsigned long long)uy << LB2_AXIS_BITS) | (unsigned long long)uz;
    return ok;
}

__device__ __forceinline__ unsigned lb2_hash(unsigned long long k) {
    k ^= k >> 33; k *= 0xff51afd7ed558ccdULL; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ULL; k ^= k >> 33;
    return (unsigned)k;
}

// row id of `key` in a built grid, or -1
__device__ __forceinline__ int lb2_grid_lookup(const unsigned long long* __restrict__ keys,
                                               const int* __restrict__ rows, unsigned mask,
                                               unsigned long long key) {
    unsigned slot = lb2_hash(key) & mask;
    while (true) {
        unsigned long long kk = __ldg(keys + slot);
        if (kk == key) return __ldg(rows + slot);
        if (kk == LB2_KEY_EMPTY) return -1;
        slot = (slot + 1) & mask;
    }
}

__device__ __forceinline__ int floor_to_multiple(int v, int ts) {
    // true floor division for negatives (ME stride maps, SURVEY.md App. A.3); ts is a power of two here
    int q = v / ts;
    if ((v % ts != 0) && ((v < 0) != (ts < 0))) --q;
    return q * ts;
}

// Stable LSD radix sort of the low key_bits (<= 64) bits of n 64-bit keys into a permutation (coords.cu; used by metrics.cu).
size_t lb2_sort_keys64_scratch_bytes(int n);
int lb2_sort_keys64(Lb2Handle* h, cudaStream_t s, const unsigned long long* keys, int n, int key_bits, int* perm, void* scratch);

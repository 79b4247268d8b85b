// Shared helpers for the xmap_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/xmap_b200.h"

namespace xmap {

extern thread_local char g_err[512];

inline int fail(const char *what, cudaError_t e, const char *file, int line) {
    snprintf(g_err, sizeof(g_err), "%s: %s (%s:%d)", what, cudaGetErrorString(e), file, line);
    return 1;
}
inline int fail_msg(const char *msg) {
    snprintf(g_err, sizeof(g_err), "%s", msg);
    return 2;
}

#define XMAP_CUDA(expr)                                                     \
    do {                                                                    \
        cudaError_t _e = (expr);                                            \
        if (_e != cudaSuccess) return ::xmap::fail(#expr, _e, __FILE__, __LINE__); \
    } while (0)
#define XMAP_LAUNCH_CHECK() XMAP_CUDA(cudaGetLastError())

// ---- entry formats (include/xmap_b200.h) ---------------------------------
constexpr uint32_t ITEM_MASK = 0x00FFFFFFu;
constexpr int GE_SHIFT = 29;
constexpr int EXP_MAX = 127;          // tcsr entries: 7-bit item exponent in bits 24-28 (low 5) and 30-31 (high 2)

__device__ __forceinline__ int ent_item(uint32_t w0) { return int(w0 & ITEM_MASK); }
__device__ __forceinline__ int ent_ge(uint32_t w0) { return int((w0 >> GE_SHIFT) & 1u); }
__device__ __forceinline__ int ent_exp(uint32_t w0) { return int(((w0 >> 24) & 31u) | ((w0 >> 25) & 0x60u)); }
__device__ __forceinline__ uint32_t exp_bits(uint32_t e) { return ((e & 31u) << 24) | ((e >> 5) << 30); }

// 2^e as a double, e in [-1022, 1023]
__device__ __forceinline__ double pow2d(int e) {
    return __longlong_as_double((long long)(1023 + e) << 52);
}

// streaming 8-byte load through the read-only path
__device__ __forceinline__ uint2 ld_ent(const uint64_t *p) {
    return __ldg(reinterpret_cast<const uint2 *>(p));
}

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

// total order used by every top-k in this library: larger |value| first,
// ties to the smaller tie-key (canonical item index).
__device__ __forceinline__ bool better(unsigned long long ka, int ta, unsigned long long kb, int tb) {
    return ka > kb || (ka == kb && ta < tb);
}

__device__ __forceinline__ unsigned long long abs_key(double v) {
    return (unsigned long long)__double_as_longlong(v) & 0x7FFFFFFFFFFFFFFFull;
}

// Histogram bin of a magnitude key (abs_key bits) for the top-k selections of sim.cu and xsim.cu:
// 16 sub-bins per octave for |v| in [2^-16, 2): bits 62..48 of the double, offset so that 2^-16 maps
// to bin 0; smaller values share bin 0, values >= 1 clamp to the top bin.
constexpr int SIM_BINS = 256;
__device__ __forceinline__ int sim_bin(unsigned long long key_bits) {
    const int hi = int((key_bits & 0x7FFFFFFFFFFFFFFFull) >> 48);       // 11 exponent bits + 4 mantissa bits
    const int base = (1023 - 16) << 4;
    return max(0, min(SIM_BINS - 1, hi - base));
}

// Philox4x32-10 (counter-based; Salmon et al. 2011): the generator of generate.cu and als.cu
__host__ __device__ inline void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)M0 * c[0], p1 = (uint64_t)M1 * c[2];
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
        k0 += W0; k1 += W1;
    }
}

// warp arg-best over (key, tie, pos); every lane gets the winner.
__device__ __forceinline__ void warp_argbest(unsigned long long &key, int &tie, int &pos) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        unsigned long long k2 = __shfl_xor_sync(0xffffffffu, key, off);
        int t2 = __shfl_xor_sync(0xffffffffu, tie, off);
        int p2 = __shfl_xor_sync(0xffffffffu, pos, off);
        bool take = (p2 >= 0) && (pos < 0 || better(k2, t2, key, tie));
        if (take) { key = k2; tie = t2; pos = p2; }
    }
}

}  // namespace xmap

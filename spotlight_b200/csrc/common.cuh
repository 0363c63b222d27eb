// Shared device/host helpers for the spotlight_b200 kernels (sm_100a).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/spotlight_b200.h"

void slb_set_error(const char* fmt, ...);
int slb_sms();

#define SLB_REQUIRE(cond, ...)                 \
    do {                                       \
        if (!(cond)) {                         \
            slb_set_error(__VA_ARGS__);        \
            return SLB_EINVAL;                 \
        }                                      \
    } while (0)

#define SLB_LAUNCH_CHECK(name)                                                   \
    do {                                                                         \
        cudaError_t e__ = cudaGetLastError();                                    \
        if (e__ != cudaSuccess) {                                                \
            slb_set_error("%s: launch failed: %s", name, cudaGetErrorString(e__)); \
            return SLB_ECUDA;                                                    \
        }                                                                        \
    } while (0)

static inline size_t slb_align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Carves sub-buffers out of a caller-owned workspace (256 B aligned).
struct WsCarver {
    char* base;
    size_t off;
    int64_t* log = nullptr;      // optional: [begin, end) byte offsets of every take, up to max_log
    int n_log = 0, max_log = 0;
    explicit WsCarver(void* p) : base(static_cast<char*>(p)), off(0) {}
    template <typename T>
    T* take(size_t count) {
        off = slb_align_up(off, 256);
        T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
        if (log && n_log < max_log) {
            log[2 * n_log] = static_cast<int64_t>(off);
            log[2 * n_log + 1] = static_cast<int64_t>(off + count * sizeof(T));
        }
        if (log) ++n_log;
        off += count * sizeof(T);
        return p;
    }
    size_t bytes() const { return slb_align_up(off, 256); }
};

#ifdef __CUDACC__

__device__ __forceinline__ float4 ldg4(const float* p) {
    return __ldg(reinterpret_cast<const float4*>(p));
}
__device__ __forceinline__ float4 ld4(const float* p) {
    return *reinterpret_cast<const float4*>(p);
}
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }

__device__ __forceinline__ float dot4(float4 a, float4 b) {
    return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w;
}
__device__ __forceinline__ void fma4(float4& acc, float g, float4 v) {
    acc.x = fmaf(g, v.x, acc.x);
    acc.y = fmaf(g, v.y, acc.y);
    acc.z = fmaf(g, v.z, acc.z);
    acc.w = fmaf(g, v.w, acc.w);
}

// Sum over the LPR consecutive lanes of a group (LPR power of two <= 32);
// every lane of the group gets the result.  `mask` names exactly the lanes
// that execute this call.
template <int LPR>
__device__ __forceinline__ float group_sum(float v, unsigned mask) {
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o);
    return v;
}

__device__ __forceinline__ unsigned group_mask(int lpr) {
    const int lane = threadIdx.x & 31;
    const unsigned m = lpr == 32 ? 0xffffffffu : ((1u << lpr) - 1u);
    return m << (lane & ~(lpr - 1));
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

// Block-wide sum; result valid in thread 0.  Fixed reduction tree -> deterministic.
template <int THREADS>
__device__ __forceinline__ float block_sum(float v, float* smem /* THREADS/32 floats */) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) smem[w] = v;
    __syncthreads();
    if (w == 0) {
        v = l < THREADS / 32 ? smem[l] : 0.f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    }
    return v;
}

// MurmurHash3_x86_32 of the 4 little-endian bytes of a 32-bit key
// (sklearn.utils.murmurhash3_32 on an int32 array; spotlight/layers.py:183).
__device__ __forceinline__ uint32_t murmur3_32(uint32_t k, uint32_t seed) {
    k *= 0xcc9e2d51u;
    k = (k << 15) | (k >> 17);
    k *= 0x1b873593u;
    uint32_t h = seed ^ k;
    h = (h << 13) | (h >> 19);
    h = h * 5u + 0xe6546b64u;
    h ^= 4u;
    h ^= h >> 16;
    h *= 0x85ebca6bu;
    h ^= h >> 13;
    h *= 0xc2b2ae35u;
    h ^= h >> 16;
    return h;
}

// BloomEmbedding row: int32(hash) floor-mod rows, 0 for the padding id
// (spotlight/layers.py:183-186).
__device__ __forceinline__ int64_t bloom_row(int64_t id, uint32_t seed, int64_t rows,
                                             int64_t padding_idx) {
    if (id == padding_idx) return 0;
    const int64_t h = static_cast<int32_t>(murmur3_32(static_cast<uint32_t>(id), seed));
    int64_t m = h % rows;
    if (m < 0) m += rows;
    return m;
}

// ---- row-wise optimizers shared by the MF and sequence kernels --------------------------------
// Adagrad step  w -= lr * g / (sqrt(s) + eps)  with MUFU-based sqrt and division (rsqrt 2 ulp,
// fast divide 2 ulp: ~5e-7 relative, far inside the 1e-5 parity budget; the IEEE sqrtf +
// division pair costs ~20 instructions per element and made the update kernels issue-bound).
__device__ __forceinline__ float adagrad_delta(float lr, float g, float s, float eps) {
    const float root = s > 0.f ? s * rsqrtf(s) : 0.f;
    return __fdividef(lr * g, root + eps);
}

struct OptV2 { int32_t opt; float lr, wd, eps; };

__device__ __forceinline__ void row_update(const OptV2& o, float4& w, float4& s, const float4& g0) {
    float gv[4] = {g0.x + o.wd * w.x, g0.y + o.wd * w.y, g0.z + o.wd * w.z, g0.w + o.wd * w.w};
    float wv[4] = {w.x, w.y, w.z, w.w};
    if (o.opt == SLB_OPT_SGD) {
#pragma unroll
        for (int q = 0; q < 4; ++q) wv[q] -= o.lr * gv[q];
    } else {
        float sv[4] = {s.x, s.y, s.z, s.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            sv[q] += gv[q] * gv[q];
            wv[q] -= adagrad_delta(o.lr, gv[q], sv[q], o.eps);
        }
        s = make_float4(sv[0], sv[1], sv[2], sv[3]);
    }
    w = make_float4(wv[0], wv[1], wv[2], wv[3]);
}

__device__ __forceinline__ void bias_update(const OptV2& o, float* bw, float* bs, float g) {
    const float gb = g + o.wd * *bw;
    if (o.opt == SLB_OPT_SGD) {
        *bw -= o.lr * gb;
    } else {
        const float sv = *bs + gb * gb;
        *bs = sv;
        *bw -= adagrad_delta(o.lr, gb, sv, o.eps);
    }
}

#endif  // __CUDACC__

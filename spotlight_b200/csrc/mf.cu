// Fused implicit-feedback matrix-factorisation training step for sm_100a.
//
// Replaces the loop body of ImplicitFactorizationModel.fit
// (spotlight/factorization/implicit.py:229-242): two BilinearNet forwards
// (spotlight/factorization/representations.py:80-91), one of
// pointwise/bpr/hinge/adaptive_hinge (spotlight/losses.py:40-50, 82-90,
// 115-124, 164-166) and loss.backward() (8x aten::embedding_dense_backward).
//
// One kernel per direction:
//   mf_fwd_tile_kernel (mf_fwd_kernel for adaptive hinge)
//                  gathers U[u], Q[i+], Q[i-] with 128-bit loads (LPR = D/4
//                  lanes per row, <=32), warp-shuffle dot, loss, d loss/d score,
//                  emits rank-1 gradient "terms" (user row, item row, g) and
//                  counts row occurrences with integer atomics.
//   mf_bwd_tile_kernel  one lane group per touched row: sums g * partner-row over
//                  the row's terms in ascending term order (deterministic), writes
//                  the gradient row once (dense or compact), or -- MODE 2 -- applies
//                  the row-wise optimizer to the user row in place.
// Between them: seg_tilesum/seg_scan + mf_fill_kernel build the inverted index
// (segindex.cuh).  mf_apply_kernel is the fused row-wise optimizer for item rows.
//
// Algorithmic HBM bytes per interaction (fp32, D = dim, R = 4D):
//   forward 3R + 3*4 + 3*8, backward re-reads 4R (partner rows), writes <= 3R.
#include <stdlib.h>

#include <algorithm>

#include "segindex.cuh"

namespace {

constexpr int MF_THREADS = 256;

struct MfDev {
    int64_t B;
    int64_t NB;  // normalising batch (== B on one GPU, the global batch when sharded)
    int64_t T;   // number of rank-1 terms (2B for a training step)
    const int64_t* users; const int64_t* items; const int64_t* negs;
    int32_t loss; int32_t n_neg;
    int64_t U, I; int32_t D;
    float* Wu; float* Wi; float* bu; float* bi;
    float* loss_out; float* pos_out; float* neg_out;
    // terms
    int32_t* t_a; int32_t* t_b; float* t_g;
    // loss reduction
    float* partial; int32_t* done;
    int32_t* err;
    SegIndex seg;
    // grads
    int32_t grad_mode;
    float* dWu; float* dWi; float* dbu; float* dbi;
    int64_t* urows; float* gWu; float* gbu;
    int64_t* irows; float* gWi; float* gbi;
    int32_t* compact_counts;
    int32_t opt; float lr, wd, eps;
    float* sWu; float* sWi; float* sbu; float* sbi;
    // hashed-table mode: bias grads are handled outside the segments; frozen rows get no grad
    int32_t no_bias;
    int64_t frozen_a, frozen_b;     // table rows that receive no gradient (-1 = none)
};

template <int LPR>
__device__ __forceinline__ float row_dot(const float* __restrict__ a, const float* __restrict__ b,
                                         int D, int gl, unsigned gmask) {
    float acc = 0.f;
    for (int c = gl * 4; c < D; c += LPR * 4) acc += dot4(ldg4(a + c), ldg4(b + c));
    return group_sum<LPR>(acc, gmask);
}

// d loss_b / d pos and d loss_b / d neg (unscaled by 1/B), and the loss term.
__device__ __forceinline__ void pair_loss(int loss, float p, float n, float& per, float& gp, float& gn) {
    if (loss == SLB_LOSS_BPR) {
        const float s = sigmoidf_(p - n);
        per = 1.0f - s;
        gp = -s * (1.0f - s);
        gn = -gp;
    } else if (loss == SLB_LOSS_POINTWISE) {
        const float sp = sigmoidf_(p), sn = sigmoidf_(n);
        per = (1.0f - sp) + sn;
        gp = -sp * (1.0f - sp);
        gn = sn * (1.0f - sn);
    } else {  // hinge / adaptive hinge on the selected negative
        const float z = n - p + 1.0f;
        per = fmaxf(z, 0.0f);
        const float act = z >= 0.0f ? 1.0f : 0.0f;  // clamp backward passes at the boundary
        gp = -act;
        gn = act;
    }
}

template <int LPR>
__global__ void __launch_bounds__(MF_THREADS) mf_fwd_kernel(MfDev a) {
    __shared__ float sh_red[MF_THREADS / 32];
    const int gl = threadIdx.x & (LPR - 1);
    const unsigned gmask = group_mask(LPR);
    constexpr int GROUPS = MF_THREADS / LPR;
    const int64_t gid = static_cast<int64_t>(blockIdx.x) * GROUPS + threadIdx.x / LPR;
    const int64_t gstride = static_cast<int64_t>(gridDim.x) * GROUPS;
    const float invB = 1.0f / static_cast<float>(a.NB);
    const int D = a.D;
    float lsum = 0.f;
    if (blockIdx.x == 0 && threadIdx.x == 0) a.seg.totals[3] = 0;     // hot-row list of the last step

    // every group runs the same number of iterations so shuffles stay converged
    const int64_t iters = (a.B + gstride - 1) / gstride;
    for (int64_t it = 0; it < iters; ++it) {
        const int64_t b = gid + it * gstride;
        const bool valid = b < a.B;
        const int64_t bb = valid ? b : 0;
        const int64_t u = a.users[bb], i = a.items[bb];
        bool bad = u < 0 || u >= a.U || i < 0 || i >= a.I;
        const int64_t uc = bad ? 0 : u, ic = bad ? 0 : i;
        const float* urow = a.Wu + uc * D;
        float p, n;
        int64_t nu, nj;
        if (a.loss != SLB_LOSS_ADAPTIVE_HINGE) {
            int64_t j = a.negs[bb];
            if (j < 0 || j >= a.I) { bad = true; j = 0; }
            const float* qi = a.Wi + ic * D;
            const float* qj = a.Wi + j * D;
            float dp = 0.f, dn = 0.f;
            for (int c = gl * 4; c < D; c += LPR * 4) {   // one trip for D <= 128
                const float4 u4 = ldg4(urow + c), i4 = ldg4(qi + c), j4 = ldg4(qj + c);
                dp += dot4(u4, i4);
                dn += dot4(u4, j4);
            }
            const float ub = __ldg(a.bu + uc);
            p = group_sum<LPR>(dp, gmask) + ub + __ldg(a.bi + ic);
            n = group_sum<LPR>(dn, gmask) + ub + __ldg(a.bi + j);
            nu = uc; nj = j;
            if (valid && gl == 0 && a.neg_out) a.neg_out[bb] = n;
        } else {
            // implicit.py:266-275: flat f = k*B + b is scored with users[f / n_neg]
            p = row_dot<LPR>(urow, a.Wi + ic * D, D, gl, gmask) + __ldg(a.bu + uc) + __ldg(a.bi + ic);
            n = -INFINITY; nu = 0; nj = 0;
            for (int k = 0; k < a.n_neg; ++k) {
                const int64_t f = static_cast<int64_t>(k) * a.B + bb;
                int64_t u2 = a.users[f / a.n_neg], j = a.negs[f];
                if (u2 < 0 || u2 >= a.U || j < 0 || j >= a.I) { bad = true; u2 = 0; j = 0; }
                const float nk = row_dot<LPR>(a.Wu + u2 * D, a.Wi + j * D, D, gl, gmask) +
                                 __ldg(a.bu + u2) + __ldg(a.bi + j);
                if (valid && gl == 0 && a.neg_out) a.neg_out[f] = nk;
                if (nk > n || k == 0) { n = nk; nu = u2; nj = j; }  // first arg-max
            }
        }
        if (valid && gl == 0) {
            if (bad) atomicExch(a.err, 1);
            float per, gp, gn;
            pair_loss(a.loss, p, n, per, gp, gn);
            lsum += per;
            gp *= invB; gn *= invB;
            if (bad) { gp = 0.f; gn = 0.f; }
            if (a.pos_out) a.pos_out[bb] = p;
            const int32_t t = static_cast<int32_t>(2 * bb);
            a.t_a[t] = static_cast<int32_t>(uc); a.t_b[t] = static_cast<int32_t>(ic); a.t_g[t] = gp;
            a.t_a[t + 1] = static_cast<int32_t>(nu); a.t_b[t + 1] = static_cast<int32_t>(nj); a.t_g[t + 1] = gn;
            if (gp != 0.f) { atomicAdd(a.seg.cnt + uc, 1); atomicAdd(a.seg.cnt + a.U + ic, 1); }
            if (gn != 0.f) { atomicAdd(a.seg.cnt + nu, 1); atomicAdd(a.seg.cnt + a.U + nj, 1); }
        }
    }

    // deterministic loss reduction: fixed tree per block, fixed order over blocks
    const float bsum = block_sum<MF_THREADS>(lsum, sh_red);
    __shared__ bool is_last;
    if (threadIdx.x == 0) {
        a.partial[blockIdx.x] = bsum;
        __threadfence();
        is_last = atomicAdd(a.done, 1) == static_cast<int>(gridDim.x) - 1;
    }
    __syncthreads();
    if (is_last && threadIdx.x < 32) {
        __threadfence();
        float v = 0.f;
        for (int k = threadIdx.x; k < static_cast<int>(gridDim.x); k += 32)
            v += *reinterpret_cast<volatile float*>(a.partial + k);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (threadIdx.x == 0) { *a.loss_out = v * invB; *a.done = 0; }
    }
}

// ---------------------------------------------------------------------------
// Tile-structured forward (pointwise / bpr / hinge).
//
// A warp owns a tile of 32 consecutive interactions.  Lane l loads the three
// ids and three biases of interaction l (coalesced 256-byte id loads, one DRAM
// round trip per 32 interactions instead of per interaction), then the warp
// walks the tile: each group of LPR lanes gathers the three rows of one
// interaction with 128-bit loads and reduces the two dots with xor shuffles;
// the results are handed back to the owning lane, which evaluates the loss,
// emits the two gradient terms with coalesced 8-byte stores and issues the
// integer row counts (32 lanes in parallel).
// ---------------------------------------------------------------------------
constexpr int MF_TILE_THREADS = 128;

template <int LPR, int LOSS, int TI, bool EX>
__global__ void __launch_bounds__(MF_TILE_THREADS) mf_fwd_tile_kernel(MfDev a) {
    __shared__ float sh_red[MF_TILE_THREADS / 32];
    __shared__ bool is_last;
    constexpr int GPW = 32 / LPR;            // groups per warp
    constexpr int ITERS = TI / GPW > 0 ? TI / GPW : 1;
    const int lane = threadIdx.x & 31;
    const int gl = lane & (LPR - 1);
    const int grp = lane / LPR;
    // EX: the row is exactly one 128-bit load per lane (D == 4 * LPR), so D is a compile-time
    // constant: no column loop, shifts for the row offsets (B200, D = 64: step 476 -> 431 us)
    const int D = EX ? LPR * 4 : a.D;
    const float invB = 1.0f / static_cast<float>(a.NB);
    const int64_t ntiles = (a.B + TI - 1) / TI;
    const int64_t wstride = static_cast<int64_t>(gridDim.x) * (MF_TILE_THREADS / 32);
    float lsum = 0.f;
    if (blockIdx.x == 0 && threadIdx.x == 0) a.seg.totals[3] = 0;     // hot-row list of the last step

    for (int64_t tile = static_cast<int64_t>(blockIdx.x) * (MF_TILE_THREADS / 32) + (threadIdx.x >> 5);
         tile < ntiles; tile += wstride) {
        const int64_t b = tile * TI + lane;
        const bool valid = lane < TI && b < a.B;
        int64_t u64 = 0, i64 = 0, j64 = 0;
        if (valid) { u64 = a.users[b]; i64 = a.items[b]; j64 = a.negs[b]; }
        const bool bad = u64 < 0 || u64 >= a.U || i64 < 0 || i64 >= a.I || j64 < 0 || j64 >= a.I;
        if (bad) { u64 = 0; i64 = 0; j64 = 0; }
        const int u = static_cast<int>(u64), i = static_cast<int>(i64), j = static_cast<int>(j64);
        const float ub = __ldg(a.bu + u), ib = __ldg(a.bi + i), jb = __ldg(a.bi + j);
        float dpm = 0.f, dnm = 0.f;
#pragma unroll 4
        for (int s = 0; s < ITERS; ++s) {
            const int src = (s * GPW + grp) % TI;       // TI < GPW: surplus groups recompute
            const int uu = __shfl_sync(0xffffffffu, u, src);
            const int ii = __shfl_sync(0xffffffffu, i, src);
            const int jj = __shfl_sync(0xffffffffu, j, src);
            const float* ur = a.Wu + static_cast<int64_t>(uu) * D;
            const float* qi = a.Wi + static_cast<int64_t>(ii) * D;
            const float* qj = a.Wi + static_cast<int64_t>(jj) * D;
            float dp = 0.f, dn = 0.f;
            for (int c = gl * 4; c < D; c += LPR * 4) {
                const float4 u4 = ldg4(ur + c), i4 = ldg4(qi + c), j4 = ldg4(qj + c);
                dp += dot4(u4, i4);
                dn += dot4(u4, j4);
            }
            dp = group_sum<LPR>(dp, 0xffffffffu);
            dn = group_sum<LPR>(dn, 0xffffffffu);
            const float tp = __shfl_sync(0xffffffffu, dp, (lane % GPW) * LPR);
            const float tn = __shfl_sync(0xffffffffu, dn, (lane % GPW) * LPR);
            if (lane / GPW == s) { dpm = tp; dnm = tn; }
        }
        if (valid) {
            const float p = dpm + ub + ib, n = dnm + ub + jb;
            float per, gp, gn;
            pair_loss(LOSS, p, n, per, gp, gn);
            lsum += per;
            gp *= invB; gn *= invB;
            if (bad) { atomicExch(a.err, 1); gp = 0.f; gn = 0.f; }
            if (a.pos_out) a.pos_out[b] = p;
            if (a.neg_out) a.neg_out[b] = n;
            *reinterpret_cast<int2*>(a.t_a + 2 * b) = make_int2(u, u);
            *reinterpret_cast<int2*>(a.t_b + 2 * b) = make_int2(i, j);
            *reinterpret_cast<float2*>(a.t_g + 2 * b) = make_float2(gp, gn);
            const int nu = (gp != 0.f) + (gn != 0.f);
            if (nu) atomicAdd(a.seg.cnt + u, nu);
            if (gp != 0.f) atomicAdd(a.seg.cnt + a.U + i, 1);
            if (gn != 0.f) atomicAdd(a.seg.cnt + a.U + j, 1);
        }
    }
    const float bsum = block_sum<MF_TILE_THREADS>(lsum, sh_red);
    if (threadIdx.x == 0) {
        a.partial[blockIdx.x] = bsum;
        __threadfence();
        is_last = atomicAdd(a.done, 1) == static_cast<int>(gridDim.x) - 1;
    }
    __syncthreads();
    if (is_last && threadIdx.x < 32) {
        __threadfence();
        float v = 0.f;
        for (int k = threadIdx.x; k < static_cast<int>(gridDim.x); k += 32)
            v += *reinterpret_cast<volatile float*>(a.partial + k);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (threadIdx.x == 0) { *a.loss_out = v * invB; *a.done = 0; }
    }
}

// ---------------------------------------------------------------------------
// Tile-structured backward: a warp owns 32 consecutive segments (touched rows).
// Lane l prefetches segment l's metadata and its first four terms (member ids
// sorted with a 5-comparator network, g, partner row index) -- the dependent
// load chain is paid once per 32 rows -- then each lane group accumulates
// g * partner_row for one segment per iteration with all row loads issued
// before the first FMA.  Longer segments sort through shared memory and
// prefetch their (g, partner) pairs lane-parallel before the row walk.
//
// MODE 0: every segment, gradients written (dense or compact).
// MODE 1: item segments only, compact gradients (fused-optimizer path, runs
//         first: it needs the *old* user rows).
// MODE 2: user segments only; the row-wise optimizer is applied in place
//         (partners are item rows, which MODE 1 no longer needs), so the user
//         gradient is never written to memory.
// ---------------------------------------------------------------------------
// Adagrad step  w -= lr * g / (sqrt(s) + eps)  with MUFU-based sqrt and division
// (rsqrt 2 ulp, fast divide 2 ulp: ~5e-7 relative, far inside the 1e-5 parity
// budget; the IEEE sqrtf + division pair costs ~20 instructions per element and
// made the update kernel issue-bound).
__device__ __forceinline__ void cswap(int& x, int& y) {
    const int lo = x < y ? x : y, hi = x < y ? y : x;
    x = lo; y = hi;
}

// Sorted (5..CAP-term) segments: once the partner row ids are known (lane-parallel, after
// the shared-memory sort) each lane asks L2 for its partners' rows, so the row walk that
// follows -- GEN_CHUNK rows in flight per lane -- runs at L2 rather than HBM latency.
// Measured at B = 524 288 (item rows average 10.5 terms): backward 301 -> 266 us.  The same
// prefetch for a segment's own weight / state rows, and for short segments' partners, was
// slower (+12 us), as were 16-row chunks and walking two user segments at once (spills).
#ifndef GEN_CHUNK
#define GEN_CHUNK 8
#endif
__device__ __forceinline__ void pf_row_l2(const float* row, int D) {
    const char* p = reinterpret_cast<const char*>(row);
    for (int o = 0; o < D * 4; o += 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + o));
}

// BWD_BULK (default 0; round-2 experiment, built only through profiles/run_variants.sh):
// the user-side kernel (MODE 2, exact row width) stages the weight / optimizer-state rows of a
// whole 32-segment tile in shared memory with one cp.async.bulk per row, completion on one
// mbarrier per warp -- 16 KB in flight per warp without holding a register.  NOT yet run on
// hardware: it compiles for sm_100a (SASS: UBLKCP) and is off in the shipped library.
#ifndef BWD_BULK
#define BWD_BULK 0
#endif
#if BWD_BULK
__device__ __forceinline__ uint32_t bulk_smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void bulk_bar_init(uint64_t* bar) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bulk_smem_u32(bar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void bulk_bar_expect(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bulk_smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(bulk_smem_u32(dst)), "l"(src), "r"(bytes), "r"(bulk_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_bar_wait(uint64_t* bar, uint32_t parity) {
    for (int spin = 0; spin < (1 << 26); ++spin) {
        uint32_t ok;
        asm volatile("{\n\t.reg .pred p;\n\t"
                     "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                     "selp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bulk_smem_u32(bar)), "r"(parity) : "memory");
        if (ok) return;
    }
    __trap();                               // a lost copy must not hang the GPU box
}
#endif

#ifndef BWD_MINB
#define BWD_MINB 6
#endif
#ifndef BWD_MINB1
#define BWD_MINB1 BWD_MINB
#endif
#ifndef BWD_FAST
#define BWD_FAST 4
#endif
template <int LPR, int MODE, int TI, bool EX>
__global__ void __launch_bounds__(MF_TILE_THREADS, MODE == 1 ? BWD_MINB1 : BWD_MINB) mf_bwd_tile_kernel(MfDev a) {
    constexpr int GPW = 32 / LPR;
    constexpr int ITERS = TI / GPW > 0 ? TI / GPW : 1;
    constexpr int WARPS = MF_TILE_THREADS / 32;
    constexpr int CAP = seg_sort_cap(LPR);
    __shared__ int32_t sh_all[WARPS * GPW * 4 * CAP];
    const int lane = threadIdx.x & 31;
    const int gl = lane & (LPR - 1);
    const int grp = lane / LPR;
    const unsigned gmask = group_mask(LPR);
    int32_t* sh = sh_all + ((threadIdx.x >> 5) * GPW + grp) * 4 * CAP;
    // EX: the row is exactly one 128-bit load per lane (D == 4 * LPR), so D is a compile-time
    // constant: no column loop, shifts for the row offsets (B200, D = 64: step 476 -> 431 us)
    const int D = EX ? LPR * 4 : a.D;
#if defined(BWD_OPT_CT)
    // round-2 experiment (off unless -DBWD_OPT_CT=<SLB_OPT_* value>): the optimizer kind is a
    // compile-time constant and weight decay is assumed zero, so the update's branches fold
    a.opt = BWD_OPT_CT;
    a.wd = 0.f;
#endif
#if BWD_BULK
    constexpr bool BULK = MODE == 2 && EX && TI == 32;
    constexpr int RB = LPR * 16;                                  // bytes per row
    extern __shared__ __align__(128) unsigned char bulk_rows[];   // WARPS x TI x 2 x RB
    __shared__ uint64_t bulk_bar[WARPS];
    unsigned char* my_rows = bulk_rows + (threadIdx.x >> 5) * (TI * 2 * RB);
    uint64_t* my_bar = &bulk_bar[threadIdx.x >> 5];
    uint32_t bulk_phase = 0;
    if (BULK) {
        if (lane == 0) bulk_bar_init(my_bar);
        __syncwarp();
    }
#endif
    const int nseg = a.seg.totals[0];
    const int nsegA = a.seg.totals[2];
    if (MODE != 2 && blockIdx.x == 0 && threadIdx.x == 0 && a.compact_counts) {
        a.compact_counts[0] = nsegA;
        a.compact_counts[1] = nseg - nsegA;
    }
    const int seg_lo = MODE == 1 ? nsegA : 0;
    const int seg_hi = MODE == 2 ? nsegA : nseg;
    const int32_t* __restrict__ t_a = a.t_a;
    const int32_t* __restrict__ t_b = a.t_b;
    const float* __restrict__ t_g = a.t_g;
    const int32_t* __restrict__ members = a.seg.members;
    const int ntiles = (seg_hi - seg_lo + TI - 1) / TI;
    const int wstride = gridDim.x * WARPS;

    for (int tile = blockIdx.x * WARPS + (threadIdx.x >> 5); tile < ntiles; tile += wstride) {
        const int sidx = seg_lo + tile * TI + lane;
        const bool valid = lane < TI && sidx < seg_hi;
        int start = 0, len = 0, row = 0;
        int p[BWD_FAST] = {};
        float g[BWD_FAST] = {};
#if BWD_BULK
        if (valid) {
            start = a.seg.seg_start[sidx];
            len = a.seg.seg_start[sidx + 1] - start;
            row = a.seg.seg_row[sidx];
        }
        if (BULK) {
            const bool stage = valid && len <= CAP && row != a.frozen_a;
            const unsigned who = __ballot_sync(0xffffffffu, stage);
            const uint32_t per = a.opt == SLB_OPT_ADAGRAD ? 2u * RB : 1u * RB;
            if (lane == 0) bulk_bar_expect(my_bar, __popc(who) * per);
            __syncwarp();
            if (stage) {
                bulk_g2s(my_rows + lane * 2 * RB, a.Wu + static_cast<int64_t>(row) * D, RB, my_bar);
                if (a.opt == SLB_OPT_ADAGRAD)
                    bulk_g2s(my_rows + lane * 2 * RB + RB, a.sWu + static_cast<int64_t>(row) * D, RB, my_bar);
            }
        }
#endif
        if (valid) {
            const bool isA = sidx < nsegA;
#if !BWD_BULK
            start = a.seg.seg_start[sidx];
            len = a.seg.seg_start[sidx + 1] - start;
            row = a.seg.seg_row[sidx];
#endif
            if (len <= BWD_FAST) {
                int m[BWD_FAST];
#pragma unroll
                for (int k = 0; k < BWD_FAST; ++k) m[k] = k < len ? members[start + k] : 0x7fffffff;
                cswap(m[0], m[1]);
                if (BWD_FAST == 4) { cswap(m[BWD_FAST - 2], m[BWD_FAST - 1]); cswap(m[0], m[BWD_FAST - 2]); cswap(m[1], m[BWD_FAST - 1]); cswap(m[1], m[BWD_FAST - 2]); }
                const int32_t* pidx = isA ? t_b : t_a;
#pragma unroll
                for (int k = 0; k < BWD_FAST; ++k)
                    if (k < len) { g[k] = t_g[m[k]]; p[k] = pidx[m[k]]; }
            }
        }
#if BWD_BULK
        if (BULK) { bulk_bar_wait(my_bar, bulk_phase); bulk_phase ^= 1u; }
#endif
        for (int it = 0; it < ITERS; ++it) {
            const int src = it * GPW + grp;               // >= TI only when TI < GPW: idle group
            const int s_len = __shfl_sync(0xffffffffu, len, src & 31);
            const int s_row = __shfl_sync(0xffffffffu, row, src & 31);
            const int s_start = __shfl_sync(0xffffffffu, start, src & 31);
            int sp[BWD_FAST];
            float sg[BWD_FAST];
#pragma unroll
            for (int k = 0; k < BWD_FAST; ++k) {
                sp[k] = __shfl_sync(0xffffffffu, p[k], src & 31);
                sg[k] = __shfl_sync(0xffffffffu, g[k], src & 31);
            }
            const int s = seg_lo + tile * TI + src;
            if (src >= TI || s >= seg_hi) continue;       // group-uniform
            const bool sA = s < nsegA;
            const float* ptab = sA ? a.Wi : a.Wu;
            const int64_t orow = sA ? s_row : s_row - a.U;
            if (orow == (sA ? a.frozen_a : a.frozen_b)) {              // padding row: no gradient
                if (MODE != 2 && gl == 0 && a.grad_mode == SLB_GRAD_COMPACT) {
                    if (sA) a.urows[s] = -1; else a.irows[s - nsegA] = -1;      // compact slot unused
                }
                continue;
            }
            if (s_len > CAP) continue;                                 // hot row: mf_bwd_long_kernel
            float* out = nullptr;
            if (MODE != 2) {
                if (a.grad_mode == SLB_GRAD_DENSE) out = (sA ? a.dWu : a.dWi) + orow * D;
                else out = sA ? a.gWu + static_cast<int64_t>(s) * D : a.gWi + static_cast<int64_t>(s - nsegA) * D;
            }
            float* wrow = MODE == 2 ? a.Wu + orow * D : nullptr;
            float* srow = (MODE == 2 && a.opt == SLB_OPT_ADAGRAD) ? a.sWu + orow * D : nullptr;
            float bacc = 0.f;

            int n_gen = 0;
            if (s_len > BWD_FAST && s_len <= CAP) {
                // sort member ids through shared memory, then prefetch (g, partner) lane-parallel
                int32_t* in = sh;
                int32_t* srt = sh + CAP;
                float* pg = reinterpret_cast<float*>(sh + 2 * CAP);
                int32_t* pp = sh + 3 * CAP;
                for (int i = gl; i < s_len; i += LPR) in[i] = members[s_start + i];
                __syncwarp(gmask);
                for (int i = gl; i < s_len; i += LPR) {
                    const int32_t m = in[i];
                    int r = 0;
                    for (int j = 0; j < s_len; ++j) r += in[j] < m;
                    srt[r] = m;
                }
                __syncwarp(gmask);
                const int32_t* pidx = sA ? t_b : t_a;
                for (int i = gl; i < s_len; i += LPR) {
                    const int32_t pr = pidx[srt[i]];
                    pg[i] = t_g[srt[i]];
                    pp[i] = pr;
                    if (!sA) pf_row_l2(ptab + static_cast<int64_t>(pr) * D, D);    // user rows: HBM; item rows sit in L2
                }
                __syncwarp(gmask);
                n_gen = s_len;
            }

            for (int c = gl * 4; c < D; c += LPR * 4) {
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                float b2 = 0.f;
                float4 w4 = make_float4(0.f, 0.f, 0.f, 0.f), s4 = w4;
#if BWD_BULK
                if (BULK) {
                    const unsigned char* staged = my_rows + src * 2 * RB + c * 4;
                    w4 = *reinterpret_cast<const float4*>(staged);
                    if (srow) s4 = *reinterpret_cast<const float4*>(staged + RB);
                } else
#endif
                if (MODE == 2) { w4 = ld4(wrow + c); if (srow) s4 = ld4(srow + c); }
                if (s_len <= BWD_FAST) {
                    float4 v[BWD_FAST];
#pragma unroll
                    for (int k = 0; k < BWD_FAST; ++k)
                        if (k < s_len) v[k] = ldg4(ptab + static_cast<int64_t>(sp[k]) * D + c);
#pragma unroll
                    for (int k = 0; k < BWD_FAST; ++k)
                        if (k < s_len) { fma4(acc, sg[k], v[k]); b2 += sg[k]; }
                } else if (n_gen) {
                    const float* pg = reinterpret_cast<const float*>(sh + 2 * CAP);
                    const int32_t* pp = sh + 3 * CAP;
                    int i = 0;
                    for (; i + GEN_CHUNK <= n_gen; i += GEN_CHUNK) {
                        float4 v[GEN_CHUNK];
#pragma unroll
                        for (int k = 0; k < GEN_CHUNK; ++k) v[k] = ldg4(ptab + static_cast<int64_t>(pp[i + k]) * D + c);
#pragma unroll
                        for (int k = 0; k < GEN_CHUNK; ++k) { fma4(acc, pg[i + k], v[k]); b2 += pg[i + k]; }
                    }
                    for (; i < n_gen; ++i) {
                        fma4(acc, pg[i], ldg4(ptab + static_cast<int64_t>(pp[i]) * D + c));
                        b2 += pg[i];
                    }
                }
                bacc = b2;
                if (MODE == 2) {
                    float gv[4] = {acc.x + a.wd * w4.x, acc.y + a.wd * w4.y, acc.z + a.wd * w4.z, acc.w + a.wd * w4.w};
                    float wv[4] = {w4.x, w4.y, w4.z, w4.w};
                    if (a.opt == SLB_OPT_SGD) {
#pragma unroll
                        for (int q = 0; q < 4; ++q) wv[q] -= a.lr * gv[q];
                    } else {
                        float sv[4] = {s4.x, s4.y, s4.z, s4.w};
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            sv[q] += gv[q] * gv[q];
                            wv[q] -= adagrad_delta(a.lr, gv[q], sv[q], a.eps);
                        }
                        st4(srow + c, make_float4(sv[0], sv[1], sv[2], sv[3]));
                    }
                    st4(wrow + c, make_float4(wv[0], wv[1], wv[2], wv[3]));
                } else {
                    st4(out + c, acc);
                }
            }
            if (n_gen) __syncwarp(gmask);        // scratch is reused by the next segment
            if (gl == 0 && MODE != 2 && a.grad_mode == SLB_GRAD_COMPACT) {
                if (sA) a.urows[s] = orow; else a.irows[s - nsegA] = orow;      // also for hashed tables (no_bias)
            }
            if (gl == 0 && !a.no_bias) {
                if (MODE == 2) {
                    float* bw = a.bu + orow;
                    const float gb = bacc + a.wd * *bw;
                    if (a.opt == SLB_OPT_SGD) {
                        *bw -= a.lr * gb;
                    } else {
                        float* bs = a.sbu + orow;
                        const float sv = *bs + gb * gb;
                        *bs = sv;
                        *bw -= adagrad_delta(a.lr, gb, sv, a.eps);
                    }
                } else if (a.grad_mode == SLB_GRAD_DENSE) {
                    if (sA) a.dbu[orow] = bacc; else a.dbi[orow] = bacc;
                } else {
                    if (sA) a.gbu[s] = bacc; else a.gbi[s - nsegA] = bacc;
                }
            }
        }
#if BWD_BULK
        if (BULK) __syncwarp();             // the next tile's copies overwrite the staged rows
#endif
    }
}

// ---------------------------------------------------------------------------
// Hot rows (more terms than the in-group sort capacity).  Their member lists were
// sorted by seg_sort_long_kernel; one CTA owns one hot row: each of its lane groups
// walks a contiguous chunk of the sorted members in order, the chunk partials are
// combined in chunk order.  Same MODE semantics as the tile kernel.
// ---------------------------------------------------------------------------
template <int LPR, int MODE>
__global__ void __launch_bounds__(256) mf_bwd_long_kernel(MfDev a) {
    constexpr int GROUPS = 256 / LPR;
    extern __shared__ float sh_part[];            // [GROUPS][D + 4]
    const int gl = threadIdx.x & (LPR - 1);
    const int gq = threadIdx.x / LPR;
    const int D = a.D;
    const int PS = D + 4;
    const int nlong = a.seg.totals[3];
    const int nsegA = a.seg.totals[2];
    const int32_t* __restrict__ members = a.seg.members;
    for (int li = blockIdx.x; li < nlong; li += gridDim.x) {
        const int s = a.seg.long_list[li];
        const bool sA = s < nsegA;
        if ((MODE == 1 && sA) || (MODE == 2 && !sA)) continue;          // block-uniform
        const int start = a.seg.seg_start[s];
        const int len = a.seg.seg_start[s + 1] - start;
        const int row = a.seg.seg_row[s];
        const int64_t orow = sA ? row : row - a.U;
        if (orow == (sA ? a.frozen_a : a.frozen_b)) {
            if (MODE != 2 && threadIdx.x == 0 && a.grad_mode == SLB_GRAD_COMPACT) {
                if (sA) a.urows[s] = -1; else a.irows[s - nsegA] = -1;
            }
            continue;
        }
        const float* ptab = sA ? a.Wi : a.Wu;
        const int32_t* pidx = sA ? a.t_b : a.t_a;
        const int chunk = (len + GROUPS - 1) / GROUPS;
        const int lo = min(gq * chunk, len), hi = min(lo + chunk, len);
        for (int c0 = 0; c0 < D; c0 += LPR * 4) {
            const int c = c0 + gl * 4;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            float b2 = 0.f;
            int i = lo;
            for (; i + 4 <= hi; i += 4) {
                int t[4]; float g[4]; float4 v[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) t[k] = members[start + i + k];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    g[k] = a.t_g[t[k]];
                    v[k] = c < D ? ldg4(ptab + static_cast<int64_t>(pidx[t[k]]) * D + c) : make_float4(0, 0, 0, 0);
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) { fma4(acc, g[k], v[k]); b2 += g[k]; }
            }
            for (; i < hi; ++i) {
                const int t = members[start + i];
                const float g = a.t_g[t];
                if (c < D) fma4(acc, g, ldg4(ptab + static_cast<int64_t>(pidx[t]) * D + c));
                b2 += g;
            }
            if (c < D) st4(sh_part + gq * PS + c, acc);
            if (gl == 0 && c0 == 0) sh_part[gq * PS + D] = b2;
        }
        __syncthreads();
        if (gq == 0) {
            float bacc = 0.f;
            for (int q = 0; q < GROUPS; ++q) bacc += sh_part[q * PS + D];
            for (int c = gl * 4; c < D; c += LPR * 4) {
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                for (int q = 0; q < GROUPS; ++q) {
                    const float4 p = ld4(sh_part + q * PS + c);
                    acc.x += p.x; acc.y += p.y; acc.z += p.z; acc.w += p.w;
                }
                if (MODE == 2) {
                    float* wrow = a.Wu + orow * D;
                    float4 w4 = ld4(wrow + c);
                    float gv[4] = {acc.x + a.wd * w4.x, acc.y + a.wd * w4.y, acc.z + a.wd * w4.z, acc.w + a.wd * w4.w};
                    float wv[4] = {w4.x, w4.y, w4.z, w4.w};
                    if (a.opt == SLB_OPT_SGD) {
#pragma unroll
                        for (int q = 0; q < 4; ++q) wv[q] -= a.lr * gv[q];
                    } else {
                        float* srow = a.sWu + orow * D;
                        float4 s4 = ld4(srow + c);
                        float sv[4] = {s4.x, s4.y, s4.z, s4.w};
#pragma unroll
                        for (int q = 0; q < 4; ++q) { sv[q] += gv[q] * gv[q]; wv[q] -= adagrad_delta(a.lr, gv[q], sv[q], a.eps); }
                        st4(srow + c, make_float4(sv[0], sv[1], sv[2], sv[3]));
                    }
                    st4(wrow + c, make_float4(wv[0], wv[1], wv[2], wv[3]));
                } else {
                    float* out;
                    if (a.grad_mode == SLB_GRAD_DENSE) out = (sA ? a.dWu : a.dWi) + orow * D;
                    else out = sA ? a.gWu + static_cast<int64_t>(s) * D : a.gWi + static_cast<int64_t>(s - nsegA) * D;
                    st4(out + c, acc);
                }
            }
            if (gl == 0 && MODE != 2 && a.grad_mode == SLB_GRAD_COMPACT) {
                if (sA) a.urows[s] = orow; else a.irows[s - nsegA] = orow;
            }
            if (gl == 0 && !a.no_bias) {
                if (MODE == 2) {
                    float* bw = a.bu + orow;
                    const float gb = bacc + a.wd * *bw;
                    if (a.opt == SLB_OPT_SGD) {
                        *bw -= a.lr * gb;
                    } else {
                        float* bs = a.sbu + orow;
                        const float sv = *bs + gb * gb;
                        *bs = sv;
                        *bw -= adagrad_delta(a.lr, gb, sv, a.eps);
                    }
                } else if (a.grad_mode == SLB_GRAD_DENSE) {
                    if (sA) a.dbu[orow] = bacc; else a.dbi[orow] = bacc;
                } else {
                    if (sA) a.gbu[s] = bacc; else a.gbi[s - nsegA] = bacc;
                }
            }
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256) mf_fill_kernel(MfDev a) {
    seg_rearm(a.seg);
    const int64_t T = a.T;
    const int64_t nth = static_cast<int64_t>(gridDim.x) * blockDim.x;
    for (int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; t < T; t += nth) {
        if (a.t_g[t] != 0.f) {
            seg_place(a.seg, a.t_a[t], static_cast<int32_t>(t));
            seg_place(a.seg, a.U + a.t_b[t], static_cast<int32_t>(t));
        }
    }
}

// Fused row-wise optimizer over the compact gradient rows (touched rows only).
// SGD:     W -= lr * (g + wd*W)
// Adagrad: g' = g + wd*W; state += g'^2; W -= lr * g' / (sqrt(state) + eps)
//          (torch.optim.Adagrad with lr_decay = 0, initial_accumulator_value = 0)
template <int LPR, int ITEMS_ONLY>
__global__ void __launch_bounds__(MF_THREADS) mf_apply_kernel(MfDev a) {
    constexpr int GROUPS = MF_THREADS / LPR;
    const int gl = threadIdx.x & (LPR - 1);
    const int gib = threadIdx.x / LPR;
    const int D = a.D;
    const int nseg = a.seg.totals[0];
    const int nsegA = a.seg.totals[2];
    for (int64_t s = (ITEMS_ONLY ? nsegA : 0) + static_cast<int64_t>(blockIdx.x) * GROUPS + gib; s < nseg;
         s += static_cast<int64_t>(gridDim.x) * GROUPS) {
        const bool isA = s < nsegA;
        const int64_t k = isA ? s : s - nsegA;
        const int64_t row = isA ? a.urows[k] : a.irows[k];
        if (row < 0) continue;                                       // frozen (padding) row: slot unused
        float* W = (isA ? a.Wu : a.Wi) + row * D;
        const float* G = (isA ? a.gWu : a.gWi) + k * D;
        float* S = a.opt == SLB_OPT_ADAGRAD ? (isA ? a.sWu : a.sWi) + row * D : nullptr;
        for (int c = gl * 4; c < D; c += LPR * 4) {
            float4 w = ld4(W + c);
            const float4 g0 = ld4(G + c);
            float gv[4] = {g0.x + a.wd * w.x, g0.y + a.wd * w.y, g0.z + a.wd * w.z, g0.w + a.wd * w.w};
            float wv[4] = {w.x, w.y, w.z, w.w};
            if (a.opt == SLB_OPT_SGD) {
#pragma unroll
                for (int q = 0; q < 4; ++q) wv[q] -= a.lr * gv[q];
            } else {
                float4 st = ld4(S + c);
                float sv[4] = {st.x, st.y, st.z, st.w};
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    sv[q] += gv[q] * gv[q];
                    wv[q] -= adagrad_delta(a.lr, gv[q], sv[q], a.eps);
                }
                st4(S + c, make_float4(sv[0], sv[1], sv[2], sv[3]));
            }
            st4(W + c, make_float4(wv[0], wv[1], wv[2], wv[3]));
        }
        if (gl == 0 && !a.no_bias) {
            float* bw = (isA ? a.bu : a.bi) + row;
            float g = (isA ? a.gbu : a.gbi)[k] + a.wd * *bw;
            if (a.opt == SLB_OPT_SGD) {
                *bw -= a.lr * g;
            } else {
                float* bs = (isA ? a.sbu : a.sbi) + row;
                const float sv = *bs + g * g;
                *bs = sv;
                *bw -= adagrad_delta(a.lr, g, sv, a.eps);
            }
        }
    }
}

constexpr int MF_MAX_GRID = 148 * 16;

#include "mf_v2.cuh"
#include "mf_adam.cuh"

template <int LPR>
__global__ void __launch_bounds__(MF_THREADS)
mf_scores_kernel(const float* __restrict__ Wu, const float* __restrict__ Wi,
                 const float* __restrict__ bu, const float* __restrict__ bi, int D,
                 const int64_t* __restrict__ users, const int64_t* __restrict__ items, int64_t n,
                 int user_broadcast, float* __restrict__ scores) {
    const int gl = threadIdx.x & (LPR - 1);
    const unsigned gmask = group_mask(LPR);
    constexpr int GROUPS = MF_THREADS / LPR;
    const int64_t gid = static_cast<int64_t>(blockIdx.x) * GROUPS + threadIdx.x / LPR;
    const int64_t gstride = static_cast<int64_t>(gridDim.x) * GROUPS;
    const int64_t iters = (n + gstride - 1) / gstride;
    for (int64_t it = 0; it < iters; ++it) {
        const int64_t b = gid + it * gstride;
        const bool valid = b < n;
        const int64_t bb = valid ? b : 0;
        const int64_t u = users[user_broadcast ? 0 : bb], i = items[bb];
        const float p = row_dot<LPR>(Wu + u * D, Wi + i * D, D, gl, gmask) + __ldg(bu + u) + __ldg(bi + i);
        if (valid && gl == 0) scores[bb] = p;
    }
}

// Terms from externally supplied score gradients (autograd of BilinearNet.forward).
__global__ void __launch_bounds__(256)
mf_terms_kernel(MfDev a, const float* __restrict__ gscores, int user_broadcast) {
    const int64_t nth = static_cast<int64_t>(gridDim.x) * blockDim.x;
    if (blockIdx.x == 0 && threadIdx.x == 0) a.seg.totals[3] = 0;
    for (int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; t < a.T; t += nth) {
        int64_t u = a.users[user_broadcast ? 0 : t], i = a.items[t];
        float g = gscores[t];
        if (u < 0 || u >= a.U || i < 0 || i >= a.I) { atomicExch(a.err, 1); u = 0; i = 0; g = 0.f; }
        a.t_a[t] = static_cast<int32_t>(u); a.t_b[t] = static_cast<int32_t>(i); a.t_g[t] = g;
        if (g != 0.f) { atomicAdd(a.seg.cnt + u, 1); atomicAdd(a.seg.cnt + a.U + i, 1); }
    }
}

// ---------------------------------------------------------------------------
// Forward for hashed (Bloom) tables: one lane group per interaction.  The user /
// item vectors are sums of H hashed rows (layers.py:240-241); the score is the dot
// of the two sums.  Emits Hu' * Hi' rank-1 terms per side (every pair of a hashed
// user row and a hashed item row), the id-space bias gradient terms, and the row
// counts.  Adaptive hinge keeps the reference's user/negative pairing
// (implicit.py:266-275).
// ---------------------------------------------------------------------------
struct BloomSpec {
    int Hu, Hi;                 // 0 = plain table
    int64_t pad_u, pad_i;
    uint32_t su[24], si[24];
    int64_t num_users, num_items;   // id spaces (bias tables)
    int64_t* ids_u2; int64_t* ids_i2;   // [2B] bias scatter ids
    float* g_u2; float* g_i2;           // [2B] bias scatter values
};

__device__ __forceinline__ int64_t hashed_row(int64_t id, int k, int H, const uint32_t* seeds,
                                              int64_t rows, int64_t pad) {
    return H == 0 ? id : bloom_row(id, seeds[k], rows, pad);
}

template <int LPR>
__device__ __forceinline__ float bloom_dot(const MfDev& a, const BloomSpec& h, int64_t u, int64_t i,
                                           int gl, unsigned gmask) {
    const int D = a.D;
    const int nu = h.Hu ? h.Hu : 1, ni = h.Hi ? h.Hi : 1;
    float acc = 0.f;
    for (int c = gl * 4; c < D; c += LPR * 4) {
        float4 us = make_float4(0, 0, 0, 0), is = make_float4(0, 0, 0, 0);
        for (int k = 0; k < nu; ++k) {
            const float4 v = ldg4(a.Wu + hashed_row(u, k, h.Hu, h.su, a.U, h.pad_u) * D + c);
            us.x += v.x; us.y += v.y; us.z += v.z; us.w += v.w;
        }
        for (int k = 0; k < ni; ++k) {
            const float4 v = ldg4(a.Wi + hashed_row(i, k, h.Hi, h.si, a.I, h.pad_i) * D + c);
            is.x += v.x; is.y += v.y; is.z += v.z; is.w += v.w;
        }
        acc += dot4(us, is);
    }
    return group_sum<LPR>(acc, gmask);
}

template <int LPR>
__global__ void __launch_bounds__(MF_THREADS) mf_fwd_bloom_kernel(MfDev a, const __grid_constant__ BloomSpec h) {
    __shared__ float sh_red[MF_THREADS / 32];
    __shared__ bool is_last;
    const int gl = threadIdx.x & (LPR - 1);
    const unsigned gmask = group_mask(LPR);
    constexpr int GROUPS = MF_THREADS / LPR;
    const int64_t gid = static_cast<int64_t>(blockIdx.x) * GROUPS + threadIdx.x / LPR;
    const int64_t gstride = static_cast<int64_t>(gridDim.x) * GROUPS;
    const float invB = 1.0f / static_cast<float>(a.NB);
    const int nu = h.Hu ? h.Hu : 1, ni = h.Hi ? h.Hi : 1;
    const int pairs = nu * ni;
    float lsum = 0.f;
    if (blockIdx.x == 0 && threadIdx.x == 0) a.seg.totals[3] = 0;
    const int64_t iters = (a.B + gstride - 1) / gstride;
    for (int64_t it = 0; it < iters; ++it) {
        const int64_t b = gid + it * gstride;
        const bool valid = b < a.B;
        const int64_t bb = valid ? b : 0;
        int64_t u = a.users[bb], i = a.items[bb];
        bool bad = u < 0 || u >= h.num_users || i < 0 || i >= h.num_items;
        if (bad) { u = 0; i = 0; }
        const float p = bloom_dot<LPR>(a, h, u, i, gl, gmask) + __ldg(a.bu + u) + __ldg(a.bi + i);
        float n = -INFINITY;
        int64_t nuid = u, njid = 0;
        for (int k = 0; k < a.n_neg; ++k) {
            const int64_t f = static_cast<int64_t>(k) * a.B + bb;
            int64_t u2 = a.loss == SLB_LOSS_ADAPTIVE_HINGE ? a.users[f / a.n_neg] : u;
            int64_t j = a.negs[f];
            if (u2 < 0 || u2 >= h.num_users || j < 0 || j >= h.num_items) { bad = true; u2 = 0; j = 0; }
            const float nk = bloom_dot<LPR>(a, h, u2, j, gl, gmask) + __ldg(a.bu + u2) + __ldg(a.bi + j);
            if (valid && gl == 0 && a.neg_out) a.neg_out[f] = nk;
            if (k == 0 || nk > n) { n = nk; nuid = u2; njid = j; }
        }
        if (valid && gl == 0) {
            if (bad) atomicExch(a.err, 1);
            float per, gp, gn;
            pair_loss(a.loss, p, n, per, gp, gn);
            lsum += per;
            gp *= invB; gn *= invB;
            if (bad) { gp = 0.f; gn = 0.f; }
            if (a.pos_out) a.pos_out[bb] = p;
            // user-bias gradient: when the negative is scored with the same user (every loss but
            // adaptive hinge) the two halves are emitted as ONE pair, so that bpr / hinge's
            // gp + gn = 0 is an exact zero (dropped downstream) and not a rounding residue of two
            // sums that Adagrad would turn into a full step
            if (nuid == u) {
                h.ids_u2[bb] = u; h.g_u2[bb] = gp + gn;
                h.ids_u2[a.B + bb] = u; h.g_u2[a.B + bb] = 0.f;
            } else {
                h.ids_u2[bb] = u; h.g_u2[bb] = gp;
                h.ids_u2[a.B + bb] = nuid; h.g_u2[a.B + bb] = gn;
            }
            h.ids_i2[bb] = i; h.g_i2[bb] = gp;
            h.ids_i2[a.B + bb] = njid; h.g_i2[a.B + bb] = gn;
            const int64_t t0 = bb * 2 * pairs;
            for (int side = 0; side < 2; ++side) {
                const float g = side ? gn : gp;
                const int64_t uu = side ? nuid : u, ii = side ? njid : i;
                for (int ku = 0; ku < nu; ++ku) {
                    const int32_t ra = static_cast<int32_t>(hashed_row(uu, ku, h.Hu, h.su, a.U, h.pad_u));
                    for (int ki = 0; ki < ni; ++ki) {
                        const int32_t rb = static_cast<int32_t>(hashed_row(ii, ki, h.Hi, h.si, a.I, h.pad_i));
                        const int64_t t = t0 + side * pairs + ku * ni + ki;
                        a.t_a[t] = ra; a.t_b[t] = rb; a.t_g[t] = g;
                        if (g != 0.f) { atomicAdd(a.seg.cnt + ra, 1); atomicAdd(a.seg.cnt + a.U + rb, 1); }
                    }
                }
            }
        }
    }
    const float bsum = block_sum<MF_THREADS>(lsum, sh_red);
    if (threadIdx.x == 0) {
        a.partial[blockIdx.x] = bsum;
        __threadfence();
        is_last = atomicAdd(a.done, 1) == static_cast<int>(gridDim.x) - 1;
    }
    __syncthreads();
    if (is_last && threadIdx.x < 32) {
        __threadfence();
        float v = 0.f;
        for (int k = threadIdx.x; k < static_cast<int>(gridDim.x); k += 32)
            v += *reinterpret_cast<volatile float*>(a.partial + k);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (threadIdx.x == 0) { *a.loss_out = v * invB; *a.done = 0; }
    }
}

struct MfLayout {
    int32_t* t_a; int32_t* t_b; float* t_g; float* partial; int32_t* done; int32_t* err;
    SegIndex seg;
    size_t bytes;
};

MfLayout mf_layout(void* base, int64_t B, int64_t U, int64_t I) {
    WsCarver ws(base);
    MfLayout l;
    // persistent (zero-at-rest) part first
    l.done = ws.take<int32_t>(8);
    l.err = l.done + 4;
    l.seg = seg_index_carve(ws, U + I, 4 * B);
    l.t_a = ws.take<int32_t>(2 * B);
    l.t_b = ws.take<int32_t>(2 * B);
    l.t_g = ws.take<float>(2 * B);
    l.partial = ws.take<float>(MF_MAX_GRID);
    l.bytes = ws.bytes();
    return l;
}

int lpr_for_dim(int D) {
    int l = D / 4;
    if (l >= 32) return 32;
    int p = 1;
    while (p < l) p <<= 1;
    return p;
}

#define DISPATCH_LPR(lpr, KERNEL, grid, block, stream, ...)                                   \
    switch (lpr) {                                                                           \
        case 1: KERNEL<1><<<grid, block, 0, stream>>>(__VA_ARGS__); break;                   \
        case 2: KERNEL<2><<<grid, block, 0, stream>>>(__VA_ARGS__); break;                   \
        case 4: KERNEL<4><<<grid, block, 0, stream>>>(__VA_ARGS__); break;                   \
        case 8: KERNEL<8><<<grid, block, 0, stream>>>(__VA_ARGS__); break;                   \
        case 16: KERNEL<16><<<grid, block, 0, stream>>>(__VA_ARGS__); break;                 \
        default: KERNEL<32><<<grid, block, 0, stream>>>(__VA_ARGS__); break;                 \
    }

#define DISPATCH_LPR2(lpr, KERNEL, P2, grid, block, stream, ...)                               \
    switch (lpr) {                                                                           \
        case 1: KERNEL<1, P2><<<grid, block, 0, stream>>>(__VA_ARGS__); break;               \
        case 2: KERNEL<2, P2><<<grid, block, 0, stream>>>(__VA_ARGS__); break;               \
        case 4: KERNEL<4, P2><<<grid, block, 0, stream>>>(__VA_ARGS__); break;               \
        case 8: KERNEL<8, P2><<<grid, block, 0, stream>>>(__VA_ARGS__); break;               \
        case 16: KERNEL<16, P2><<<grid, block, 0, stream>>>(__VA_ARGS__); break;             \
        default: KERNEL<32, P2><<<grid, block, 0, stream>>>(__VA_ARGS__); break;             \
    }

#define DISPATCH_LPR3_EX(L, KERNEL, P2, P3, grid, block, stream, a)                              \
    if ((a).D == (L) * 4) KERNEL<L, P2, P3, true><<<grid, block, 0, stream>>>(a);                \
    else KERNEL<L, P2, P3, false><<<grid, block, 0, stream>>>(a);
#define DISPATCH_LPR3(lpr, KERNEL, P2, P3, grid, block, stream, a)                               \
    switch (lpr) {                                                                               \
        case 1: KERNEL<1, P2, P3, false><<<grid, block, 0, stream>>>(a); break;                  \
        case 2: KERNEL<2, P2, P3, false><<<grid, block, 0, stream>>>(a); break;                  \
        case 4: KERNEL<4, P2, P3, false><<<grid, block, 0, stream>>>(a); break;                  \
        case 8: DISPATCH_LPR3_EX(8, KERNEL, P2, P3, grid, block, stream, a) break;               \
        case 16: DISPATCH_LPR3_EX(16, KERNEL, P2, P3, grid, block, stream, a) break;             \
        default: DISPATCH_LPR3_EX(32, KERNEL, P2, P3, grid, block, stream, a) break;             \
    }

template <int MODE>
void launch_long(int lpr, cudaStream_t st, const MfDev& a) {
    const size_t smem = static_cast<size_t>(256 / lpr) * (a.D + 4) * sizeof(float);
    switch (lpr) {
        case 1: mf_bwd_long_kernel<1, MODE><<<SEG_LONG_CTAS * 4, 256, smem, st>>>(a); break;
        case 2: mf_bwd_long_kernel<2, MODE><<<SEG_LONG_CTAS * 4, 256, smem, st>>>(a); break;
        case 4: mf_bwd_long_kernel<4, MODE><<<SEG_LONG_CTAS * 4, 256, smem, st>>>(a); break;
        case 8: mf_bwd_long_kernel<8, MODE><<<SEG_LONG_CTAS * 4, 256, smem, st>>>(a); break;
        case 16: mf_bwd_long_kernel<16, MODE><<<SEG_LONG_CTAS * 4, 256, smem, st>>>(a); break;
        default: mf_bwd_long_kernel<32, MODE><<<SEG_LONG_CTAS * 4, 256, smem, st>>>(a); break;
    }
}

bool v2_eligible(const slb_mf_step_args* x);

int validate(const slb_mf_step_args* x) {
    SLB_REQUIRE(x != nullptr, "mf_train_step: null args");
    SLB_REQUIRE(x->batch > 0, "mf_train_step: batch must be > 0");
    SLB_REQUIRE(x->dim >= 4 && x->dim % 4 == 0, "mf_train_step: dim must be a positive multiple of 4 (got %d)", x->dim);
    SLB_REQUIRE(x->loss >= 0 && x->loss <= 3, "mf_train_step: bad loss kind %d", x->loss);
    SLB_REQUIRE(x->n_neg >= 1, "mf_train_step: n_neg must be >= 1");
    SLB_REQUIRE(x->loss == SLB_LOSS_ADAPTIVE_HINGE || x->n_neg == 1, "mf_train_step: n_neg > 1 only for adaptive hinge");
    SLB_REQUIRE(x->num_users > 0 && x->num_items > 0, "mf_train_step: empty tables");
    SLB_REQUIRE(x->num_users + x->num_items < (1ll << 31) - SEG_SCAN_TILE, "mf_train_step: num_users + num_items must be < 2^31");
    SLB_REQUIRE(x->batch * 4 < (1ll << 31), "mf_train_step: batch too large");
    SLB_REQUIRE(x->users && x->items && x->negs && x->Wu && x->Wi && x->bu && x->bi && x->loss_out,
                "mf_train_step: null pointer");
    SLB_REQUIRE(x->workspace != nullptr, "mf_train_step: null workspace");
    if (x->grad_mode == SLB_GRAD_DENSE) {
        if (x->opt != SLB_OPT_NONE) {
            SLB_REQUIRE(x->opt_users_only, "mf_train_step: a fully fused optimizer needs compact grads");
            SLB_REQUIRE(x->dWi && x->dbi, "mf_train_step: users-only optimizer needs dWi/dbi for the item side");
        } else {
            SLB_REQUIRE(x->dWu && x->dWi && x->dbu && x->dbi, "mf_train_step: dense mode needs dWu/dWi/dbu/dbi");
        }
    } else {
        SLB_REQUIRE(x->grad_mode == SLB_GRAD_COMPACT, "mf_train_step: bad grad_mode");
        // the planned step updates both tables in place and never materialises the compact rows
        SLB_REQUIRE(v2_eligible(x) || (x->urows && x->gWu && x->gbu && x->irows && x->gWi && x->gbi && x->compact_counts),
                    "mf_train_step: compact mode needs urows/gWu/gbu/irows/gWi/gbi/compact_counts");
    }
    SLB_REQUIRE(x->opt >= SLB_OPT_NONE && x->opt <= SLB_OPT_ADAM, "mf_train_step: bad optimizer");
    if (x->opt == SLB_OPT_ADAM) {
        SLB_REQUIRE(x->grad_mode == SLB_GRAD_COMPACT && !x->opt_users_only, "mf_train_step: fused Adam needs compact grads");
        SLB_REQUIRE(x->state_Wu && x->state_Wi && x->state_bu && x->state_bi && x->state2_Wu && x->state2_Wi &&
                    x->state2_bu && x->state2_bi && x->last_u && x->last_i && x->adam_sched && x->adam_step >= 1,
                    "mf_train_step: fused Adam needs exp_avg / exp_avg_sq / last / schedule and adam_step >= 1");
    }
    if (x->opt == SLB_OPT_ADAGRAD) {
        SLB_REQUIRE(x->state_Wu && x->state_bu, "mf_train_step: adagrad needs state");
        SLB_REQUIRE(x->opt_users_only || (x->state_Wi && x->state_bi), "mf_train_step: adagrad needs item state");
    }
#if defined(BWD_OPT_CT)
    // experiment build: the first-generation user-side kernel folds this optimizer and zero decay in
    SLB_REQUIRE(x->opt == SLB_OPT_NONE || (x->opt == BWD_OPT_CT && x->weight_decay == 0.f),
                "mf_train_step: this build was compiled with -DBWD_OPT_CT=%d and weight_decay 0", BWD_OPT_CT);
#endif
    const size_t need = slb_mf_step_workspace_bytes(x->batch, x->n_neg, x->loss, x->num_users, x->num_items);
    if (x->workspace_bytes < need) {
        slb_set_error("mf_train_step: workspace too small (%zu < %zu)", x->workspace_bytes, need);
        return SLB_ENOSPC;
    }
    return SLB_OK;
}

int launch_step(const slb_mf_step_args* x, const int64_t* users, const int64_t* items,
                const int64_t* negs, int64_t B, float* loss_out, cudaStream_t st,
                int phases = 0x1f, int64_t step_idx = 0) {
    // layout is sized for x->batch so that short last batches reuse the same carve
    MfLayout l = mf_layout(x->workspace, x->batch, x->num_users, x->num_items);
    MfDev a;
    a.B = B; a.NB = x->norm_batch > 0 ? x->norm_batch : B; a.T = 2 * B; a.users = users; a.items = items; a.negs = negs;
    a.loss = x->loss; a.n_neg = x->n_neg;
    a.U = x->num_users; a.I = x->num_items; a.D = x->dim;
    a.Wu = x->Wu; a.Wi = x->Wi; a.bu = x->bu; a.bi = x->bi;
    a.loss_out = loss_out; a.pos_out = x->pos_out; a.neg_out = x->neg_out;
    a.t_a = l.t_a; a.t_b = l.t_b; a.t_g = l.t_g; a.partial = l.partial; a.done = l.done; a.err = l.err;
    a.seg = l.seg;
    a.seg.long_cap = seg_sort_cap(lpr_for_dim(x->dim));
    a.no_bias = 0; a.frozen_a = -1; a.frozen_b = -1;
    a.grad_mode = x->grad_mode;
    a.dWu = x->dWu; a.dWi = x->dWi; a.dbu = x->dbu; a.dbi = x->dbi;
    a.urows = x->urows; a.gWu = x->gWu; a.gbu = x->gbu;
    a.irows = x->irows; a.gWi = x->gWi; a.gbi = x->gbi;
    a.compact_counts = x->compact_counts;
    a.opt = x->opt; a.lr = x->lr; a.wd = x->weight_decay; a.eps = x->eps;
    a.sWu = x->state_Wu; a.sWi = x->state_Wi; a.sbu = x->state_bu; a.sbi = x->state_bi;

    const int lpr = lpr_for_dim(x->dim);
    const int groups = MF_THREADS / lpr;
    const int sms = slb_sms();
    int64_t want = (B + groups - 1) / groups;
    int grid = static_cast<int>(want < static_cast<int64_t>(sms) * 8 ? want : static_cast<int64_t>(sms) * 8);
    if (grid < 1) grid = 1;
    if (grid > MF_MAX_GRID) grid = MF_MAX_GRID;
    if ((phases & 1) && x->opt == SLB_OPT_ADAM) {
        // lazy-exact Adam: the rows this minibatch reads become current (through step t-1) first
        AdamDev o = {x->beta1, x->beta2, x->one_minus_beta1, x->one_minus_beta2, x->eps, x->weight_decay, x->adam_sched,
                     static_cast<int32_t>(x->adam_step + step_idx)};
        const int64_t refs = (2 + x->n_neg) * B;
        const int64_t pw = (refs + groups - 1) / groups;
        const int pgrid = static_cast<int>(pw < static_cast<int64_t>(sms) * 8 ? (pw < 1 ? 1 : pw) : static_cast<int64_t>(sms) * 8);
        DISPATCH_LPR(lpr, mf_adam_prepass_kernel, pgrid, MF_THREADS, st, a, o, x->state2_Wu, x->state2_Wi,
                     x->state2_bu, x->state2_bi, x->last_u, x->last_i);
        SLB_LAUNCH_CHECK("mf_adam_prepass_kernel");
    }
    if (phases & 1) {
        if (x->loss == SLB_LOSS_ADAPTIVE_HINGE) {
            DISPATCH_LPR(lpr, mf_fwd_kernel, grid, MF_THREADS, st, a);
        } else {
            // small batches: 8-interaction tiles so that every SM still gets ~36 warps
            const bool small = B < static_cast<int64_t>(sms) * 36 * 32;
            const int ti = small ? 8 : 32;
            int64_t tw = ((B + ti - 1) / ti + 3) / 4;
            int tgrid = static_cast<int>(tw < MF_MAX_GRID ? tw : MF_MAX_GRID);
#define FWD_TILE(L)                                                                             \
    if (small) { DISPATCH_LPR3(lpr, mf_fwd_tile_kernel, L, 8, tgrid, MF_TILE_THREADS, st, a); } \
    else { DISPATCH_LPR3(lpr, mf_fwd_tile_kernel, L, 32, tgrid, MF_TILE_THREADS, st, a); }
            switch (x->loss) {
                case SLB_LOSS_POINTWISE: FWD_TILE(SLB_LOSS_POINTWISE); break;
                case SLB_LOSS_BPR: FWD_TILE(SLB_LOSS_BPR); break;
                default: FWD_TILE(SLB_LOSS_HINGE); break;
            }
        }
        SLB_LAUNCH_CHECK("mf_fwd_kernel");
    }
    if (phases & 2) {
        seg_scan_launch(a.seg, a.U, st);
        SLB_LAUNCH_CHECK("seg_scan_kernel");
    }
    int fgrid = static_cast<int>((2 * B + 255) / 256);
    if (fgrid > sms * 8) fgrid = sms * 8;
    if (phases & 4) {
        mf_fill_kernel<<<fgrid, 256, 0, st>>>(a);
        SLB_LAUNCH_CHECK("mf_fill_kernel");
        seg_sort_long_kernel<<<SEG_LONG_CTAS, 256, 0, st>>>(a.seg);     // no-op unless hot rows exist
        SLB_LAUNCH_CHECK("seg_sort_long_kernel");
    }
    int64_t bwant = (2 * B + groups - 1) / groups;
    int bgrid = static_cast<int>(bwant < static_cast<int64_t>(sms) * 8 ? bwant : static_cast<int64_t>(sms) * 8);
    // small batches: 8-segment tiles so that every SM still gets enough warps
    const bool bsmall = 2 * B < static_cast<int64_t>(sms) * 24 * 32;
    const int bti = bsmall ? 8 : 32;
    const int64_t tw = ((2 * B + bti - 1) / bti + 3) / 4;     // upper bound on segment tiles
    const int tgrid = static_cast<int>(tw < static_cast<int64_t>(sms) * 16 ? tw : static_cast<int64_t>(sms) * 16);
    const int blpr = lpr;
#define BWD_TILE(MODE)                                                                               \
    if (bsmall) { DISPATCH_LPR3(blpr, mf_bwd_tile_kernel, MODE, 8, tgrid, MF_TILE_THREADS, st, a); } \
    else { DISPATCH_LPR3(blpr, mf_bwd_tile_kernel, MODE, 32, tgrid, MF_TILE_THREADS, st, a); }
    if (x->opt == SLB_OPT_NONE || x->opt == SLB_OPT_ADAM) {
        if (phases & 8) {
            BWD_TILE(0);
            SLB_LAUNCH_CHECK("mf_bwd_tile_kernel");
            launch_long<0>(lpr, st, a);
            SLB_LAUNCH_CHECK("mf_bwd_long_kernel");
        }
        if (x->opt == SLB_OPT_ADAM && (phases & 16)) {
            // lazy-exact Adam on the touched rows (mf_adam.cuh): a.sW* hold exp_avg
            AdamDev o = {x->beta1, x->beta2, x->one_minus_beta1, x->one_minus_beta2, x->eps, x->weight_decay, x->adam_sched,
                         static_cast<int32_t>(x->adam_step + step_idx)};
            DISPATCH_LPR(lpr, mf_adam_apply_kernel, bgrid, MF_THREADS, st, a, o, x->state2_Wu, x->state2_Wi,
                         x->state2_bu, x->state2_bi, x->last_u, x->last_i);
            SLB_LAUNCH_CHECK("mf_adam_apply_kernel");
        }
    } else {
        // fused optimizer: item gradients first (they read the old user rows), then
        // the user pass updates its rows in place, then the item rows are updated
        if (phases & 8) {
            BWD_TILE(1);
            SLB_LAUNCH_CHECK("mf_bwd_tile_kernel<items>");
            launch_long<1>(lpr, st, a);
            SLB_LAUNCH_CHECK("mf_bwd_long_kernel<items>");
#if BWD_BULK
            if (lpr == 16 && a.D == 64 && !bsmall) {
                auto kern = mf_bwd_tile_kernel<16, 2, 32, true>;
                constexpr int BULK_SMEM = (MF_TILE_THREADS / 32) * 32 * 2 * 256;
                static bool configured = false;
                if (!configured) {
                    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, BULK_SMEM);
                    configured = true;
                }
                kern<<<tgrid, MF_TILE_THREADS, BULK_SMEM, st>>>(a);
            } else
#endif
            { BWD_TILE(2); }
            SLB_LAUNCH_CHECK("mf_bwd_tile_kernel<users+opt>");
            launch_long<2>(lpr, st, a);
            SLB_LAUNCH_CHECK("mf_bwd_long_kernel<users+opt>");
        }
        if ((phases & 16) && !x->opt_users_only) {
            DISPATCH_LPR2(lpr, mf_apply_kernel, 1, bgrid, MF_THREADS, st, a);
            SLB_LAUNCH_CHECK("mf_apply_kernel<items>");
        }
    }
    return SLB_OK;
}


// ---------------------------------------------------------------------------
// Planned two-kernel step (mf_v2.cuh): workspace layout and launches.
// ---------------------------------------------------------------------------
struct V2Layout {
    PlanDev plan[2];
    StepV2 st;
    size_t bytes;
};

// B is the layout's capacity; a step over fewer interactions passes its own count to the kernels.
// `log` (optional) receives the [begin, end) byte offsets of every array taken.
V2Layout v2_layout(void* base, int64_t B, int64_t U, int64_t I, int D, WsCarver* log = nullptr) {
    WsCarver own(base);
    WsCarver& ws = log ? *log : own;
    V2Layout l;
    const int64_t R = U + I;
    const int64_t Rpad = (R + SEG_SCAN_TILE - 1) / SEG_SCAN_TILE * SEG_SCAN_TILE;
    l.st.done = ws.take<int32_t>(8);
    int32_t* cnt[2] = {ws.take<int32_t>(Rpad), ws.take<int32_t>(Rpad)};
    for (int k = 0; k < 2; ++k) {
        PlanDev& p = l.plan[k];
        SegIndex& s = p.seg;
        s.R = R;
        s.Rpad = Rpad;
        s.ntiles = s.Rpad / SEG_SCAN_TILE;
        s.Tmax = 3 * B;
        s.cnt = cnt[k];
        s.off = ws.take<int32_t>(s.Rpad);
        s.sid = ws.take<int32_t>(s.Rpad);
        s.status = ws.take<unsigned long long>(s.ntiles);
        s.ticket = ws.take<int32_t>(8);
        s.totals = s.ticket + 4;
        s.seg_row = ws.take<int32_t>(3 * B + 1);
        s.seg_start = ws.take<int32_t>(3 * B + 2);
        s.long_list = ws.take<int32_t>(3 * B / 16 + 2);
        s.members = nullptr; s.long_tmp = nullptr; s.long_bits = nullptr; s.long_words = 0;
        s.long_cap = 0;
        p.mu = ws.take<URec>(B + 1);
        p.mi = ws.take<IRec>(2 * B + 1);
        p.mu_tmp = ws.take<URec>(B + 1);
        p.mi_tmp = ws.take<IRec>(2 * B + 1);
        p.words = (2 * B + 31) / 32;
        p.bits = ws.take<uint32_t>(static_cast<size_t>(SEG_LONG_CTAS) * 2 * p.words);
        p.slot = ws.take<int32_t>(3 * B);
        p.multi = ws.take<int32_t>(3 * B / 2 + 1);
        p.nmulti = ws.take<int32_t>(8);
        p.B = B; p.U = U; p.I = I;
        p.err = nullptr; p.users = nullptr; p.items = nullptr; p.negs = nullptr;
    }
    l.st.t_g = ws.take<float>(2 * B);
    l.st.stash = ws.take<float>(static_cast<size_t>(B) * D);
    l.st.partial = ws.take<float>(MF_MAX_GRID);
    l.st.partial_long = ws.take<float>(SEG_LONG_CTAS * 4);
    l.bytes = ws.bytes();
    return l;
}

bool v2_dim_ok(int D) { return D == 8 || D == 16 || D == 32 || D == 64 || D == 128; }

bool v2_eligible(const slb_mf_step_args* x) {
    if (x->fused_workspace == nullptr || x->loss == SLB_LOSS_ADAPTIVE_HINGE || x->opt == SLB_OPT_NONE ||
        x->opt == SLB_OPT_ADAM ||
        !v2_dim_ok(x->dim) || x->pos_out != nullptr || x->neg_out != nullptr)
        return false;
    // single GPU: both tables updated in place (compact mode, nothing materialised); sharded item
    // rows: users updated in place, the dense item gradient handed out (dWi / dbi)
    if (x->opt_users_only) return x->grad_mode == SLB_GRAD_DENSE && x->dWi != nullptr && x->dbi != nullptr;
    return x->grad_mode == SLB_GRAD_COMPACT;
}

int v2_launch_plan(const slb_mf_step_args* x, PlanDev p, int32_t* err, const int64_t* users, const int64_t* items,
                   const int64_t* negs, int64_t B, cudaStream_t st) {
    p.B = B; p.users = users; p.items = items; p.negs = negs; p.err = err;
    p.seg.long_cap = seg_sort_cap(lpr_for_dim(x->dim));
    const int64_t cap = static_cast<int64_t>(slb_sms()) * PLAN_GRID_PER_SM;
    const int g = static_cast<int>(std::min<int64_t>((B + 255) / 256, cap));
    plan_count_kernel<<<g, 256, 0, st>>>(p);
    SLB_LAUNCH_CHECK("plan_count_kernel");
    plan_scan_kernel<<<static_cast<unsigned>(p.seg.ntiles), SEG_SCAN_THREADS, 0, st>>>(p);
    SLB_LAUNCH_CHECK("plan_scan_kernel");
    plan_fill_kernel<<<g, 256, 0, st>>>(p);
    SLB_LAUNCH_CHECK("plan_fill_kernel");
    // sort: hot-row blocks first, then enough warps for the longest possible `multi` list, capped
    const int64_t tiles = ((3 * B / 2 + 1 + 31) / 32 + PLAN_SORT_THREADS / 32 - 1) / (PLAN_SORT_THREADS / 32);
    const int sg = SEG_LONG_CTAS + static_cast<int>(std::min<int64_t>(tiles, 2 * cap));
    plan_sort_kernel<<<sg, PLAN_SORT_THREADS, 0, st>>>(p, p.seg.long_cap);
    SLB_LAUNCH_CHECK("plan_sort_kernel");
    return SLB_OK;
}

MfDev v2_dev(const slb_mf_step_args* x, int64_t B, float* loss_out) {
    MfDev a = {};
    a.B = B; a.NB = x->norm_batch > 0 ? x->norm_batch : B; a.T = 2 * B;
    a.loss = x->loss; a.n_neg = 1;
    a.U = x->num_users; a.I = x->num_items; a.D = x->dim;
    a.Wu = x->Wu; a.Wi = x->Wi; a.bu = x->bu; a.bi = x->bi;
    a.loss_out = loss_out;
    a.opt = x->opt; a.lr = x->lr; a.wd = x->weight_decay; a.eps = x->eps;
    a.sWu = x->state_Wu; a.sWi = x->state_Wi; a.sbu = x->state_bu; a.sbi = x->state_bi;
    a.frozen_a = -1; a.frozen_b = -1;
    if (x->opt_users_only) { a.dWi = x->dWi; a.dbi = x->dbi; }      // item kernel hands the gradient out
    return a;
}

template <int LPR, int LOSS>
void v2_user_launch(const MfDev& a, const PlanDev& p, const StepV2& v, bool small, int grid, cudaStream_t st) {
    const size_t smem = static_cast<size_t>(256 / LPR) * (LPR * 4 + 4) * sizeof(float);
    mf_user_long_kernel<LPR, LOSS><<<SEG_LONG_CTAS * 4, 256, smem, st>>>(a, p, v);
    if (small) mf_user_kernel<LPR, 1, LOSS, 8><<<grid, MF_TILE_THREADS, 0, st>>>(a, p, v, SEG_LONG_CTAS * 4);
    else if (V2_UVPL == 2 && LPR >= 16) {
        // the BASELINE dims (64, 128): two 128-bit pieces per lane, half the lanes per row
        mf_user_kernel<LPR / 2, 2, LOSS, 32><<<grid, MF_TILE_THREADS, 0, st>>>(a, p, v, SEG_LONG_CTAS * 4);
    } else mf_user_kernel<LPR, 1, LOSS, 32><<<grid, MF_TILE_THREADS, 0, st>>>(a, p, v, SEG_LONG_CTAS * 4);
}

template <int LPR>
void v2_user_dispatch(const MfDev& a, const PlanDev& p, const StepV2& v, bool small, int grid, cudaStream_t st) {
    switch (a.loss) {
        case SLB_LOSS_POINTWISE: v2_user_launch<LPR, SLB_LOSS_POINTWISE>(a, p, v, small, grid, st); break;
        case SLB_LOSS_BPR: v2_user_launch<LPR, SLB_LOSS_BPR>(a, p, v, small, grid, st); break;
        default: v2_user_launch<LPR, SLB_LOSS_HINGE>(a, p, v, small, grid, st); break;
    }
}

template <int LPR>
void v2_item_launch(const MfDev& a, const PlanDev& p, const StepV2& v, bool small, int grid, cudaStream_t st) {
    const size_t smem = static_cast<size_t>(256 / LPR) * (LPR * 4 + 4) * sizeof(float);
    mf_item_long_kernel<LPR><<<SEG_LONG_CTAS * 4, 256, smem, st>>>(a, p, v);
    if (small) mf_item_kernel<LPR, 8><<<grid, MF_TILE_THREADS, 0, st>>>(a, p, v);
    else mf_item_kernel<LPR, 32><<<grid, MF_TILE_THREADS, 0, st>>>(a, p, v);
}

// phases: 1 plan, 2 user kernels (forward + user update), 4 item kernels
int v2_launch_step(const slb_mf_step_args* x, const V2Layout& l, int slot, int32_t* err, const int64_t* users,
                   const int64_t* items, const int64_t* negs, int64_t B, float* loss_out, cudaStream_t st,
                   int phases) {
    if (phases & 1) {
        const int rc = v2_launch_plan(x, l.plan[slot], err, users, items, negs, B, st);
        if (rc != SLB_OK) return rc;
    }
    PlanDev p = l.plan[slot];
    p.B = B; p.users = users; p.items = items; p.negs = negs; p.err = err;
    p.seg.long_cap = seg_sort_cap(lpr_for_dim(x->dim));
    const MfDev a = v2_dev(x, B, loss_out);
    const int sms = slb_sms();
    const int lpr = x->dim / 4;
    if (phases & 2) {
        const bool small = B < static_cast<int64_t>(sms) * 24 * 32;
        const int64_t tw = ((B + (small ? 8 : 32) - 1) / (small ? 8 : 32) + 3) / 4;
        const int grid = static_cast<int>(tw < MF_MAX_GRID ? (tw < 1 ? 1 : tw) : MF_MAX_GRID);
        switch (lpr) {
            case 2: v2_user_dispatch<2>(a, p, l.st, small, grid, st); break;
            case 4: v2_user_dispatch<4>(a, p, l.st, small, grid, st); break;
            case 8: v2_user_dispatch<8>(a, p, l.st, small, grid, st); break;
            case 16: v2_user_dispatch<16>(a, p, l.st, small, grid, st); break;
            default: v2_user_dispatch<32>(a, p, l.st, small, grid, st); break;
        }
        SLB_LAUNCH_CHECK("mf_user_kernel");
    }
    if (phases & 4) {
        const bool small = 2 * B < static_cast<int64_t>(sms) * 24 * 32;
        const int64_t tw = ((2 * B + (small ? 8 : 32) - 1) / (small ? 8 : 32) + 3) / 4;
        const int grid = static_cast<int>(tw < static_cast<int64_t>(sms) * 16 ? (tw < 1 ? 1 : tw) : static_cast<int64_t>(sms) * 16);
        switch (lpr) {
            case 2: v2_item_launch<2>(a, p, l.st, small, grid, st); break;
            case 4: v2_item_launch<4>(a, p, l.st, small, grid, st); break;
            case 8: v2_item_launch<8>(a, p, l.st, small, grid, st); break;
            case 16: v2_item_launch<16>(a, p, l.st, small, grid, st); break;
            default: v2_item_launch<32>(a, p, l.st, small, grid, st); break;
        }
        SLB_LAUNCH_CHECK("mf_item_kernel");
    }
    return SLB_OK;
}

int v2_check_ws(const slb_mf_step_args* x) {
    const size_t need = v2_layout(nullptr, x->batch, x->num_users, x->num_items, x->dim).bytes;
    if (x->fused_workspace_bytes < need) {
        slb_set_error("mf_train_step: fused workspace too small (%zu < %zu)", x->fused_workspace_bytes, need);
        return SLB_ENOSPC;
    }
    return SLB_OK;
}

// The capacity a fused workspace is laid out for: the largest batch whose layout fits its bytes.
// It depends on the workspace alone, never on the calling step's batch, so every call sharing a
// workspace sees the same offsets.  That matters while two steps are in flight with different
// batches (the sharded step's local batch changes every step, and the plan of step k+1 runs under
// the float kernels of step k): neither plan slot then lands on the other, or on the step state.
int64_t v2_capacity(size_t bytes, int64_t U, int64_t I, int D) {
    int64_t lo = 0, hi = static_cast<int64_t>(bytes / (4 * static_cast<size_t>(D))) + 1;   // the stash alone
    while (hi - lo > 1) {                                                                 // outgrows `hi`
        const int64_t mid = lo + (hi - lo) / 2;
        if (v2_layout(nullptr, mid, U, I, D).bytes <= bytes) lo = mid;
        else hi = mid;
    }
    return lo;
}

// The layout every call on x->fused_workspace uses (after v2_check_ws: capacity >= x->batch).
V2Layout v2_layout_ws(const slb_mf_step_args* x, void* base, WsCarver* log = nullptr) {
    return v2_layout(base, v2_capacity(x->fused_workspace_bytes, x->num_users, x->num_items, x->dim),
                     x->num_users, x->num_items, x->dim, log);
}

}  // namespace

extern "C" {

size_t slb_mf_step_workspace_bytes(int64_t batch, int32_t n_neg, int32_t loss,
                                   int64_t num_users, int64_t num_items) {
    (void)n_neg; (void)loss;
    return mf_layout(nullptr, batch, num_users, num_items).bytes;
}

int64_t slb_mf_compact_rows(int64_t batch, int32_t n_neg, int32_t loss, int32_t which) {
    (void)n_neg; (void)loss; (void)which;
    return 2 * batch;  // positive + selected negative term per interaction
}

size_t slb_mf_fused_workspace_bytes(int64_t batch, int64_t num_users, int64_t num_items, int32_t dim) {
    if (batch <= 0 || !v2_dim_ok(dim)) return 0;
    return v2_layout(nullptr, batch, num_users, num_items, dim).bytes;
}

int slb_mf_train_step(const slb_mf_step_args* x, slb_stream_t stream) {
    const int rc = validate(x);
    if (rc != SLB_OK) return rc;
    if (v2_eligible(x)) {
        const int r2 = v2_check_ws(x);
        if (r2 != SLB_OK) return r2;
        const V2Layout l = v2_layout_ws(x, x->fused_workspace);
        MfLayout old = mf_layout(x->workspace, x->batch, x->num_users, x->num_items);
        return v2_launch_step(x, l, 0, old.err, x->users, x->items, x->negs, x->batch, x->loss_out,
                              static_cast<cudaStream_t>(stream), 7);
    }
    return launch_step(x, x->users, x->items, x->negs, x->batch, x->loss_out,
                       static_cast<cudaStream_t>(stream));
}

int slb_mf_train_step_phases(const slb_mf_step_args* x, int32_t phases, slb_stream_t stream) {
    const int rc = validate(x);
    if (rc != SLB_OK) return rc;
    if (v2_eligible(x)) {          // planned step: 1 plan, 2 user kernels, 4 item kernels
        const int r2 = v2_check_ws(x);
        if (r2 != SLB_OK) return r2;
        const V2Layout l = v2_layout_ws(x, x->fused_workspace);
        MfLayout old = mf_layout(x->workspace, x->batch, x->num_users, x->num_items);
        return v2_launch_step(x, l, (phases >> 8) & 1, old.err, x->users, x->items, x->negs, x->batch, x->loss_out,
                              static_cast<cudaStream_t>(stream), phases & 7);
    }
    return launch_step(x, x->users, x->items, x->negs, x->batch, x->loss_out,
                       static_cast<cudaStream_t>(stream), phases);
}

int slb_mf_plan_copy(const slb_mf_step_args* x, int32_t slot, int64_t batch, int32_t* totals, int32_t* seg_row,
                     int32_t* seg_start, int32_t* sid, int32_t* long_list, void* mu, void* mi, slb_stream_t stream) {
    SLB_REQUIRE(x && x->fused_workspace && v2_dim_ok(x->dim), "mf_plan_copy: needs a planned-step workspace");
    SLB_REQUIRE(slot == 0 || slot == 1, "mf_plan_copy: slot must be 0 or 1");
    SLB_REQUIRE(batch > 0 && batch <= x->batch, "mf_plan_copy: batch must be in [1, args.batch]");
    SLB_REQUIRE(totals && seg_row && seg_start && sid && long_list && mu && mi, "mf_plan_copy: null output");
    const int r = v2_check_ws(x);
    if (r != SLB_OK) return r;
    const PlanDev& p = v2_layout_ws(x, x->fused_workspace).plan[slot];
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const auto copy = [&](void* dst, const void* src, size_t n) {
        return cudaMemcpyAsync(dst, src, n, cudaMemcpyDeviceToDevice, st) == cudaSuccess;
    };
    const bool ok = copy(totals, p.seg.totals, 4 * sizeof(int32_t)) &&
                    copy(seg_row, p.seg.seg_row, (3 * batch + 1) * sizeof(int32_t)) &&
                    copy(seg_start, p.seg.seg_start, (3 * batch + 2) * sizeof(int32_t)) &&
                    copy(sid, p.seg.sid, (x->num_users + x->num_items) * sizeof(int32_t)) &&
                    copy(long_list, p.seg.long_list, (3 * batch / 16 + 2) * sizeof(int32_t)) &&
                    copy(mu, p.mu, batch * sizeof(URec)) && copy(mi, p.mi, 2 * batch * sizeof(IRec));
    if (!ok) { slb_set_error("mf_plan_copy: cudaMemcpyAsync failed"); return SLB_ECUDA; }
    return SLB_OK;
}

int32_t slb_mf_fused_layout(const slb_mf_step_args* x, int64_t* out, int32_t max_arrays) {
    SLB_REQUIRE(x && v2_dim_ok(x->dim) && x->batch > 0 && x->num_users > 0 && x->num_items > 0,
                "mf_fused_layout: needs batch, num_users, num_items and a planned-step dim");
    SLB_REQUIRE(out || max_arrays == 0, "mf_fused_layout: null output");
    const int r = v2_check_ws(x);
    if (r != SLB_OK) return r;
    // a stand-in base address, never dereferenced: the layout's pointers become byte offsets
    char* const base = reinterpret_cast<char*>(static_cast<uintptr_t>(1) << 40);
    int64_t log[2 * 64];
    WsCarver ws(base);
    ws.log = log;
    ws.max_log = 64;
    const V2Layout l = v2_layout_ws(x, base, &ws);
    SLB_REQUIRE(ws.n_log <= 64, "mf_fused_layout: more arrays than expected");
    const auto at = [&](const void* q) { return static_cast<int64_t>(static_cast<const char*>(q) - base); };
    for (int n = 0; n < ws.n_log && n < max_arrays; ++n) {
        int64_t group = -1;
        for (int k = 0; k < 2; ++k) {
            const PlanDev& p = l.plan[k];
            const void* mine[] = {p.seg.cnt, p.seg.off, p.seg.sid, p.seg.status, p.seg.ticket, p.seg.seg_row,
                                  p.seg.seg_start, p.seg.long_list, p.mu, p.mi, p.mu_tmp, p.mi_tmp, p.bits,
                                  p.slot, p.multi, p.nmulti};
            for (const void* q : mine) if (at(q) == log[2 * n]) group = k;
        }
        const void* step[] = {l.st.done, l.st.t_g, l.st.stash, l.st.partial, l.st.partial_long};
        for (const void* q : step) if (at(q) == log[2 * n]) group = 2;
        out[3 * n] = group;
        out[3 * n + 1] = log[2 * n];
        out[3 * n + 2] = log[2 * n + 1];
    }
    return ws.n_log;
}

static int fit_epoch_impl(const slb_mf_step_args* x, const int64_t* users, const int64_t* items,
                          const int64_t* negs, int64_t n, float* losses_out, slb_stream_t stream,
                          const int64_t* wait_steps, void* const* wait_events, int32_t n_waits) {
    slb_mf_step_args tmp = *x;
    tmp.users = users; tmp.items = items; tmp.negs = negs; tmp.loss_out = losses_out;
    const int rc = validate(&tmp);
    if (rc != SLB_OK) return rc;
    SLB_REQUIRE(x->grad_mode == SLB_GRAD_COMPACT && x->opt != SLB_OPT_NONE,
                "mf_fit_epoch: needs compact grads and a fused optimizer");
    SLB_REQUIRE(n > 0, "mf_fit_epoch: n must be > 0");
    cudaStream_t main_st = static_cast<cudaStream_t>(stream);
    if (v2_eligible(&tmp)) {
        // planned step: the plan of step k+1 (integer work on ids only) is enqueued on the plan
        // stream before the float kernels of step k, double-buffered, so it runs under them
        const int r2 = v2_check_ws(&tmp);
        if (r2 != SLB_OK) return r2;
        const V2Layout l = v2_layout_ws(x, x->fused_workspace);
        MfLayout old = mf_layout(x->workspace, x->batch, x->num_users, x->num_items);
        cudaStream_t plan_st = x->plan_stream ? static_cast<cudaStream_t>(x->plan_stream) : main_st;
        const bool two = plan_st != main_st;
        const int64_t nsteps = (n + x->batch - 1) / x->batch;
        cudaEvent_t ev_plan[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr}, ev_in = nullptr;
        int rc2 = SLB_OK;
        if (two) {
            bool ok = cudaEventCreateWithFlags(&ev_in, cudaEventDisableTiming) == cudaSuccess;
            for (int k = 0; k < 2 && ok; ++k)
                ok = cudaEventCreateWithFlags(&ev_plan[k], cudaEventDisableTiming) == cudaSuccess &&
                     cudaEventCreateWithFlags(&ev_done[k], cudaEventDisableTiming) == cudaSuccess;
            if (!ok) { slb_set_error("mf_fit_epoch: cannot create events"); rc2 = SLB_ECUDA; }
            if (rc2 == SLB_OK) {           // the plan stream starts after everything queued on the main stream so far
                cudaEventRecord(ev_in, main_st);
                cudaStreamWaitEvent(plan_st, ev_in, 0);
            }
        }
        int next_wait = 0;
        auto plan_of = [&](int64_t k) {
            const int64_t lo = k * x->batch;
            const int64_t B = n - lo < x->batch ? n - lo : x->batch;
            const int slot = static_cast<int>(k & 1);
            // inputs of step k onwards become ready with this event (e.g. a chunk of negatives drawn
            // on another stream); the float kernels inherit the dependency through ev_plan
            while (next_wait < n_waits && wait_steps[next_wait] <= k) {
                cudaStreamWaitEvent(plan_st, static_cast<cudaEvent_t>(wait_events[next_wait]), 0);
                ++next_wait;
            }
            if (two && k >= 2) cudaStreamWaitEvent(plan_st, ev_done[slot], 0);      // slot free again
            const int r = v2_launch_plan(&tmp, l.plan[slot], old.err, users + lo, items + lo, negs + lo, B, plan_st);
            if (two) cudaEventRecord(ev_plan[slot], plan_st);
            return r;
        };
        if (rc2 == SLB_OK) rc2 = plan_of(0);
        for (int64_t k = 0; k < nsteps && rc2 == SLB_OK; ++k) {
            const int64_t lo = k * x->batch;
            const int64_t B = n - lo < x->batch ? n - lo : x->batch;
            const int slot = static_cast<int>(k & 1);
            if (k + 1 < nsteps) rc2 = plan_of(k + 1);
            if (rc2 != SLB_OK) break;
            if (two) cudaStreamWaitEvent(main_st, ev_plan[slot], 0);
            rc2 = v2_launch_step(&tmp, l, slot, old.err, users + lo, items + lo, negs + lo, B, losses_out + k,
                                 main_st, 6);
            if (two) cudaEventRecord(ev_done[slot], main_st);
        }
        if (two) {
            // later work on the plan stream must not overtake this epoch's float kernels
            if (ev_in) { cudaEventRecord(ev_in, main_st); cudaStreamWaitEvent(plan_st, ev_in, 0); }
            for (int k = 0; k < 2; ++k) {
                if (ev_plan[k]) cudaEventDestroy(ev_plan[k]);
                if (ev_done[k]) cudaEventDestroy(ev_done[k]);
            }
            if (ev_in) cudaEventDestroy(ev_in);
        }
        return rc2;
    }
    int64_t step = 0;
    int next_wait = 0;
    for (int64_t lo = 0; lo < n; lo += x->batch, ++step) {
        const int64_t B = n - lo < x->batch ? n - lo : x->batch;
        while (next_wait < n_waits && wait_steps[next_wait] <= step) {
            cudaStreamWaitEvent(main_st, static_cast<cudaEvent_t>(wait_events[next_wait]), 0);
            ++next_wait;
        }
        // adaptive hinge: negatives of step k are the flat [B*n_neg] block the
        // reference's per-batch randint would have produced (implicit.py:256-259)
        const int64_t* ng = negs + lo * x->n_neg;
        const int r = launch_step(x, users + lo, items + lo, ng, B, losses_out + step, main_st, 0x1f, step);
        if (r != SLB_OK) return r;
    }
    return SLB_OK;
}

int slb_mf_fit_epoch(const slb_mf_step_args* x, const int64_t* users, const int64_t* items,
                     const int64_t* negs, int64_t n, float* losses_out, slb_stream_t stream) {
    return fit_epoch_impl(x, users, items, negs, n, losses_out, stream, nullptr, nullptr, 0);
}

int slb_mf_fit_epoch_events(const slb_mf_step_args* x, const int64_t* users, const int64_t* items,
                            const int64_t* negs, int64_t n, float* losses_out, slb_stream_t stream,
                            const int64_t* wait_steps, void* const* wait_events, int32_t n_waits) {
    SLB_REQUIRE(n_waits == 0 || (wait_steps && wait_events), "mf_fit_epoch_events: null wait list");
    for (int32_t k = 1; k < n_waits; ++k)
        SLB_REQUIRE(wait_steps[k] >= wait_steps[k - 1], "mf_fit_epoch_events: wait_steps must ascend");
    return fit_epoch_impl(x, users, items, negs, n, losses_out, stream, wait_steps, wait_events, n_waits);
}

int slb_adam_flush(float* W, float* exp_avg, float* exp_avg_sq, float* bias, float* bias_avg, float* bias_avg_sq,
                   int32_t* last, int64_t rows, int32_t dim, const float* sched, int64_t step,
                   float beta1, float beta2, float one_minus_beta1, float one_minus_beta2, float eps,
                   float weight_decay, slb_stream_t stream) {
    SLB_REQUIRE(W && exp_avg && exp_avg_sq && bias && bias_avg && bias_avg_sq && last && sched, "adam_flush: null pointer");
    SLB_REQUIRE(rows > 0 && dim >= 4 && dim % 4 == 0 && step >= 0 && step < (1ll << 31), "adam_flush: bad sizes");
    if (step == 0) return SLB_OK;
    AdamDev o = {beta1, beta2, one_minus_beta1, one_minus_beta2, eps, weight_decay, sched, static_cast<int32_t>(step)};
    const int lpr = lpr_for_dim(dim);
    const int groups = MF_THREADS / lpr;
    const int64_t want = (rows + groups - 1) / groups;
    const int sms = slb_sms();
    const int grid = static_cast<int>(want < static_cast<int64_t>(sms) * 16 ? want : static_cast<int64_t>(sms) * 16);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    DISPATCH_LPR(lpr, adam_flush_kernel, grid, MF_THREADS, st, W, exp_avg, exp_avg_sq, bias, bias_avg, bias_avg_sq,
                 last, rows, dim, o);
    SLB_LAUNCH_CHECK("adam_flush_kernel");
    return SLB_OK;
}

int slb_mf_scores(const float* Wu, const float* Wi, const float* bu, const float* bi,
                  int32_t dim, const int64_t* users, const int64_t* items, int64_t n,
                  int32_t user_broadcast, float* scores, slb_stream_t stream) {
    SLB_REQUIRE(dim >= 4 && dim % 4 == 0, "mf_scores: dim must be a positive multiple of 4 (got %d)", dim);
    SLB_REQUIRE(Wu && Wi && bu && bi && users && items && scores, "mf_scores: null pointer");
    if (n <= 0) return SLB_OK;
    const int lpr = lpr_for_dim(dim);
    const int groups = MF_THREADS / lpr;
    const int sms = slb_sms();
    int64_t want = (n + groups - 1) / groups;
    int grid = static_cast<int>(want < static_cast<int64_t>(sms) * 8 ? want : static_cast<int64_t>(sms) * 8);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    DISPATCH_LPR(lpr, mf_scores_kernel, grid, MF_THREADS, st, Wu, Wi, bu, bi, dim, users, items, n,
                 user_broadcast, scores);
    SLB_LAUNCH_CHECK("mf_scores_kernel");
    return SLB_OK;
}

int slb_mf_scores_backward(const float* gscores, const int64_t* users, const int64_t* items,
                           int64_t n, int32_t user_broadcast, const float* Wu, const float* Wi,
                           int64_t num_users, int64_t num_items, int32_t dim,
                           float* dWu, float* dWi, float* dbu, float* dbi,
                           void* workspace, size_t workspace_bytes, slb_stream_t stream) {
    SLB_REQUIRE(dim >= 4 && dim % 4 == 0, "mf_scores_backward: dim must be a positive multiple of 4 (got %d)", dim);
    SLB_REQUIRE(gscores && users && items && Wu && Wi && dWu && dWi && dbu && dbi && workspace,
                "mf_scores_backward: null pointer");
    SLB_REQUIRE(num_users + num_items < (1ll << 31) - SEG_SCAN_TILE && n * 2 < (1ll << 31), "mf_scores_backward: too large");
    if (n <= 0) return SLB_OK;
    const int64_t Bcap = (n + 1) / 2;           // layout holds 2*Bcap >= n terms
    MfLayout l = mf_layout(workspace, Bcap, num_users, num_items);
    if (workspace_bytes < l.bytes) {
        slb_set_error("mf_scores_backward: workspace too small (%zu < %zu)", workspace_bytes, l.bytes);
        return SLB_ENOSPC;
    }
    MfDev a = {};
    a.B = n; a.NB = n; a.T = n; a.users = users; a.items = items;
    a.U = num_users; a.I = num_items; a.D = dim;
    a.Wu = const_cast<float*>(Wu); a.Wi = const_cast<float*>(Wi);
    a.t_a = l.t_a; a.t_b = l.t_b; a.t_g = l.t_g; a.partial = l.partial; a.done = l.done; a.err = l.err;
    a.seg = l.seg;
    a.seg.long_cap = seg_sort_cap(lpr_for_dim(dim));
    a.no_bias = 0; a.frozen_a = -1; a.frozen_b = -1;
    a.grad_mode = SLB_GRAD_DENSE;
    a.dWu = dWu; a.dWi = dWi; a.dbu = dbu; a.dbi = dbi;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int sms = slb_sms();
    int g1 = static_cast<int>((n + 255) / 256);
    if (g1 > sms * 8) g1 = sms * 8;
    mf_terms_kernel<<<g1, 256, 0, st>>>(a, gscores, user_broadcast);
    SLB_LAUNCH_CHECK("mf_terms_kernel");
    seg_scan_launch(a.seg, a.U, st);
    SLB_LAUNCH_CHECK("seg_scan_kernel");
    mf_fill_kernel<<<g1, 256, 0, st>>>(a);
    SLB_LAUNCH_CHECK("mf_fill_kernel");
    seg_sort_long_kernel<<<SEG_LONG_CTAS, 256, 0, st>>>(a.seg);
    SLB_LAUNCH_CHECK("seg_sort_long_kernel");
    const int lpr = lpr_for_dim(dim);
    int64_t tw = ((n + 31) / 32 + 3) / 4;
    int tgrid = static_cast<int>(tw < static_cast<int64_t>(sms) * 16 ? tw : static_cast<int64_t>(sms) * 16);
    DISPATCH_LPR3(lpr, mf_bwd_tile_kernel, 0, 32, tgrid, MF_TILE_THREADS, st, a);
    SLB_LAUNCH_CHECK("mf_bwd_tile_kernel");
    launch_long<0>(lpr, st, a);
    SLB_LAUNCH_CHECK("mf_bwd_long_kernel");
    return SLB_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------
// Sparse update of an id-indexed bias table from n (id, g) pairs -- the unhashed bias tables
// next to BloomEmbedding layers (representations.py:58-59) have one row per raw id (50 M at
// BASELINE config 4), so neither a dense gradient nor a scan over the id space is affordable.
// The pairs are grouped through a hash-bucket segment index (bucket = id & (NB - 1), NB ~ 2n a
// power of two: count -> scan -> fill), each bucket's few members are ordered by (id, pair) and
// every distinct id gets its gradient summed in pair order and one optimizer update.
// Deterministic, O(n) traffic.
// ---------------------------------------------------------------------------
namespace {

struct BiasSparse {
    SegIndex seg;
    const int64_t* ids; const float* g; int64_t n; int64_t mask;
    float* b; float* sb;
    int32_t opt; float lr, wd, eps;
};

__global__ void __launch_bounds__(256) bias_count_kernel(BiasSparse p) {
    const int64_t nth = static_cast<int64_t>(gridDim.x) * blockDim.x;
    for (int64_t k = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; k < p.n; k += nth)
        if (p.g[k] != 0.f) atomicAdd(p.seg.cnt + (p.ids[k] & p.mask), 1);
}

__global__ void __launch_bounds__(256) bias_fill_kernel(BiasSparse p) {
    const int64_t nth = static_cast<int64_t>(gridDim.x) * blockDim.x;
    for (int64_t k = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; k < p.n; k += nth)
        if (p.g[k] != 0.f) seg_place(p.seg, p.ids[k] & p.mask, static_cast<int32_t>(k));
}

__global__ void __launch_bounds__(256) bias_apply_kernel(BiasSparse p) {
    const int nseg = p.seg.totals[0];
    const OptV2 o = {p.opt, p.lr, p.wd, p.eps};
    const int nth = gridDim.x * blockDim.x;
    for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < nseg; s += nth) {
        const int start = p.seg.seg_start[s], len = p.seg.seg_start[s + 1] - start;
        // members of one bucket: process distinct ids in ascending (id, pair) order by repeated
        // selection (buckets hold ~1 pair; O(len^2) is irrelevant)
        int64_t last_id = -1;
        for (;;) {
            int64_t cur = INT64_MAX;
            for (int m = 0; m < len; ++m) {
                const int64_t id = p.ids[p.seg.members[start + m]];
                if (id > last_id && id < cur) cur = id;
            }
            if (cur == INT64_MAX) break;
            // sum this id's pairs in ascending pair order
            float acc = 0.f;
            int prev = -1;
            for (;;) {
                int best = INT32_MAX;
                for (int m = 0; m < len; ++m) {
                    const int k = p.seg.members[start + m];
                    if (k > prev && k < best && p.ids[k] == cur) best = k;
                }
                if (best == INT32_MAX) break;
                acc += p.g[best];
                prev = best;
            }
            bias_update(o, p.b + cur, p.sb ? p.sb + cur : nullptr, acc);
            last_id = cur;
        }
    }
}

size_t bias_sparse_bytes(int64_t n) {
    int64_t nb = 4096;
    while (nb < 2 * n) nb <<= 1;
    WsCarver ws(nullptr);
    seg_index_carve(ws, nb, n);
    return ws.bytes();
}

int bias_sparse_apply(void* wsp, const int64_t* ids, const float* g, int64_t n, float* b, float* sb,
                      int32_t opt, float lr, float wd, float eps, cudaStream_t st) {
    int64_t nb = 4096;
    while (nb < 2 * n) nb <<= 1;
    WsCarver ws(wsp);
    BiasSparse p;
    p.seg = seg_index_carve(ws, nb, n);
    p.ids = ids; p.g = g; p.n = n; p.mask = nb - 1; p.b = b; p.sb = sb;
    p.opt = opt; p.lr = lr; p.wd = wd; p.eps = eps;
    const int sms = slb_sms();
    int grid = static_cast<int>((n + 255) / 256);
    if (grid > sms * 8) grid = sms * 8;
    bias_count_kernel<<<grid, 256, 0, st>>>(p);
    SLB_LAUNCH_CHECK("bias_count_kernel");
    seg_scan_launch(p.seg, p.seg.Rpad, st);
    SLB_LAUNCH_CHECK("seg_scan_kernel");
    bias_fill_kernel<<<grid, 256, 0, st>>>(p);
    SLB_LAUNCH_CHECK("bias_fill_kernel");
    bias_apply_kernel<<<grid, 256, 0, st>>>(p);
    SLB_LAUNCH_CHECK("bias_apply_kernel");
    return SLB_OK;
}

}  // namespace

struct BloomLayout {
    int32_t* t_a; int32_t* t_b; float* t_g; float* partial; int32_t* done; int32_t* err;
    SegIndex seg;
    int64_t* ids_u2; int64_t* ids_i2; float* g_u2; float* g_i2;
    void* ws_u; size_t ws_u_bytes; void* ws_i; size_t ws_i_bytes;
    // fused-optimizer mode: compact item-row gradients + hash-bucket bias workspaces
    int64_t* irows; float* gWi; int32_t* compact_counts; void* bws_u; void* bws_i;
    size_t bytes;
};

static BloomLayout bloom_layout(void* base, const slb_mf_bloom_args* x) {
    const int nu = x->user_hashes ? x->user_hashes : 1, ni = x->item_hashes ? x->item_hashes : 1;
    const int64_t B = x->base.batch, T = 2 * B * nu * ni;
    WsCarver ws(base);
    BloomLayout l;
    l.done = ws.take<int32_t>(8);
    l.err = l.done + 4;
    l.seg = seg_index_carve(ws, x->user_rows + x->item_rows, 2 * T);
    l.t_a = ws.take<int32_t>(T);
    l.t_b = ws.take<int32_t>(T);
    l.t_g = ws.take<float>(T);
    l.partial = ws.take<float>(MF_MAX_GRID);
    l.ids_u2 = ws.take<int64_t>(2 * B);
    l.ids_i2 = ws.take<int64_t>(2 * B);
    l.g_u2 = ws.take<float>(2 * B);
    l.g_i2 = ws.take<float>(2 * B);
    l.irows = nullptr; l.gWi = nullptr; l.compact_counts = nullptr; l.bws_u = nullptr; l.bws_i = nullptr;
    l.ws_u = nullptr; l.ws_i = nullptr; l.ws_u_bytes = 0; l.ws_i_bytes = 0;
    if (x->base.opt == SLB_OPT_NONE) {
        l.ws_u_bytes = slb_embedding_backward_workspace_bytes(2 * B, x->base.num_users);
        l.ws_u = ws.take<char>(l.ws_u_bytes);
        l.ws_i_bytes = slb_embedding_backward_workspace_bytes(2 * B, x->base.num_items);
        l.ws_i = ws.take<char>(l.ws_i_bytes);
    } else {
        // the two bias workspaces are zero-at-rest and must precede the batch-sized scratch?  No:
        // this workspace is dedicated to one (shapes, batch), so every offset is fixed.
        l.bws_u = ws.take<char>(bias_sparse_bytes(2 * B));
        l.bws_i = ws.take<char>(bias_sparse_bytes(2 * B));
        const int64_t irow_cap = T < x->item_rows ? T : x->item_rows;
        l.irows = ws.take<int64_t>(irow_cap + 1);
        l.gWi = ws.take<float>(static_cast<size_t>(irow_cap + 1) * x->base.dim);
        l.compact_counts = ws.take<int32_t>(4);
    }
    l.bytes = ws.bytes();
    return l;
}

extern "C" {

size_t slb_mf_bloom_workspace_bytes(const slb_mf_bloom_args* x) {
    if (!x || x->base.batch <= 0) return 0;
    return bloom_layout(nullptr, x).bytes;
}

int slb_mf_bloom_train_step(const slb_mf_bloom_args* x, slb_stream_t stream) {
    SLB_REQUIRE(x != nullptr, "mf_bloom_train_step: null args");
    const slb_mf_step_args& b = x->base;
    SLB_REQUIRE(b.batch > 0 && b.dim >= 4 && b.dim % 4 == 0, "mf_bloom_train_step: bad batch / dim");
    SLB_REQUIRE(b.loss >= 0 && b.loss <= 3 && b.n_neg >= 1, "mf_bloom_train_step: bad loss / n_neg");
    SLB_REQUIRE(b.loss == SLB_LOSS_ADAPTIVE_HINGE || b.n_neg == 1, "mf_bloom_train_step: n_neg > 1 only for adaptive hinge");
    const bool fused = b.opt != SLB_OPT_NONE;
    SLB_REQUIRE(fused ? (b.opt == SLB_OPT_SGD || b.opt == SLB_OPT_ADAGRAD) : b.grad_mode == SLB_GRAD_DENSE,
                "mf_bloom_train_step: dense gradients, or a fused SGD / Adagrad optimizer");
    SLB_REQUIRE(!fused || b.opt == SLB_OPT_SGD || (b.state_Wu && b.state_Wi && b.state_bu && b.state_bi),
                "mf_bloom_train_step: adagrad needs state");
    SLB_REQUIRE(x->user_hashes >= 0 && x->user_hashes <= 24 && x->item_hashes >= 0 && x->item_hashes <= 24,
                "mf_bloom_train_step: at most 24 hash functions");
    SLB_REQUIRE(x->user_rows > 0 && x->item_rows > 0 && b.num_users > 0 && b.num_items > 0, "mf_bloom_train_step: empty tables");
    SLB_REQUIRE(x->user_hashes > 0 || x->user_rows == b.num_users, "mf_bloom_train_step: plain user table must have num_users rows");
    SLB_REQUIRE(x->item_hashes > 0 || x->item_rows == b.num_items, "mf_bloom_train_step: plain item table must have num_items rows");
    const bool pairs_u = x->pair_ids_u && x->pair_g_u, pairs_i = x->pair_ids_i && x->pair_g_i;
    SLB_REQUIRE(b.users && b.items && b.negs && b.Wu && b.Wi && b.bu && b.bi && b.loss_out && b.workspace &&
                (fused || (b.dWu && b.dWi && (b.dbu || pairs_u) && (b.dbi || pairs_i))), "mf_bloom_train_step: null pointer");
    const int nu = x->user_hashes ? x->user_hashes : 1, ni = x->item_hashes ? x->item_hashes : 1;
    const int64_t B = b.batch, T = 2 * B * nu * ni;
    SLB_REQUIRE(x->user_rows + x->item_rows < (1ll << 31) - SEG_SCAN_TILE && 2 * T < (1ll << 31),
                "mf_bloom_train_step: too large");
    BloomLayout l = bloom_layout(b.workspace, x);
    if (b.workspace_bytes < l.bytes) {
        slb_set_error("mf_bloom_train_step: workspace too small (%zu < %zu)", b.workspace_bytes, l.bytes);
        return SLB_ENOSPC;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MfDev a = {};
    a.B = B; a.NB = b.norm_batch > 0 ? b.norm_batch : B; a.T = T;
    a.users = b.users; a.items = b.items; a.negs = b.negs; a.loss = b.loss; a.n_neg = b.n_neg;
    a.U = x->user_rows; a.I = x->item_rows; a.D = b.dim;      // key spaces = table rows
    a.Wu = b.Wu; a.Wi = b.Wi; a.bu = b.bu; a.bi = b.bi;
    a.loss_out = b.loss_out; a.pos_out = b.pos_out; a.neg_out = b.neg_out;
    a.t_a = l.t_a; a.t_b = l.t_b; a.t_g = l.t_g; a.partial = l.partial; a.done = l.done; a.err = l.err;
    a.seg = l.seg;
    const int lpr = lpr_for_dim(b.dim);
    a.seg.long_cap = seg_sort_cap(lpr);
    a.grad_mode = fused ? SLB_GRAD_COMPACT : SLB_GRAD_DENSE;
    a.dWu = b.dWu; a.dWi = b.dWi; a.dbu = b.dbu; a.dbi = b.dbi;
    a.irows = l.irows; a.gWi = l.gWi; a.compact_counts = l.compact_counts;
    a.opt = b.opt; a.lr = b.lr; a.wd = b.weight_decay; a.eps = b.eps;
    a.sWu = b.state_Wu; a.sWi = b.state_Wi; a.sbu = b.state_bu; a.sbi = b.state_bi;
    a.no_bias = 1;
    a.frozen_a = x->user_hashes ? x->user_padding_idx : -1;
    a.frozen_b = x->item_hashes ? x->item_padding_idx : -1;
    BloomSpec h = {};
    h.Hu = x->user_hashes; h.Hi = x->item_hashes;
    h.pad_u = x->user_padding_idx; h.pad_i = x->item_padding_idx;
    for (int k = 0; k < 24; ++k) { h.su[k] = x->user_seeds[k]; h.si[k] = x->item_seeds[k]; }
    h.num_users = b.num_users; h.num_items = b.num_items;
    h.ids_u2 = l.ids_u2; h.ids_i2 = l.ids_i2; h.g_u2 = l.g_u2; h.g_i2 = l.g_i2;
    if (!fused && pairs_u) { h.ids_u2 = x->pair_ids_u; h.g_u2 = x->pair_g_u; }
    if (!fused && pairs_i) { h.ids_i2 = x->pair_ids_i; h.g_i2 = x->pair_g_i; }

    const int groups = MF_THREADS / lpr;
    const int sms = slb_sms();
    int64_t want = (B + groups - 1) / groups;
    int grid = static_cast<int>(want < static_cast<int64_t>(sms) * 8 ? want : static_cast<int64_t>(sms) * 8);
    if (grid > MF_MAX_GRID) grid = MF_MAX_GRID;
    switch (lpr) {
        case 1: mf_fwd_bloom_kernel<1><<<grid, MF_THREADS, 0, st>>>(a, h); break;
        case 2: mf_fwd_bloom_kernel<2><<<grid, MF_THREADS, 0, st>>>(a, h); break;
        case 4: mf_fwd_bloom_kernel<4><<<grid, MF_THREADS, 0, st>>>(a, h); break;
        case 8: mf_fwd_bloom_kernel<8><<<grid, MF_THREADS, 0, st>>>(a, h); break;
        case 16: mf_fwd_bloom_kernel<16><<<grid, MF_THREADS, 0, st>>>(a, h); break;
        default: mf_fwd_bloom_kernel<32><<<grid, MF_THREADS, 0, st>>>(a, h); break;
    }
    SLB_LAUNCH_CHECK("mf_fwd_bloom_kernel");
    seg_scan_launch(a.seg, a.U, st);
    SLB_LAUNCH_CHECK("seg_scan_kernel");
    int fgrid = static_cast<int>((T + 255) / 256);
    if (fgrid > sms * 8) fgrid = sms * 8;
    mf_fill_kernel<<<fgrid, 256, 0, st>>>(a);
    SLB_LAUNCH_CHECK("mf_fill_kernel");
    seg_sort_long_kernel<<<SEG_LONG_CTAS, 256, 0, st>>>(a.seg);
    SLB_LAUNCH_CHECK("seg_sort_long_kernel");
    const int64_t tw = ((2 * T + 31) / 32 + 3) / 4;
    const int tgrid = static_cast<int>(tw < static_cast<int64_t>(sms) * 16 ? tw : static_cast<int64_t>(sms) * 16);
    if (fused) {
        // hashed item rows first (compact gradients from the old user rows), user rows updated in
        // place, item rows updated from the compact gradients, then the id-space biases
        DISPATCH_LPR3(lpr, mf_bwd_tile_kernel, 1, 32, tgrid, MF_TILE_THREADS, st, a);
        SLB_LAUNCH_CHECK("mf_bwd_tile_kernel<items>");
        launch_long<1>(lpr, st, a);
        DISPATCH_LPR3(lpr, mf_bwd_tile_kernel, 2, 32, tgrid, MF_TILE_THREADS, st, a);
        SLB_LAUNCH_CHECK("mf_bwd_tile_kernel<users+opt>");
        launch_long<2>(lpr, st, a);
        const int64_t aw = (2 * T + groups - 1) / groups;
        const int agrid = static_cast<int>(aw < static_cast<int64_t>(sms) * 8 ? aw : static_cast<int64_t>(sms) * 8);
        DISPATCH_LPR2(lpr, mf_apply_kernel, 1, agrid, MF_THREADS, st, a);
        SLB_LAUNCH_CHECK("mf_apply_kernel<items>");
        int rcb = bias_sparse_apply(l.bws_u, l.ids_u2, l.g_u2, 2 * B, b.bu, b.state_bu, b.opt, b.lr, b.weight_decay, b.eps, st);
        if (rcb != SLB_OK) return rcb;
        return bias_sparse_apply(l.bws_i, l.ids_i2, l.g_i2, 2 * B, b.bi, b.state_bi, b.opt, b.lr, b.weight_decay, b.eps, st);
    }
    DISPATCH_LPR3(lpr, mf_bwd_tile_kernel, 0, 32, tgrid, MF_TILE_THREADS, st, a);
    SLB_LAUNCH_CHECK("mf_bwd_tile_kernel");
    launch_long<0>(lpr, st, a);
    SLB_LAUNCH_CHECK("mf_bwd_long_kernel");
    // id-space bias gradients: deterministic scalar scatter (D = 1), unless handed out as pairs
    int rc = SLB_OK;
    if (!pairs_u)
        rc = slb_embedding_backward(l.g_u2, l.ids_u2, 2 * B, 0, nullptr, b.num_users, 1, -1, b.dbu, l.ws_u,
                                    l.ws_u_bytes, stream);
    if (rc != SLB_OK) return rc;
    if (!pairs_i)
        rc = slb_embedding_backward(l.g_i2, l.ids_i2, 2 * B, 0, nullptr, b.num_items, 1, -1, b.dbi, l.ws_i,
                                    l.ws_i_bytes, stream);
    return rc;
}

size_t slb_bias_sparse_workspace_bytes(int64_t n) { return n > 0 ? bias_sparse_bytes(n) : 0; }

int slb_bias_sparse_apply(const int64_t* ids, const float* g, int64_t n, float* bias, float* state,
                          int32_t opt, float lr, float weight_decay, float eps,
                          void* workspace, size_t workspace_bytes, slb_stream_t stream) {
    if (n <= 0) return SLB_OK;
    SLB_REQUIRE(ids && g && bias && workspace, "bias_sparse_apply: null pointer");
    SLB_REQUIRE(opt == SLB_OPT_SGD || (opt == SLB_OPT_ADAGRAD && state), "bias_sparse_apply: SGD, or Adagrad with state");
    SLB_REQUIRE(n < (1ll << 30), "bias_sparse_apply: too many pairs");
    if (workspace_bytes < bias_sparse_bytes(n)) {
        slb_set_error("bias_sparse_apply: workspace too small");
        return SLB_ENOSPC;
    }
    return bias_sparse_apply(workspace, ids, g, n, bias, state, opt, lr, weight_decay, eps,
                             static_cast<cudaStream_t>(stream));
}

}  // extern "C"

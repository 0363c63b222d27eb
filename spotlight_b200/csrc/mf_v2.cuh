// Planned two-kernel training step (pointwise / bpr / hinge with a fused row-wise optimizer).
//
// The gradient of a minibatch depends on its ids only through *which* interactions share a
// row.  That grouping is integer work on ids that are known before the step runs (the epoch's
// shuffle and negative draw are done), so it is split off as a PLAN that can run ahead of the
// floating-point kernels, on a second stream, double-buffered:
//
//   plan (ids only)   count rows -> scan -> fill member records -> sort each member list
//                     user segment s : rows of {b, i_b, j_b}  (interactions of one user)
//                     item segment s : rows of {t, useg}      (terms 2b / 2b+1 on one item row,
//                                                              with the user segment of b)
//   mf_user_kernel    ONE pass over the touched user rows: load U[u] once, score every
//                     interaction of that user against its two item rows (item table is L2
//                     resident), loss, d loss / d score, accumulate dU, stash the old row for
//                     the item side, apply the optimizer in place.  Forward and the user half
//                     of the backward are the same kernel: the user row is read once per step
//                     instead of once per interaction and again in the backward.
//   mf_item_kernel    one pass over the touched item rows: sum g * U_old[u] over the row's
//                     terms in ascending term order (from the stash, mostly L2 hits), apply
//                     the optimizer in place.
//
// Replaces, for this route, mf_fwd_tile + seg scan + fill + bwd<items> + bwd<users> + apply
// (10 launches, user rows gathered twice) of the first-generation step; semantics identical:
// spotlight/factorization/implicit.py:229-243 with a row-wise SGD / Adagrad optimizer.
// Deterministic: no float atomics, every row has one writer that sums in ascending
// interaction order.
#pragma once

struct __align__(16) URec { int32_t b, i, j, pad; };
struct __align__(8) IRec { int32_t t, useg; };

struct PlanDev {
    SegIndex seg;          // cnt / off / sid / status / totals / seg_row / seg_start / long_list
    URec* mu;              // [B]   user-side member records (segment order)
    IRec* mi;              // [2B]  item-side member records
    URec* mu_tmp;          // [B]   scratch of the hot-row sort
    IRec* mi_tmp;          // [2B]
    uint32_t* bits;        // [SEG_LONG_CTAS][2 * words] bitmap + prefix of the hot-row sort
    int64_t words;
    int32_t* slot;         // [3B]  a member's place in its row's list: the count's atomicAdd (u, i, j blocks)
    int32_t* multi;        // [3B / 2 + 1] segments with 2..long_cap members, in no particular order
    int32_t* nmulti;       // [1]   length of `multi`
    int32_t* err;
    int64_t B, U, I;
    const int64_t* users; const int64_t* items; const int64_t* negs;
};

struct StepV2 {
    float* t_g;            // [2B] d loss / d score of term t (already / B)
    float* stash;          // [B][D] old user rows, by user segment
    float* partial;        // [MF_MAX_GRID] loss partials of mf_user_kernel
    float* partial_long;   // [SEG_LONG_CTAS * 4] loss partials of the hot-row kernel
    int32_t* done;
};

// ------------------------------------------------------------------ plan kernels
//
// count -> scan -> fill -> sort, four launches.  The plan runs under the previous step's float
// kernels, so what it costs the step is mostly the SM time its CTAs take from them: the kernels
// are small grid-stride grids (PLAN_GRID_PER_SM CTAs per SM) with short dependence chains.

#ifndef PLAN_GRID_PER_SM
#define PLAN_GRID_PER_SM 4
#endif

__device__ __forceinline__ bool plan_ids_ok(const PlanDev& p, int64_t u, int64_t i, int64_t j) {
    return u >= 0 && u < p.U && i >= 0 && i < p.I && j >= 0 && j < p.I;
}

// Counts the members of every row and keeps each member's slot (the value its atomicAdd returned):
// the fill then places it at off[row] + slot without a second round of atomics.  Also re-arms this
// plan's scan (look-back words, tile ticket, list lengths); the previous scan of the same plan slot
// has completed, by stream order.
__global__ void __launch_bounds__(256) plan_count_kernel(PlanDev p) {
    const int64_t tid = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t nth = static_cast<int64_t>(gridDim.x) * blockDim.x;
    for (int64_t t = tid; t < p.seg.ntiles; t += nth) p.seg.status[t] = 0ull;
    if (tid == 0) { *p.seg.ticket = 0; p.seg.totals[3] = 0; *p.nmulti = 0; }
    for (int64_t b = tid; b < p.B; b += nth) {
        const int64_t u = p.users[b], i = p.items[b], j = p.negs[b];
        if (!plan_ids_ok(p, u, i, j)) { atomicExch(p.err, 1); continue; }
        const int su = atomicAdd(p.seg.cnt + u, 1);
        const int si = atomicAdd(p.seg.cnt + p.U + i, 1);
        const int sj = atomicAdd(p.seg.cnt + p.U + j, 1);
        p.slot[b] = su;
        p.slot[p.B + b] = si;
        p.slot[2 * p.B + b] = sj;
    }
}

// Single-pass scan of cnt[0..Rpad) (decoupled look-back over dynamically numbered tiles: a tile
// only waits for tiles that took their number earlier, so it needs no co-residency).  Warp w of a
// tile owns rows tile * 4096 + w * 512 + 32 k + lane, so every load and store of a warp covers
// consecutive rows.  Emits off / sid per touched row, the segment list (seg_row, seg_start),
// long_list (> long_cap members), `multi` (2..long_cap members: the sort's work list) and the
// totals, and zeroes the counters it consumed.
constexpr int PLAN_SCAN_WARPS = SEG_SCAN_THREADS / 32;
constexpr int PLAN_SCAN_ITEMS = SEG_SCAN_TILE / SEG_SCAN_THREADS;     // rows per lane

__global__ void __launch_bounds__(SEG_SCAN_THREADS) plan_scan_kernel(PlanDev p) {
    __shared__ uint32_t sh_w[3][PLAN_SCAN_WARPS];      // per warp: sum, non-zero rows, multi rows
    __shared__ uint32_t sh_pre[3];                     // tile prefix: sum, segments, multi position
    __shared__ int sh_tile;
    const SegIndex& s = p.seg;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int cap = s.long_cap;
    if (threadIdx.x == 0) sh_tile = atomicAdd(s.ticket, 1);
    __syncthreads();
    const int tile = sh_tile;
    const int64_t base = static_cast<int64_t>(tile) * SEG_SCAN_TILE + warp * (32 * PLAN_SCAN_ITEMS) + lane;

    int32_t c[PLAN_SCAN_ITEMS];
#pragma unroll
    for (int k = 0; k < PLAN_SCAN_ITEMS; ++k) c[k] = s.cnt[base + 32 * k];
    uint32_t tsum = 0, tnz = 0, tmul = 0;
#pragma unroll
    for (int k = 0; k < PLAN_SCAN_ITEMS; ++k) {
        tsum += c[k]; tnz += c[k] != 0; tmul += c[k] >= 2 && c[k] <= cap;
        if (c[k] != 0) s.cnt[base + 32 * k] = 0;        // zero at rest again
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        tsum += __shfl_xor_sync(0xffffffffu, tsum, o);
        tnz += __shfl_xor_sync(0xffffffffu, tnz, o);
        tmul += __shfl_xor_sync(0xffffffffu, tmul, o);
    }
    if (lane == 0) { sh_w[0][warp] = tsum; sh_w[1][warp] = tnz; sh_w[2][warp] = tmul; }
    __syncthreads();
    if (warp == 0) {
        uint32_t v[3];
#pragma unroll
        for (int q = 0; q < 3; ++q) v[q] = lane < PLAN_SCAN_WARPS ? sh_w[q][lane] : 0u;
        uint32_t inc[3] = {v[0], v[1], v[2]};
#pragma unroll
        for (int o = 1; o < PLAN_SCAN_WARPS; o <<= 1)
#pragma unroll
            for (int q = 0; q < 3; ++q) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, inc[q], o);
                if (lane >= o) inc[q] += t;
            }
        uint32_t agg[3];
#pragma unroll
        for (int q = 0; q < 3; ++q) agg[q] = __shfl_sync(0xffffffffu, inc[q], PLAN_SCAN_WARPS - 1);
        if (lane < PLAN_SCAN_WARPS)
#pragma unroll
            for (int q = 0; q < 3; ++q) sh_w[q][lane] = inc[q] - v[q];      // exclusive, per warp
        volatile unsigned long long* st = s.status;
        if (lane == 0) st[tile] = seg_pack(tile == 0 ? SEG_FLAG_INC : SEG_FLAG_AGG, agg[0], agg[1]);
        unsigned long long pre = 0;                     // [63:32] segments, [31:0] sum of earlier tiles
        for (int hi = tile - 1; hi >= 0; hi -= 32) {
            const int j = hi - lane;
            unsigned long long w = seg_pack(SEG_FLAG_INC, 0u, 0u);
            if (j >= 0) do { w = st[j]; } while (seg_flag(w) == 0);
            const unsigned incm = __ballot_sync(0xffffffffu, seg_flag(w) == SEG_FLAG_INC);
            const int last = incm ? __ffs(incm) - 1 : 31;     // nearest inclusive prefix ends the walk
            unsigned long long mine = lane <= last ? (static_cast<unsigned long long>(seg_nz(w)) << 32) | seg_sum(w) : 0ull;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
            pre += mine;
            if (incm) break;
        }
        if (lane == 0) {
            const uint32_t psum = static_cast<uint32_t>(pre & 0xffffffffull), pnz = static_cast<uint32_t>(pre >> 32);
            if (tile > 0) st[tile] = seg_pack(SEG_FLAG_INC, psum + agg[0], pnz + agg[1]);
            sh_pre[0] = psum;
            sh_pre[1] = pnz;
            sh_pre[2] = agg[2] ? static_cast<uint32_t>(atomicAdd(p.nmulti, static_cast<int>(agg[2]))) : 0u;
        }
    }
    __syncthreads();
    uint32_t run = sh_pre[0] + sh_w[0][warp], seg = sh_pre[1] + sh_w[1][warp], mpos = sh_pre[2] + sh_w[2][warp];
    const unsigned below = (1u << lane) - 1u;
    const int64_t RA = p.U;
#pragma unroll
    for (int k = 0; k < PLAN_SCAN_ITEMS; ++k) {
        const int64_t row = base + 32 * k;
        uint32_t inc = c[k];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        const bool mul = c[k] >= 2 && c[k] <= cap;
        const unsigned nzm = __ballot_sync(0xffffffffu, c[k] != 0);
        const unsigned mm = __ballot_sync(0xffffffffu, mul);
        const uint32_t my_seg = seg + __popc(nzm & below);
        if (row == RA) s.totals[2] = static_cast<int32_t>(my_seg);
        if (c[k] != 0) {
            const uint32_t my_run = run + inc - c[k];
            s.off[row] = static_cast<int32_t>(my_run);
            s.sid[row] = static_cast<int32_t>(my_seg);
            s.seg_row[my_seg] = static_cast<int32_t>(row);
            s.seg_start[my_seg] = static_cast<int32_t>(my_run);
            if (cap > 0 && c[k] > cap) s.long_list[atomicAdd(s.totals + 3, 1)] = static_cast<int32_t>(my_seg);
            if (mul) p.multi[mpos + __popc(mm & below)] = static_cast<int32_t>(my_seg);
        }
        run += __shfl_sync(0xffffffffu, inc, 31);
        seg += __popc(nzm);
        mpos += __popc(mm);
    }
    if (tile == s.ntiles - 1 && threadIdx.x == SEG_SCAN_THREADS - 1) {
        s.totals[0] = static_cast<int32_t>(seg);
        s.totals[1] = static_cast<int32_t>(run);
        s.seg_start[seg] = static_cast<int32_t>(run);
        if (RA >= s.Rpad) s.totals[2] = static_cast<int32_t>(seg);
    }
}

// Places every member at off[row] + slot: independent loads, no atomics.  Members of a row land in
// the order of the count's atomics; plan_sort_kernel restores ascending term order.
__global__ void __launch_bounds__(256) plan_fill_kernel(PlanDev p) {
    const int64_t nth = static_cast<int64_t>(gridDim.x) * blockDim.x;
    const int ubase = p.seg.seg_start[p.seg.totals[2]];     // user-side members come first
    for (int64_t b = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; b < p.B; b += nth) {
        const int64_t u = p.users[b], i = p.items[b], j = p.negs[b];
        if (!plan_ids_ok(p, u, i, j)) continue;
        const int su = p.seg.off[u] + p.slot[b];
        const int useg = p.seg.sid[u];
        const int si = p.seg.off[p.U + i] + p.slot[p.B + b] - ubase;
        const int sj = p.seg.off[p.U + j] + p.slot[2 * p.B + b] - ubase;
        URec r;
        r.b = static_cast<int32_t>(b); r.i = static_cast<int32_t>(i); r.j = static_cast<int32_t>(j); r.pad = 0;
        p.mu[su] = r;
        IRec a; a.t = static_cast<int32_t>(2 * b); a.useg = useg;
        IRec c; c.t = static_cast<int32_t>(2 * b + 1); c.useg = useg;
        p.mi[si] = a;
        p.mi[sj] = c;
    }
}

__device__ __forceinline__ int rec_key(const URec& r) { return r.b; }
__device__ __forceinline__ int rec_key(const IRec& r) { return r.t; }

constexpr int PLAN_SORT_SMALL = 16;

__device__ __forceinline__ URec rec_shfl_xor(const URec& r, int j) {
    URec o;
    o.b = __shfl_xor_sync(0xffffffffu, r.b, j); o.i = __shfl_xor_sync(0xffffffffu, r.i, j);
    o.j = __shfl_xor_sync(0xffffffffu, r.j, j); o.pad = 0;
    return o;
}
__device__ __forceinline__ IRec rec_shfl_xor(const IRec& r, int j) {
    IRec o;
    o.t = __shfl_xor_sync(0xffffffffu, r.t, j); o.useg = __shfl_xor_sync(0xffffffffu, r.useg, j);
    return o;
}
__device__ __forceinline__ void rec_set_key(URec& r, int k) { r.b = k; r.i = 0; r.j = 0; r.pad = 0; }
__device__ __forceinline__ void rec_set_key(IRec& r, int k) { r.t = k; r.useg = 0; }

// Sorts each member list of a 32-segment tile ascending by key (the fill placed members in
// atomic order).  Lists of two: one compare-exchange by the owning lane.  Lists of 3..16: a
// 16-wide bitonic network over half a warp, one record per lane, two lists per pass.  Lists
// up to `cap`: ranked by counting by the whole warp.  Hot rows (> cap): plan_sort_long_one.
// `len` is 0 for the lanes whose segment belongs to the other table.
template <typename Rec>
__device__ __forceinline__ void plan_sort_tile(Rec* base, int start, int len, int cap, Rec* tmp_base) {
    const int lane = threadIdx.x & 31;
    if (len == 2) {
        const Rec x = base[start], y = base[start + 1];
        if (rec_key(x) > rec_key(y)) { base[start] = y; base[start + 1] = x; }
    }
    unsigned net = __ballot_sync(0xffffffffu, len > 2 && len <= PLAN_SORT_SMALL);
    const int half = lane >> 4, lid = lane & 15;
    while (net) {
        const int s0 = __ffs(net) - 1;
        net &= net - 1;
        int s1 = -1;
        if (net) { s1 = __ffs(net) - 1; net &= net - 1; }
        const int mine = half == 0 ? s0 : s1;
        const int m_start = __shfl_sync(0xffffffffu, start, mine < 0 ? 0 : mine);
        const int t_len = __shfl_sync(0xffffffffu, len, mine < 0 ? 0 : mine);     // every lane takes part
        const int m_len = mine < 0 ? 0 : t_len;
        Rec v;
        if (lid < m_len) v = base[m_start + lid];
        else rec_set_key(v, 0x7fffffff);
#pragma unroll
        for (int k = 2; k <= 16; k <<= 1) {
#pragma unroll
            for (int j = k >> 1; j > 0; j >>= 1) {
                const Rec o = rec_shfl_xor(v, j);
                const bool keep_min = ((lid & j) == 0) == ((lid & k) == 0);
                const bool other_smaller = rec_key(o) < rec_key(v);
                if (keep_min == other_smaller) v = o;
            }
        }
        if (lid < m_len) base[m_start + lid] = v;
    }
    // medium lists: the warp ranks one list at a time
    unsigned med = __ballot_sync(0xffffffffu, len > PLAN_SORT_SMALL && len <= cap);
    while (med) {
        const int src = __ffs(med) - 1;
        med &= med - 1;
        const int s_start = __shfl_sync(0xffffffffu, start, src);
        const int s_len = __shfl_sync(0xffffffffu, len, src);
        for (int i = lane; i < s_len; i += 32) {
            const Rec x = base[s_start + i];
            int r = 0;
            for (int m = 0; m < s_len; ++m) r += rec_key(base[s_start + m]) < rec_key(x);
            tmp_base[s_start + r] = x;
        }
        __syncwarp();
        for (int i = lane; i < s_len; i += 32) base[s_start + i] = tmp_base[s_start + i];
        __syncwarp();
    }
}

// Hot rows: keys are distinct and < nbits, so the rank of a record is the number of set bits
// below its key in a bitmap of the list (bitmap -> per-word prefix popcount -> rank).
template <int NT, typename Rec>
__device__ void plan_sort_long_one(Rec* base, Rec* tmp, int start, int len, uint32_t* bits, uint32_t* pre,
                                   int W, uint32_t* sh_scan) {
    const int per = (W + NT - 1) / NT;
    for (int w = threadIdx.x; w < W; w += NT) bits[w] = 0u;
    __syncthreads();
    for (int i = threadIdx.x; i < len; i += NT) {
        const int t = rec_key(base[start + i]);
        atomicOr(bits + (t >> 5), 1u << (t & 31));
    }
    __syncthreads();
    const int lo = threadIdx.x * per, hi = lo + per < W ? lo + per : W;
    uint32_t sum = 0;
    for (int w = lo; w < hi; ++w) sum += __popc(bits[w]);
    sh_scan[threadIdx.x] = sum;
    __syncthreads();
    for (int o = 1; o < NT; o <<= 1) {
        const uint32_t v = threadIdx.x >= o ? sh_scan[threadIdx.x - o] : 0u;
        __syncthreads();
        sh_scan[threadIdx.x] += v;
        __syncthreads();
    }
    uint32_t run = sh_scan[threadIdx.x] - sum;
    for (int w = lo; w < hi; ++w) { pre[w] = run; run += __popc(bits[w]); }
    __syncthreads();
    for (int i = threadIdx.x; i < len; i += NT) {
        const Rec x = base[start + i];
        const int t = rec_key(x);
        const uint32_t r = pre[t >> 5] + __popc(bits[t >> 5] & ((1u << (t & 31)) - 1u));
        tmp[start + r] = x;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < len; i += NT) base[start + i] = tmp[start + i];
    __syncthreads();
}

// The leading SEG_LONG_CTAS blocks sort the hot rows (long_list), one row per block at a time;
// every other warp takes 32 entries of `multi` at a time.  Rows with one member (three quarters
// of the user rows of a uniform batch) are never visited.
constexpr int PLAN_SORT_THREADS = 128;

__global__ void __launch_bounds__(PLAN_SORT_THREADS) plan_sort_kernel(PlanDev p, int cap) {
    __shared__ uint32_t sh_scan[PLAN_SORT_THREADS];
    const int nsegA = p.seg.totals[2];
    const int ubase = p.seg.seg_start[nsegA];
    if (blockIdx.x < SEG_LONG_CTAS) {
        const int nlong = p.seg.totals[3];
        uint32_t* bits = p.bits + static_cast<size_t>(blockIdx.x) * 2 * p.words;
        uint32_t* pre = bits + p.words;
        for (int li = blockIdx.x; li < nlong; li += SEG_LONG_CTAS) {
            const int s = p.seg.long_list[li];
            const int start = p.seg.seg_start[s];
            const int len = p.seg.seg_start[s + 1] - start;
            if (s < nsegA)
                plan_sort_long_one<PLAN_SORT_THREADS, URec>(p.mu, p.mu_tmp, start, len, bits, pre,
                                                            static_cast<int>((p.B + 31) / 32), sh_scan);
            else
                plan_sort_long_one<PLAN_SORT_THREADS, IRec>(p.mi, p.mi_tmp, start - ubase, len, bits, pre,
                                                            static_cast<int>((2 * p.B + 31) / 32), sh_scan);
        }
        return;
    }
    constexpr int WARPS = PLAN_SORT_THREADS / 32;
    const int nmul = *p.nmulti;
    const int lane = threadIdx.x & 31;
    const int ntiles = (nmul + 31) / 32;
    const int wstride = (gridDim.x - SEG_LONG_CTAS) * WARPS;
    for (int tile = (blockIdx.x - SEG_LONG_CTAS) * WARPS + (threadIdx.x >> 5); tile < ntiles; tile += wstride) {
        const int k = tile * 32 + lane;
        int s = -1, start = 0, len = 0;
        if (k < nmul) { s = p.multi[k]; start = p.seg.seg_start[s]; len = p.seg.seg_start[s + 1] - start; }
        // a tile mixes user and item segments: two passes with the other side masked
        plan_sort_tile<URec>(p.mu, start, (s >= 0 && s < nsegA) ? len : 0, cap, p.mu_tmp);
        plan_sort_tile<IRec>(p.mi, start - ubase, s >= nsegA ? len : 0, cap, p.mi_tmp);
    }
}

// ------------------------------------------------------------------ optimizer

// ------------------------------------------------------------------ user side (forward + dU + update)

#ifndef V2_UMINB
#define V2_UMINB 8
#endif
#ifndef V2_UMINB2
#define V2_UMINB2 6
#endif
#ifndef V2_UVPL
#define V2_UVPL 2
#endif
#ifndef V2_UPF
#define V2_UPF 0
#endif

// A lane holds VPL 128-bit pieces of a row: columns gl*4 + v*LPR*4 (every load of a group covers
// whole 128-byte lines).  VPL = 2 halves the lanes per row, so a warp iteration carries twice the
// segments -- twice the bytes in flight per warp, one shuffle level less per reduction.
template <int VPL>
struct RowV { float4 v[VPL]; };

template <int LPR, int VPL>
__device__ __forceinline__ RowV<VPL> row_ldg(const float* row, int gl) {
    RowV<VPL> r;
#pragma unroll
    for (int q = 0; q < VPL; ++q) r.v[q] = ldg4(row + gl * 4 + q * LPR * 4);
    return r;
}
template <int LPR, int VPL>
__device__ __forceinline__ RowV<VPL> row_ldcs(const float* row, int gl) {
    RowV<VPL> r;
#pragma unroll
    for (int q = 0; q < VPL; ++q) r.v[q] = __ldcs(reinterpret_cast<const float4*>(row + gl * 4 + q * LPR * 4));
    return r;
}
template <int VPL>
__device__ __forceinline__ RowV<VPL> row_zero() {
    RowV<VPL> r;
#pragma unroll
    for (int q = 0; q < VPL; ++q) r.v[q] = make_float4(0.f, 0.f, 0.f, 0.f);
    return r;
}

// One interaction of a user segment: two dots, loss, d loss / d score, gradient accumulation.
// FULL: the whole warp is converged on this call (every group runs it), so the group reductions
// shuffle under the constant full mask -- plain SHFL.BFLY, no per-shuffle WARPSYNC / MATCH
// sequence that a run-time group mask compiles to.
template <int LPR, int VPL, int LOSS, bool FULL>
__device__ __forceinline__ void user_member(const RowV<VPL>& w, float ub, const RowV<VPL>& qi, const RowV<VPL>& qj,
                                            float bi_, float bj_, int b, float invB, unsigned gmask, int gl,
                                            float* t_g, RowV<VPL>& acc, float& bacc, bool& nz, float& lsum) {
    float dp = 0.f, dn = 0.f;
#pragma unroll
    for (int q = 0; q < VPL; ++q) { dp += dot4(w.v[q], qi.v[q]); dn += dot4(w.v[q], qj.v[q]); }
    dp = group_sum<LPR>(dp, FULL ? 0xffffffffu : gmask);
    dn = group_sum<LPR>(dn, FULL ? 0xffffffffu : gmask);
    float per, gp, gn;
    pair_loss(LOSS, dp + ub + bi_, dn + ub + bj_, per, gp, gn);
    gp *= invB; gn *= invB;
    if (gl == 0) {
        lsum += per;
        *reinterpret_cast<float2*>(t_g + 2 * static_cast<int64_t>(b)) = make_float2(gp, gn);
    }
#pragma unroll
    for (int q = 0; q < VPL; ++q) { fma4(acc.v[q], gp, qi.v[q]); fma4(acc.v[q], gn, qj.v[q]); }
    bacc += gp + gn;
    nz = nz || gp != 0.f || gn != 0.f;
}

// Stash the pre-update row for the item side, apply the optimizer in place.  The weight and
// state rows stream through (evict-first loads / stores): they are touched once per step,
// while the stash is re-read by mf_item_kernel and the item table by every other segment.
template <int LPR, int VPL>
__device__ __forceinline__ void user_finish(const MfDev& a, const OptV2& o, float* stash_row, float* wrow, float* srow,
                                            RowV<VPL> w, RowV<VPL> s, const RowV<VPL>& acc, float bacc, bool nz,
                                            int row, int gl) {
#pragma unroll
    for (int q = 0; q < VPL; ++q) st4(stash_row + gl * 4 + q * LPR * 4, w.v[q]);
    if (nz) {                                        // all-zero gradients leave the row untouched
#pragma unroll
        for (int q = 0; q < VPL; ++q) {
            row_update(o, w.v[q], s.v[q], acc.v[q]);
            __stcs(reinterpret_cast<float4*>(wrow + gl * 4 + q * LPR * 4), w.v[q]);
            if (srow) __stcs(reinterpret_cast<float4*>(srow + gl * 4 + q * LPR * 4), s.v[q]);
        }
        if (gl == 0) bias_update(o, a.bu + row, a.sbu ? a.sbu + row : nullptr, bacc);
    }
}

template <int LPR, int VPL, int LOSS, int TI>
__global__ void __launch_bounds__(MF_TILE_THREADS, (VPL == 1 ? V2_UMINB : V2_UMINB2)) mf_user_kernel(MfDev a, PlanDev p, StepV2 v, int n_long_partials) {
    constexpr int D = LPR * 4 * VPL;
    constexpr int GPW = 32 / LPR;
    constexpr int WARPS = MF_TILE_THREADS / 32;
    __shared__ float sh_red[WARPS];
    __shared__ int sh_inv[WARPS][32];
    __shared__ bool is_last;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int gl = lane & (LPR - 1);
    const int grp = lane / LPR;
    const unsigned gmask = group_mask(LPR);
    const unsigned below = (1u << lane) - 1u;
    const float invB = 1.0f / static_cast<float>(a.NB);
    const OptV2 o = {a.opt, a.lr, a.wd, a.eps};
    const int nsegA = p.seg.totals[2];
    const int ntiles = (nsegA + TI - 1) / TI;
    const int wstride = gridDim.x * WARPS;
    const int cap = p.seg.long_cap;
    const bool adagrad = a.opt == SLB_OPT_ADAGRAD;
    float lsum = 0.f;

    for (int tile = blockIdx.x * WARPS + warp; tile < ntiles; tile += wstride) {
        const int sidx = tile * TI + lane;
        const bool valid = lane < TI && sidx < nsegA;
        int start = 0, len = 0, row = 0;
        int4 r0 = make_int4(0, 0, 0, 0), r1 = r0;
        if (valid) {
            start = p.seg.seg_start[sidx];
            len = p.seg.seg_start[sidx + 1] - start;
            row = p.seg.seg_row[sidx];
            r0 = __ldg(reinterpret_cast<const int4*>(p.mu + start));
            if (len == 2) r1 = __ldg(reinterpret_cast<const int4*>(p.mu + start + 1));
#if V2_UPF
            // experiment: ask L2 for this segment's weight / state rows a whole tile ahead
            pf_row_l2(a.Wu + static_cast<int64_t>(row) * D, D);
            if (adagrad) pf_row_l2(a.sWu + static_cast<int64_t>(row) * D, D);
#endif
        }
        // Order the tile's segments by length class (1, 2, longer, none) so that a whole warp
        // iteration runs one specialised, unpredicated code path: three quarters of the user
        // rows of a uniform batch have one interaction, a fifth have two.
        const unsigned m1 = __ballot_sync(0xffffffffu, len == 1);
        const unsigned m2 = __ballot_sync(0xffffffffu, len == 2);
        const unsigned m3 = __ballot_sync(0xffffffffu, len > 2);
        const int n1 = __popc(m1), n2 = __popc(m2), n3 = __popc(m3);
        int pos;
        if (len == 1) pos = __popc(m1 & below);
        else if (len == 2) pos = n1 + __popc(m2 & below);
        else if (len > 2) pos = n1 + n2 + __popc(m3 & below);
        else pos = n1 + n2 + n3 + __popc(~(m1 | m2 | m3) & below);
        __syncwarp();
        sh_inv[warp][pos] = lane;
        __syncwarp();
        const int nvalid = n1 + n2 + n3;

        for (int q0 = 0; q0 < nvalid; q0 += GPW) {
            const int q = q0 + grp;
            const int src = sh_inv[warp][q & 31];
            const int s_len = __shfl_sync(0xffffffffu, len, src);
            const int s_row = __shfl_sync(0xffffffffu, row, src);
            const int b0 = __shfl_sync(0xffffffffu, r0.x, src);
            const int i0 = __shfl_sync(0xffffffffu, r0.y, src);
            const int j0 = __shfl_sync(0xffffffffu, r0.z, src);
            const int s = tile * TI + src;
            float* wrow = a.Wu + static_cast<int64_t>(s_row) * D;
            float* srow = adagrad ? a.sWu + static_cast<int64_t>(s_row) * D : nullptr;
            float* stash_row = v.stash + static_cast<int64_t>(s) * D;
            RowV<VPL> acc = row_zero<VPL>();
            float bacc = 0.f;
            bool nz = false;
            if (q0 + GPW <= n1) {
                // ---- every group of the warp: one interaction
                const RowV<VPL> w = row_ldcs<LPR, VPL>(wrow, gl);
                RowV<VPL> st_ = row_zero<VPL>();
                if (adagrad) st_ = row_ldcs<LPR, VPL>(srow, gl);
                const RowV<VPL> qi = row_ldg<LPR, VPL>(a.Wi + static_cast<int64_t>(i0) * D, gl);
                const RowV<VPL> qj = row_ldg<LPR, VPL>(a.Wi + static_cast<int64_t>(j0) * D, gl);
                const float ub = a.bu[s_row], bi_ = __ldg(a.bi + i0), bj_ = __ldg(a.bi + j0);
                user_member<LPR, VPL, LOSS, true>(w, ub, qi, qj, bi_, bj_, b0, invB, gmask, gl, v.t_g, acc, bacc, nz, lsum);
                user_finish<LPR, VPL>(a, o, stash_row, wrow, srow, w, st_, acc, bacc, nz, s_row, gl);
            } else if (q0 >= n1 && q0 + GPW <= n1 + n2) {
                // ---- every group of the warp: two interactions
                const int b1 = __shfl_sync(0xffffffffu, r1.x, src);
                const int i1 = __shfl_sync(0xffffffffu, r1.y, src);
                const int j1 = __shfl_sync(0xffffffffu, r1.z, src);
                const RowV<VPL> w = row_ldcs<LPR, VPL>(wrow, gl);
                RowV<VPL> st_ = row_zero<VPL>();
                if (adagrad) st_ = row_ldcs<LPR, VPL>(srow, gl);
                const RowV<VPL> qi0 = row_ldg<LPR, VPL>(a.Wi + static_cast<int64_t>(i0) * D, gl);
                const RowV<VPL> qj0 = row_ldg<LPR, VPL>(a.Wi + static_cast<int64_t>(j0) * D, gl);
                const float ub = a.bu[s_row];
                const float bi0 = __ldg(a.bi + i0), bj0 = __ldg(a.bi + j0), bi1 = __ldg(a.bi + i1), bj1 = __ldg(a.bi + j1);
                user_member<LPR, VPL, LOSS, true>(w, ub, qi0, qj0, bi0, bj0, b0, invB, gmask, gl, v.t_g, acc, bacc, nz, lsum);
                const RowV<VPL> qi1 = row_ldg<LPR, VPL>(a.Wi + static_cast<int64_t>(i1) * D, gl);
                const RowV<VPL> qj1 = row_ldg<LPR, VPL>(a.Wi + static_cast<int64_t>(j1) * D, gl);
                user_member<LPR, VPL, LOSS, true>(w, ub, qi1, qj1, bi1, bj1, b1, invB, gmask, gl, v.t_g, acc, bacc, nz, lsum);
                user_finish<LPR, VPL>(a, o, stash_row, wrow, srow, w, st_, acc, bacc, nz, s_row, gl);
            } else {
                // ---- mixed iteration (class boundaries, lists of 3+): group-divergent generic path
                const int s_start = __shfl_sync(0xffffffffu, start, src);
                if (q >= nvalid || s_len > cap) continue;         // idle group / hot row (mf_user_long_kernel)
                const RowV<VPL> w = row_ldcs<LPR, VPL>(wrow, gl);
                RowV<VPL> st_ = row_zero<VPL>();
                if (adagrad) st_ = row_ldcs<LPR, VPL>(srow, gl);
                const float ub = a.bu[s_row];
                for (int k = 0; k < s_len; ++k) {
                    // every lane of the group reads the same (sorted) record: one broadcast transaction
                    const int4 r = __ldg(reinterpret_cast<const int4*>(p.mu + s_start + k));
                    const RowV<VPL> qi = row_ldg<LPR, VPL>(a.Wi + static_cast<int64_t>(r.y) * D, gl);
                    const RowV<VPL> qj = row_ldg<LPR, VPL>(a.Wi + static_cast<int64_t>(r.z) * D, gl);
                    user_member<LPR, VPL, LOSS, false>(w, ub, qi, qj, __ldg(a.bi + r.y), __ldg(a.bi + r.z), r.x, invB, gmask,
                                                       gl, v.t_g, acc, bacc, nz, lsum);
                }
                user_finish<LPR, VPL>(a, o, stash_row, wrow, srow, w, st_, acc, bacc, nz, s_row, gl);
            }
        }
    }

    // deterministic loss reduction: fixed tree per block, fixed order over blocks (+ hot-row partials)
    const float bsum = block_sum<MF_TILE_THREADS>(lsum, sh_red);
    if (threadIdx.x == 0) {
        v.partial[blockIdx.x] = bsum;
        __threadfence();
        is_last = atomicAdd(v.done, 1) == static_cast<int>(gridDim.x) - 1;
    }
    __syncthreads();
    if (is_last && threadIdx.x < 32) {
        __threadfence();
        float t = 0.f;
        for (int k = threadIdx.x; k < static_cast<int>(gridDim.x); k += 32)
            t += *reinterpret_cast<volatile float*>(v.partial + k);
        for (int k = threadIdx.x; k < n_long_partials; k += 32)
            t += *reinterpret_cast<volatile float*>(v.partial_long + k);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) t += __shfl_down_sync(0xffffffffu, t, off);
        if (threadIdx.x == 0) { *a.loss_out = t * invB; *v.done = 0; }
    }
}

// Hot user rows (more interactions in this batch than the tile kernel's cap): one CTA per row,
// each lane group scores a contiguous chunk of the sorted member list, chunk partials are
// combined in chunk order.  Runs before mf_user_kernel (its loss partials are folded there).
template <int LPR, int LOSS>
__global__ void __launch_bounds__(256) mf_user_long_kernel(MfDev a, PlanDev p, StepV2 v) {
    constexpr int D = LPR * 4;
    constexpr int GROUPS = 256 / LPR;
    constexpr int PS = D + 4;
    extern __shared__ float sh_part[];            // [GROUPS][D + 4]
    __shared__ float sh_red[8];
    const int gl = threadIdx.x & (LPR - 1);
    const int gq = threadIdx.x / LPR;
    const int c = gl * 4;
    const unsigned gmask = group_mask(LPR);
    const float invB = 1.0f / static_cast<float>(a.NB);
    const OptV2 o = {a.opt, a.lr, a.wd, a.eps};
    const int nlong = p.seg.totals[3];
    const int nsegA = p.seg.totals[2];
    float lsum = 0.f;
    for (int li = blockIdx.x; li < nlong; li += gridDim.x) {
        const int s = p.seg.long_list[li];
        if (s >= nsegA) continue;                 // block-uniform
        const int start = p.seg.seg_start[s];
        const int len = p.seg.seg_start[s + 1] - start;
        const int row = p.seg.seg_row[s];
        float* wrow = a.Wu + static_cast<int64_t>(row) * D + c;
        const float4 w4 = ld4(wrow);
        const float ub = a.bu[row];
        const int chunk = (len + GROUPS - 1) / GROUPS;
        const int lo = min(gq * chunk, len), hi = min(lo + chunk, len);
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        float bacc = 0.f, nzf = 0.f;
        for (int k = lo; k < hi; ++k) {
            const int4 r0 = __ldg(reinterpret_cast<const int4*>(p.mu + start + k));
            const float4 a0 = ldg4(a.Wi + static_cast<int64_t>(r0.y) * D + c), b0 = ldg4(a.Wi + static_cast<int64_t>(r0.z) * D + c);
            const float dp = group_sum<LPR>(dot4(w4, a0), gmask);
            const float dn = group_sum<LPR>(dot4(w4, b0), gmask);
            float per, gp, gn;
            pair_loss(LOSS, dp + ub + __ldg(a.bi + r0.y), dn + ub + __ldg(a.bi + r0.z), per, gp, gn);
            gp *= invB; gn *= invB;
            if (gl == 0) {
                lsum += per;
                *reinterpret_cast<float2*>(v.t_g + 2 * static_cast<int64_t>(r0.x)) = make_float2(gp, gn);
            }
            fma4(acc, gp, a0);
            fma4(acc, gn, b0);
            bacc += gp + gn;
            if (gp != 0.f || gn != 0.f) nzf = 1.f;
        }
        st4(sh_part + gq * PS + c, acc);
        if (gl == 0) { sh_part[gq * PS + D] = bacc; sh_part[gq * PS + D + 1] = nzf; }
        __syncthreads();
        if (gq == 0) {
            float4 tot = make_float4(0.f, 0.f, 0.f, 0.f);
            float bt = 0.f, nzt = 0.f;
            for (int q = 0; q < GROUPS; ++q) {
                const float4 x = ld4(sh_part + q * PS + c);
                tot.x += x.x; tot.y += x.y; tot.z += x.z; tot.w += x.w;
                bt += sh_part[q * PS + D];
                nzt += sh_part[q * PS + D + 1];
            }
            st4(v.stash + static_cast<int64_t>(s) * D + c, w4);
            if (nzt != 0.f) {
                float4 wn = w4, s4 = make_float4(0.f, 0.f, 0.f, 0.f);
                float* srow = a.opt == SLB_OPT_ADAGRAD ? a.sWu + static_cast<int64_t>(row) * D + c : nullptr;
                if (srow) s4 = ld4(srow);
                row_update(o, wn, s4, tot);
                st4(wrow, wn);
                if (srow) st4(srow, s4);
                if (gl == 0) bias_update(o, a.bu + row, a.sbu ? a.sbu + row : nullptr, bt);
            }
        }
        __syncthreads();
    }
    const float bsum = block_sum<256>(lsum, sh_red);
    if (threadIdx.x == 0) v.partial_long[blockIdx.x] = bsum;
}

// ------------------------------------------------------------------ item side (dQ + update)

#ifndef V2_IFAST
#define V2_IFAST 4
#endif
#ifndef V2_IMINB
#define V2_IMINB 6
#endif
#ifndef V2_ICHUNK
#define V2_ICHUNK 8
#endif

template <int LPR, int TI>
__global__ void __launch_bounds__(MF_TILE_THREADS, V2_IMINB) mf_item_kernel(MfDev a, PlanDev p, StepV2 v) {
    constexpr int D = LPR * 4;
    constexpr int GPW = 32 / LPR;
    constexpr int ITERS = TI / GPW > 0 ? TI / GPW : 1;
    constexpr int WARPS = MF_TILE_THREADS / 32;
    constexpr int CAP = seg_sort_cap(LPR);
    __shared__ int32_t sh_all[WARPS * GPW * 2 * CAP];
    const int lane = threadIdx.x & 31;
    const int gl = lane & (LPR - 1);
    const int grp = lane / LPR;
    const int c = gl * 4;
    const unsigned gmask = group_mask(LPR);
    int32_t* sh = sh_all + ((threadIdx.x >> 5) * GPW + grp) * 2 * CAP;
    const OptV2 o = {a.opt, a.lr, a.wd, a.eps};
    const int nseg = p.seg.totals[0];
    const int nsegA = p.seg.totals[2];
    const int ubase = p.seg.seg_start[nsegA];
    const int ntiles = (nseg - nsegA + TI - 1) / TI;
    const int wstride = gridDim.x * WARPS;
    const float* __restrict__ t_g = v.t_g;

    for (int tile = blockIdx.x * WARPS + (threadIdx.x >> 5); tile < ntiles; tile += wstride) {
        const int sidx = nsegA + tile * TI + lane;
        const bool valid = lane < TI && sidx < nseg;
        int start = 0, len = 0, row = 0;
        int pu[V2_IFAST] = {};
        float pg[V2_IFAST] = {};
        if (valid) {
            start = p.seg.seg_start[sidx] - ubase;
            len = p.seg.seg_start[sidx + 1] - ubase - start;
            row = p.seg.seg_row[sidx] - static_cast<int>(a.U);
            if (len <= V2_IFAST) {
#pragma unroll
                for (int k = 0; k < V2_IFAST; ++k)
                    if (k < len) {
                        const int2 r = __ldg(reinterpret_cast<const int2*>(p.mi + start + k));
                        pu[k] = r.y;
                        pg[k] = t_g[r.x];
                    }
            }
        }
        for (int it = 0; it < ITERS; ++it) {
            const int src = it * GPW + grp;
            const int s_len = __shfl_sync(0xffffffffu, len, src & 31);
            const int s_row = __shfl_sync(0xffffffffu, row, src & 31);
            const int s_start = __shfl_sync(0xffffffffu, start, src & 31);
            int su[V2_IFAST];
            float sg[V2_IFAST];
#pragma unroll
            for (int k = 0; k < V2_IFAST; ++k) {
                su[k] = __shfl_sync(0xffffffffu, pu[k], src & 31);
                sg[k] = __shfl_sync(0xffffffffu, pg[k], src & 31);
            }
            const int s = nsegA + tile * TI + src;
            if (src >= TI || s >= nseg) continue;             // group-uniform
            if (s_len > CAP) continue;                        // hot row: mf_item_long_kernel
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            float bacc = 0.f;
            bool nz = false;
            if (s_len <= V2_IFAST) {
                float4 x[V2_IFAST];
#pragma unroll
                for (int k = 0; k < V2_IFAST; ++k)
                    if (k < s_len) x[k] = ld4(v.stash + static_cast<int64_t>(su[k]) * D + c);
#pragma unroll
                for (int k = 0; k < V2_IFAST; ++k)
                    if (k < s_len) { fma4(acc, sg[k], x[k]); bacc += sg[k]; nz = nz || sg[k] != 0.f; }
            } else {
                float* lg = reinterpret_cast<float*>(sh);
                int32_t* lu = sh + CAP;
                for (int i = gl; i < s_len; i += LPR) {
                    const int2 r = __ldg(reinterpret_cast<const int2*>(p.mi + s_start + i));
                    lg[i] = t_g[r.x];
                    lu[i] = r.y;
                    pf_row_l2(v.stash + static_cast<int64_t>(r.y) * D, D);      // the walk below then runs at L2 latency
                }
                __syncwarp(gmask);
                int i = 0;
                for (; i + V2_ICHUNK <= s_len; i += V2_ICHUNK) {
                    float4 x[V2_ICHUNK];
#pragma unroll
                    for (int k = 0; k < V2_ICHUNK; ++k) x[k] = ld4(v.stash + static_cast<int64_t>(lu[i + k]) * D + c);
#pragma unroll
                    for (int k = 0; k < V2_ICHUNK; ++k) { fma4(acc, lg[i + k], x[k]); bacc += lg[i + k]; nz = nz || lg[i + k] != 0.f; }
                }
                for (; i < s_len; ++i) {
                    fma4(acc, lg[i], ld4(v.stash + static_cast<int64_t>(lu[i]) * D + c));
                    bacc += lg[i];
                    nz = nz || lg[i] != 0.f;
                }
                __syncwarp(gmask);                            // scratch is reused by the next segment
            }
            if (a.dWi) {
                // item rows owned elsewhere (multi-GPU): hand the gradient out, dense, caller-zeroed
                st4(a.dWi + static_cast<int64_t>(s_row) * D + c, acc);
                if (gl == 0) a.dbi[s_row] = bacc;
            } else if (nz) {
                float* wrow = a.Wi + static_cast<int64_t>(s_row) * D + c;
                float* srow = a.opt == SLB_OPT_ADAGRAD ? a.sWi + static_cast<int64_t>(s_row) * D + c : nullptr;
                float4 w4 = ld4(wrow);
                float4 s4 = make_float4(0.f, 0.f, 0.f, 0.f);
                if (srow) s4 = ld4(srow);
                row_update(o, w4, s4, acc);
                st4(wrow, w4);
                if (srow) st4(srow, s4);
                if (gl == 0) bias_update(o, a.bi + s_row, a.sbi ? a.sbi + s_row : nullptr, bacc);
            }
        }
    }
}

template <int LPR>
__global__ void __launch_bounds__(256) mf_item_long_kernel(MfDev a, PlanDev p, StepV2 v) {
    constexpr int D = LPR * 4;
    constexpr int GROUPS = 256 / LPR;
    constexpr int PS = D + 4;
    extern __shared__ float sh_part[];            // [GROUPS][D + 4]
    const int gl = threadIdx.x & (LPR - 1);
    const int gq = threadIdx.x / LPR;
    const int c = gl * 4;
    const OptV2 o = {a.opt, a.lr, a.wd, a.eps};
    const int nlong = p.seg.totals[3];
    const int nsegA = p.seg.totals[2];
    const int ubase = p.seg.seg_start[nsegA];
    for (int li = blockIdx.x; li < nlong; li += gridDim.x) {
        const int s = p.seg.long_list[li];
        if (s < nsegA) continue;                  // block-uniform
        const int start = p.seg.seg_start[s] - ubase;
        const int len = p.seg.seg_start[s + 1] - ubase - start;
        const int row = p.seg.seg_row[s] - static_cast<int>(a.U);
        const int chunk = (len + GROUPS - 1) / GROUPS;
        const int lo = min(gq * chunk, len), hi = min(lo + chunk, len);
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        float bacc = 0.f, nzf = 0.f;
        int i = lo;
        for (; i + 4 <= hi; i += 4) {
            int2 r[4]; float g[4]; float4 x[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) r[k] = __ldg(reinterpret_cast<const int2*>(p.mi + start + i + k));
#pragma unroll
            for (int k = 0; k < 4; ++k) { g[k] = v.t_g[r[k].x]; x[k] = ld4(v.stash + static_cast<int64_t>(r[k].y) * D + c); }
#pragma unroll
            for (int k = 0; k < 4; ++k) { fma4(acc, g[k], x[k]); bacc += g[k]; if (g[k] != 0.f) nzf = 1.f; }
        }
        for (; i < hi; ++i) {
            const int2 r = __ldg(reinterpret_cast<const int2*>(p.mi + start + i));
            const float g = v.t_g[r.x];
            fma4(acc, g, ld4(v.stash + static_cast<int64_t>(r.y) * D + c));
            bacc += g;
            if (g != 0.f) nzf = 1.f;
        }
        st4(sh_part + gq * PS + c, acc);
        if (gl == 0) { sh_part[gq * PS + D] = bacc; sh_part[gq * PS + D + 1] = nzf; }
        __syncthreads();
        if (gq == 0) {
            float4 tot = make_float4(0.f, 0.f, 0.f, 0.f);
            float bt = 0.f, nzt = 0.f;
            for (int q = 0; q < GROUPS; ++q) {
                const float4 x = ld4(sh_part + q * PS + c);
                tot.x += x.x; tot.y += x.y; tot.z += x.z; tot.w += x.w;
                bt += sh_part[q * PS + D];
                nzt += sh_part[q * PS + D + 1];
            }
            if (a.dWi) {
                st4(a.dWi + static_cast<int64_t>(row) * D + c, tot);
                if (gl == 0) a.dbi[row] = bt;
            } else if (nzt != 0.f) {
                float* wrow = a.Wi + static_cast<int64_t>(row) * D + c;
                float* srow = a.opt == SLB_OPT_ADAGRAD ? a.sWi + static_cast<int64_t>(row) * D + c : nullptr;
                float4 w4 = ld4(wrow), s4 = make_float4(0.f, 0.f, 0.f, 0.f);
                if (srow) s4 = ld4(srow);
                row_update(o, w4, s4, tot);
                st4(wrow, w4);
                if (srow) st4(srow, s4);
                if (gl == 0) bias_update(o, a.bi + row, a.sbi ? a.sbi + row : nullptr, bt);
            }
        }
        __syncthreads();
    }
}

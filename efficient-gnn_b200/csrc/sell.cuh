// Column-blocked sliced-ELL ("SELL-32, 16-bit local indices") path for the
// narrow (F = 1) Chebyshev orders - the reference's default configuration
// (X0 = log1p(degree), calibration/WATS.py:58-59) on graphs whose CSR streams
// from HBM (Reddit shape: 114.6 M entries, 459 MB of int32 indices per order).
//
// Why: with F = 1 every stored entry costs one 4-byte random gather of
// T_{k-1}[j].  Through L1/L2 that gather rate (~1.5 per clock per SM, one
// 128-byte line per wavefront) is 8x short of what HBM can stream.  Shared
// memory serves ~9 random 4-byte reads per clock per SM, so the operand vector
// is staged in shared memory one COLUMN BLOCK (<= 49152 floats) at a time and
// the matrix is re-laid-out once per graph so that
//   * entries are grouped by column block and carry 16-bit block-local column
//     indices (halves the index stream: 2 B per entry),
//   * rows are cut into "virtual rows" of <= lmax entries (hub rows split, so
//     power-law graphs balance), sorted by length and packed 32 to a slice in
//     lane-interleaved order: lane r of a warp walks virtual row r with 16-byte
//     loads (8 indices), the warp's loads are one contiguous 512-byte segment,
//   * stored self loops and padding point at zero slots, so the inner loop has
//     no predicate: load 8 indices -> 8 LDS -> 8 FADD,
//   * the order of the entries inside a virtual row is free, so it is chosen
//     to spread the warp's 32 simultaneous gathers over the 32 banks (greedy
//     edge colouring of lanes x banks per slice, see sell_fill_kernel), and the slices of a
//     block are stored longest first: the hot kernel hands them out dynamically,
//     so the short ones at the end of a block's queue keep the tail short.
// This file: the plan build and the gather primitives.  The hot kernel
// (sell_step.cuh) runs all orders of a step in one persistent launch: every CTA
// serves one column block, warps pull slices from a per-block counter, one
// partial sum per virtual row goes to a row-major array, and after a grid
// barrier the same kernel adds each row's partials in a fixed order
// (deterministic) and applies the Laplacian scaling, the three-term recurrence
// and the scale accumulation.
#pragma once

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "cheb.cuh"
#include "common.cuh"
#include "peer.cuh"

namespace egnn {

constexpr int kSellThreads = 1024;
constexpr int kSellThreadsPerCta = kSellThreads;
constexpr int kSellCtrStride = 32;        // one 128-byte line per column block's slice counter
constexpr int kSellSchedWords = 64 * kSellCtrStride + 64;   // counters, then the grid-barrier counter
constexpr int kSellSliceRows = 32;
constexpr int kSellGroup = 8;           // indices per 16-byte load
constexpr int kSellMaxBlocks = 64;

// totals the host needs after the prepare pass (device int64[8])
enum SellTotals { kTotU = 0, kTotV = 1, kTotSlices = 2, kTotEntries = 3, kTotRowV = 4, kTotHub = 5 };

// ---- build pass 1: per (column block, row) segment of the sorted CSR row ----
__global__ void __launch_bounds__(256)
sell_count_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx, int n, int C,
                  int CB, int lmax, int32_t* __restrict__ seg_start, int32_t* __restrict__ seg_cnt,
                  int32_t* __restrict__ nv, int32_t* __restrict__ nvrow) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int e = rowptr[i + 1];
    int prev = rowptr[i];
    int total = 0;
    for (int c = 0; c < C; ++c) {
        int pos = e;
        if (c + 1 < C) {                       // first position with column >= (c+1)*CB
            const int bound = (c + 1) * CB;
            int lo = prev, hi = e;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (__ldg(colidx + mid) < bound) lo = mid + 1; else hi = mid;
            }
            pos = lo;
        }
        const int cnt = pos - prev;
        const int v = (cnt + lmax - 1) / lmax;
        seg_start[(size_t)c * n + i] = prev;
        seg_cnt[(size_t)c * n + i] = cnt;
        nv[(size_t)c * n + i] = v;
        total += v;
        prev = pos;
    }
    nvrow[i] = total;
}

// ---- build pass 2: one record per virtual row -------------------------------
__global__ void __launch_bounds__(256)
sell_emit_kernel(int n, int C, int lmax, const int32_t* __restrict__ seg_start,
                 const int32_t* __restrict__ seg_cnt, const int32_t* __restrict__ nv,
                 const int32_t* __restrict__ u_off, const int32_t* __restrict__ rv_ptr,
                 uint32_t* __restrict__ key, int32_t* __restrict__ uval, int32_t* __restrict__ vsrc,
                 int32_t* __restrict__ vslot, int32_t* __restrict__ vrow) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (int64_t)C * n) return;
    const int c = (int)(t / n), i = (int)(t % n);
    const int cnt = seg_cnt[t];
    if (cnt == 0) return;
    int slot = rv_ptr[i];
    for (int cc = 0; cc < c; ++cc) slot += nv[(size_t)cc * n + i];
    const int u0 = u_off[t];
    const int start = seg_start[t];
    const int chunks = nv[t];
    for (int j = 0; j < chunks; ++j) {
        const int len = min(lmax, cnt - j * lmax);
        const int u = u0 + j;
        key[u] = ((uint32_t)c << 16) | (uint32_t)(lmax - len);     // block-major, longest first
        uval[u] = u;
        vsrc[u] = start + j * lmax;
        vslot[u] = slot + j;
        vrow[u] = i;
    }
}

// ---- build pass 3: block pointers (padded to whole slices) ------------------
// Slices of a block are stored in the order of their length rank (longest
// first); blk_stride stays in the layout as a coprime multiplier of the rank
// (1 now; a golden-ratio stride served the earlier static split of slices).
__global__ void sell_blocks_kernel(int n, int C, const int32_t* __restrict__ u_off,
                                   int32_t* __restrict__ q_ptr, int32_t* __restrict__ vp_ptr,
                                   int32_t* __restrict__ blk_slice_ptr, int32_t* __restrict__ blk_stride,
                                   int64_t* __restrict__ totals) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    int vp = 0;
    for (int c = 0; c < C; ++c) {
        const int q0 = u_off[(size_t)c * n];
        const int q1 = u_off[(size_t)(c + 1) * n];
        q_ptr[c] = q0;
        vp_ptr[c] = vp;
        blk_slice_ptr[c] = vp / kSellSliceRows;
        const int n_c = (q1 - q0 + kSellSliceRows - 1) / kSellSliceRows;
        blk_stride[c] = 1;
        vp += n_c * kSellSliceRows;
    }
    q_ptr[C] = u_off[(size_t)C * n];
    vp_ptr[C] = vp;
    blk_slice_ptr[C] = vp / kSellSliceRows;
    totals[kTotU] = q_ptr[C];
    totals[kTotV] = vp;
    totals[kTotSlices] = vp / kSellSliceRows;
}

__device__ __forceinline__ int sell_block_of_slice(const int32_t* blk_slice_ptr, int C, int s) {
    int c = 0;
    while (c + 1 < C && s >= blk_slice_ptr[c + 1]) ++c;
    return c;
}

// length rank (in slices) of the rows stored in slice s of block c
__device__ __forceinline__ int sell_rank_of_slice(const int32_t* blk_slice_ptr, const int32_t* blk_stride, int c, int s) {
    const int n_c = blk_slice_ptr[c + 1] - blk_slice_ptr[c];
    return (int)(((int64_t)(s - blk_slice_ptr[c]) * blk_stride[c]) % n_c);
}

// ---- build pass 4: padded size of every slice --------------------------------
__global__ void __launch_bounds__(256)
sell_slice_kernel(int C, int lmax, const uint32_t* __restrict__ key_sorted,
                  const int32_t* __restrict__ q_ptr, const int32_t* __restrict__ blk_slice_ptr,
                  const int32_t* __restrict__ blk_stride, const int64_t* __restrict__ totals,
                  int32_t* __restrict__ slice_sz) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= (int)totals[kTotSlices]) return;
    const int c = sell_block_of_slice(blk_slice_ptr, C, s);
    const int rank0 = sell_rank_of_slice(blk_slice_ptr, blk_stride, c, s) * kSellSliceRows;
    const int len = lmax - (int)(key_sorted[q_ptr[c] + rank0] & 0xffffu);     // longest row of the slice
    slice_sz[s] = (len + kSellGroup - 1) / kSellGroup * kSellGroup * kSellSliceRows;
}

// Which column block every CTA of the hot kernel serves: CTAs are dealt to the
// blocks in proportion to their padded entries (largest remainder; every
// non-empty block gets at least one), so a CTA stages ONE operand block per
// order and the CTAs of a block share its slices dynamically.
// cta_info: [n_cta] block (-1: none), [n_cta] rank of the CTA inside its block,
// [kSellMaxBlocks] start value of the block's slice counter (32 x its CTAs: the
// first slice of every warp is fixed), [n_cta + 1] first row of every CTA's epilogue range
// (sell_cta_rows_kernel).  sched: the counters themselves + the
// grid-barrier counter, initialised here.
__global__ void sell_cta_blocks_kernel(const int32_t* __restrict__ slice_off, const int32_t* __restrict__ blk_slice_ptr,
                                       int C, int n_cta, int32_t* __restrict__ cta_info, unsigned* __restrict__ sched) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    double w[kSellMaxBlocks], total = 0.0;
    int cnt[kSellMaxBlocks];
    for (int c = 0; c < C; ++c) {
        w[c] = (double)(slice_off[blk_slice_ptr[c + 1]] - slice_off[blk_slice_ptr[c]]);
        total += w[c];
    }
    int used = 0;
    for (int c = 0; c < C; ++c) {
        cnt[c] = w[c] > 0 ? max(1, (int)(w[c] / total * n_cta)) : 0;
        used += cnt[c];
    }
    while (used > n_cta) {                           // more non-empty blocks' minimums than CTAs can not happen (C <= 64 < SMs)
        int big = 0;
        for (int c = 1; c < C; ++c) if (cnt[c] > cnt[big]) big = c;
        --cnt[big]; --used;
    }
    while (used < n_cta && total > 0) {              // leftover CTAs go where the load per CTA is highest
        int best = -1;
        double best_load = 0.0;
        for (int c = 0; c < C; ++c)
            if (cnt[c] > 0 && w[c] / cnt[c] > best_load) { best_load = w[c] / cnt[c]; best = c; }
        if (best < 0) break;
        ++cnt[best]; ++used;
    }
    // CTAs of a block are interleaved with the other blocks' (block ids cycle over the grid), so
    // every block's share of the SMs is spread over the whole chip
    int g = 0, max_cnt = 0;
    for (int c = 0; c < C; ++c) max_cnt = max(max_cnt, cnt[c]);
    for (int r = 0; r < max_cnt; ++r)
        for (int c = 0; c < C; ++c)
            if (r < cnt[c]) { cta_info[g] = c; cta_info[n_cta + g] = r; ++g; }
    for (; g < n_cta; ++g) { cta_info[g] = -1; cta_info[n_cta + g] = 0; }
    for (int i = 0; i < kSellSchedWords; ++i) sched[i] = 0u;
    for (int c = 0; c < kSellMaxBlocks; ++c) {
        const int start = c < C ? cnt[c] * (kSellThreadsPerCta / 32) : 0;
        cta_info[2 * n_cta + c] = start;
        sched[c * kSellCtrStride] = (unsigned)start;
    }
}

// Row ranges of the epilogue phases, one per CTA, balanced by cost instead of by row count: a
// row with more than kSellEpiWarpRow partial sums is summed by a whole warp and costs several
// times a row a single thread finishes.  With random node ids the two agree; with ids sorted by
// degree (or hubs clustered any other way) equal row counts left one CTA with every long row
// and the grid barrier waiting for it (measured: +17 us per order on a degree-sorted Reddit shape).
constexpr int kSellEpiWarpRow = 24;
__device__ __forceinline__ bool sell_is_hub_row(const int32_t* rv_ptr, int i) {
    return rv_ptr[i + 1] - rv_ptr[i] > kSellEpiWarpRow;
}

// cost[i] of the epilogue ranges and hub[i] = 1 for the rows a warp sums ([n + 1] each, last 0)
__global__ void sell_row_cost_kernel(const int32_t* __restrict__ rv_ptr, int n, int32_t* __restrict__ cost,
                                     int32_t* __restrict__ hub) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    if (i == n) { cost[i] = 0; hub[i] = 0; return; }
    const int parts = rv_ptr[i + 1] - rv_ptr[i];
    cost[i] = parts > kSellEpiWarpRow ? 28 + parts / 8 : 4;
    hub[i] = parts > kSellEpiWarpRow ? 1 : 0;
}

// number of hub rows (prepare: the caller sizes the plan's hub list with it)
__global__ void sell_hub_count_kernel(const int32_t* __restrict__ rv_ptr, int n, int64_t* __restrict__ totals) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool hub = i < n && sell_is_hub_row(rv_ptr, i);
    const unsigned m = __ballot_sync(0xffffffffu, hub);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(reinterpret_cast<unsigned long long*>(totals + kTotHub), (unsigned long long)__popc(m));
}

// cta_rows[g] = first row of CTA g (g = 0 .. n_cta): the first row whose cost prefix reaches
// g / n_cta of the total (cost_prefix = exclusive sums, [n + 1])
__global__ void sell_cta_rows_kernel(const int32_t* __restrict__ cost_prefix, int n, int n_cta, int32_t* __restrict__ cta_rows) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g > n_cta) return;
    if (g == 0) { cta_rows[0] = 0; return; }
    if (g == n_cta) { cta_rows[g] = n; return; }
    const int64_t target = (int64_t)cost_prefix[n] * g / n_cta;
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (cost_prefix[mid] < target) lo = mid + 1; else hi = mid;
    }
    cta_rows[g] = lo;
}

// The hub rows of every CTA's epilogue range, listed once per plan so that the step kernel hands
// them to its warps statically: CTA g's are hub[n_cta + 1 + hub[g] .. n_cta + 1 + hub[g + 1]),
// ascending (hub_prefix = exclusive sums of the hub flags, [n + 1]).  Grid: max(n, n_cta + 1) threads.
__global__ void sell_cta_hubs_kernel(const int32_t* __restrict__ hub_flag, const int32_t* __restrict__ hub_prefix,
                                     const int32_t* __restrict__ cta_rows, int n, int n_cta, int32_t* __restrict__ hub) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= n_cta) hub[i] = hub_prefix[cta_rows[i]];
    if (i < n && hub_flag[i]) hub[n_cta + 1 + hub_prefix[i]] = i;
}

__global__ void sell_totals_kernel(const int32_t* __restrict__ slice_off, const int32_t* __restrict__ rv_ptr,
                                   int n, int64_t* __restrict__ totals) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    totals[kTotEntries] = slice_off[totals[kTotSlices]];
    totals[kTotRowV] = rv_ptr[n];
}

// ---- build pass 5: write the lane-interleaved 16-bit index stream -----------
// Entry order inside a virtual row is free (the partial sum is a plain sum), so
// it is chosen to keep the hot kernel's shared-memory gathers off each other's
// banks: the warp's LDS for position j reads one entry per lane, so a slice is
// conflict-free when, at every position, the 32 lanes hold 32 different banks
// (bank = local column mod 32).  That is an edge colouring of the bipartite
// multigraph lanes x banks with the positions as colours; it is done greedily
// (first fit): lane r walks its own virtual row, and each entry takes the
// lowest position that is free both in the lane and in the entry's bank.  One
// warp per slice; lanes whose current entries share a bank go one at a time
// (match_any), so a bank's position mask has one writer per round.  The few
// entries (2-5 %) with no common free position take the lane's lowest free
// one; unused positions point at the zero slot of bank (r + j) mod 32 (32 zero
// slots at CB .. CB+31; stored self loops too).  Measured on the Reddit shape:
// 3.7 wavefronts per LDS unordered, 2.5 with a fixed diagonal rule, see
// DESIGN.md for the first-fit figure.  The 16-bit stream is written straight
// to global memory (2-byte stores that L2 merges).
constexpr int kSellFillWarps = 8;
constexpr int kSellLmaxCap = 256;          // longest virtual row
constexpr int kSellMaskWords = kSellLmaxCap / 32;
constexpr size_t kSellFillSmem = (size_t)kSellFillWarps * 32 * kSellMaskWords * sizeof(uint32_t);   // bank masks

__global__ void __launch_bounds__(kSellFillWarps * 32)
sell_fill_kernel(const int32_t* __restrict__ colidx, int C, int CB, int lmax, int n_slices,
                 const uint32_t* __restrict__ key_sorted, const int32_t* __restrict__ perm,
                 const int32_t* __restrict__ vsrc, const int32_t* __restrict__ vslot_u,
                 const int32_t* __restrict__ vrow, const int32_t* __restrict__ q_ptr,
                 const int32_t* __restrict__ vp_ptr, const int32_t* __restrict__ blk_slice_ptr,
                 const int32_t* __restrict__ blk_stride, const int32_t* __restrict__ slice_off,
                 uint16_t* __restrict__ idx, int32_t* __restrict__ vslot_out, int row0) {
    extern __shared__ __align__(16) uint32_t fill_smem[];
    const int lane = threadIdx.x & 31;
    const int wid = threadIdx.x >> 5;
    const int s = blockIdx.x * kSellFillWarps + wid;
    if (s >= n_slices) return;
    uint32_t* bank_used = fill_smem + (size_t)wid * 32 * kSellMaskWords;   // [bank][word]: positions taken in that bank

    const int c = sell_block_of_slice(blk_slice_ptr, C, s);
    const int v = s * kSellSliceRows + lane;                          // storage slot of this lane's virtual row
    const int rank = sell_rank_of_slice(blk_slice_ptr, blk_stride, c, s) * kSellSliceRows + lane;
    const bool valid = rank < (q_ptr[c + 1] - q_ptr[c]);
    int len = 0, src = 0, row = -1, slot = -1;
    if (valid) {
        const int q = q_ptr[c] + rank;
        const int u = perm[q];
        len = lmax - (int)(key_sorted[q] & 0xffffu);
        src = vsrc[u];
        row = vrow[u] + row0;             // global id of the row (diagonal test)
        slot = vslot_u[u];
    }
    vslot_out[v] = slot;                  // -1: padding lane of the block's last slice
    const int off = slice_off[s];
    const int lpad = (slice_off[s + 1] - off) / kSellSliceRows;      // positions per lane
    const int col0 = c * CB;
    // position j of this lane lives at idx[off + ((j >> 3) * 32 + lane) * 8 + (j & 7)]
    uint16_t* mine = idx + off + lane * kSellGroup;

    uint32_t lane_used[kSellMaskWords];                               // positions taken in this lane (>= lpad: never free)
#pragma unroll
    for (int w = 0; w < kSellMaskWords; ++w) {
        const int lo = w * 32;
        lane_used[w] = lpad >= lo + 32 ? 0u : (lpad <= lo ? 0xffffffffu : ~((1u << (lpad - lo)) - 1u));
        bank_used[lane * kSellMaskWords + w] = 0u;
    }
    __syncwarp();

    // the lane's next CSR entry is requested one step ahead of its use
    int i = 0, loc = -1;
    int col_next = len > 0 ? __ldg(colidx + src) : 0;
    while (true) {
        while (loc < 0 && i < len) {                                  // take the next entry (skip a stored self loop)
            const int col = col_next;
            ++i;
            if (i < len) col_next = __ldg(colidx + src + i);
            if (col != row) loc = col - col0;
        }
        const bool pending = loc >= 0;
        if (!__any_sync(0xffffffffu, pending)) break;
        const int b = loc & 31;
        const unsigned grp = __match_any_sync(0xffffffffu, pending ? b : 32 + lane);
        if (pending && (__ffs(grp) - 1) == lane) {                    // one lane per bank and round
            uint32_t* bu = bank_used + b * kSellMaskWords;
            int p = -1;
#pragma unroll
            for (int w = 0; w < kSellMaskWords; ++w) {
                const uint32_t m = ~(lane_used[w] | bu[w]);
                if (p < 0 && m) p = w * 32 + __ffs(m) - 1;
            }
            const bool clean = p >= 0;
            if (!clean) {                                             // no common free position: lowest free in the lane
#pragma unroll
                for (int w = 0; w < kSellMaskWords; ++w) {
                    const uint32_t m = ~lane_used[w];
                    if (p < 0 && m) p = w * 32 + __ffs(m) - 1;
                }
            }
            const int wp = p >> 5;
            const uint32_t bit = 1u << (p & 31);
#pragma unroll
            for (int w = 0; w < kSellMaskWords; ++w) lane_used[w] |= (w == wp) ? bit : 0u;   // stays in registers
            if (clean) bu[wp] |= bit;
            mine[(p >> 3) * (kSellGroup * kSellSliceRows) + (p & 7)] = (uint16_t)loc;
            loc = -1;
        }
        __syncwarp();
    }
    // unused positions -> zero slot of bank (lane + p) mod 32
#pragma unroll
    for (int w = 0; w < kSellMaskWords; ++w) {
        uint32_t m = ~lane_used[w];
        while (m) {
            const int bit = __ffs(m) - 1;
            m &= m - 1;
            const int p = w * 32 + bit;
            mine[(p >> 3) * (kSellGroup * kSellSliceRows) + (p & 7)] = (uint16_t)(CB + ((lane + p) & 31));
        }
    }
}

// ---- gather primitives of the hot kernel (sell_step.cuh) -----------------------
// The partial sum of virtual row v goes to vpart[vslot[v]] (row-major: a row's
// partials are contiguous for the epilogue).  Shared memory: (CB + 32) floats.
__device__ __forceinline__ uint4 ld_stream_u32x4(const uint4* p) {
    uint4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}

__device__ __forceinline__ float sell_gather8(const float* ysm, const uint4 q) {
    const float a0 = ysm[q.x & 0xffffu], a1 = ysm[q.x >> 16];
    const float a2 = ysm[q.y & 0xffffu], a3 = ysm[q.y >> 16];
    const float a4 = ysm[q.z & 0xffffu], a5 = ysm[q.z >> 16];
    const float a6 = ysm[q.w & 0xffffu], a7 = ysm[q.w >> 16];
    return ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

constexpr int kSellZeroSlots = 32;
constexpr int kSellUnroll = 8;            // 16-byte index loads in flight per lane (measured best of 2/4/6/8)

}  // namespace egnn

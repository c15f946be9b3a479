// Wide-signal Chebyshev order kernel (F >= 8): CSR SpMM over the implicit
// scaled Laplacian with the three-term recurrence, the scale accumulation and
// the row L1 normalisation fused (reference: calibration/WATS.py:29-37, :55,
// :65-68, :71-72).  What bounds it is the latency and L2 bandwidth of the row
// gathers of T_{k-1}, so:
//
//  * the gather source is y = dinv (.) T_{k-1} in slabs whose row stride ldy is
//    a multiple of 4 floats (16-byte rows), written by the previous order's
//    epilogue: an entry costs one index and one 16-byte gather per lane, no
//    dinv lookup; own-row T_{k-1}, T_{k-2} are recovered as y / dinv_i;
//  * a warp owns one row x one feature tile (<= 128 columns: 32 lanes x float4,
//    or NZ entries side by side when the tile is narrower); the row's indices
//    are fetched 32 at a time with one coalesced load and broadcast by shuffle,
//    4 row gathers are in flight per lane (32 warps per SM), full groups run branch-free, and the
//    NEXT row's pointers, first index batch and own-row operand are requested
//    while this row is summed;
//  * rows are dealt out cyclically from the degree-descending order
//    (egnn_row_order) to a persistent grid, longest first; rows of at least
//    kHubDegree entries are summed by a whole CTA (fixed-order shared-memory
//    reduction: deterministic);
//  * gathers carry an L2 evict_last policy, streamed own-row operands and
//    results evict_first.
// A variant that staged the gathered rows in a shared-memory ring with cp.async
// (no register staging, chunks pipelined across rows) measured slower on every
// shape but Physics (12 warps/SM, two chunks in flight) and was dropped; see
// DESIGN.md section 7.
#pragma once

#include "cheb.cuh"
#include "common.cuh"
#include "peer.cuh"

namespace egnn {

constexpr int kWideBlock = 256;
constexpr int kWideWarps = kWideBlock / 32;
// Measured on arxiv F=128 / Reddit F=64 / Physics F=8415 (ms per order): unroll 8 x 3 CTAs/SM
// 0.35 / 2.81 / 3.15; 4 x 4: 0.285 / 2.14 / 2.73; 6 x 3: 0.29 / 2.50 / 2.75; 8 x 2: 0.30 / 2.27 /
// 3.26; 4 x 5 and 2 x 6..8 (spilling): worse on arxiv.  More resident warps beat deeper unrolling.
#ifndef EGNN_WIDE_UNROLL
#define EGNN_WIDE_UNROLL 4
#endif
#ifndef EGNN_WIDE_BLOCKS
#define EGNN_WIDE_BLOCKS 4
#endif
constexpr int kWideUnroll = EGNN_WIDE_UNROLL;      // row gathers in flight per lane
constexpr int kWideMinBlocks = EGNN_WIDE_BLOCKS;   // CTAs per SM the register budget is sized for
constexpr int kHubDegree = 2048;         // rows at least this long are summed by a whole CTA

struct WideParams {
    const int32_t* rowptr;
    const int32_t* colidx;
    const float* vals;          // NULL: binary adjacency
    const int32_t* perm;        // processing order (degree-descending) or NULL: identity
    const int32_t* n_hub;       // device scalar: leading rows of perm summed by a whole CTA (NULL: none)
    unsigned* row_counter;      // [gridDim.y] zeroed: rows of phase B are handed out dynamically, longest first
                                // (NULL: dealt out cyclically - the sharded entry, which has no workspace)
    const float* dinv;          // [n_global]
    const uint8_t* iso;         // [n_global]
    const float* ysrc;          // dinv (.) T_{k-1}, [n_global, ldy], indexed by GLOBAL column
    const float* x0_own;        // order 1: exact T_0 rows of this launch [n_rows, F]; NULL later
    const float* y2_own;        // dinv (.) T_{k-2} rows of this launch [n_rows, ldy] (may alias y_out)
    float* y_out;               // dinv (.) T_k rows [n_rows, ldy], or NULL
    float* tk_out;              // T_k rows [n_rows, F] (all orders requested), or NULL
    float* out;                 // [n_rows, S, F]
    int64_t n_rows;
    int64_t row0;
    int32_t F, ldy, S;
    float a, b;                 // operator = a * L_sym + b * I
    int32_t first, normalize;
    float c_prev[EGNN_MAX_SCALES];
    float c_k[EGNN_MAX_SCALES];
    DeltaList delta;
    PeerPush peer;              // world > 1: y_out rows also go to every rank's exchange window
    // adjoint instantiation (ADJ): b_k = c_adj * (M^T b_{k+1}) - b_{k+2} + v_k with
    // v_k = tbar + sum_s c_k[s] * cbar[:, s, :]; ysrc = dinv (.) b_{k+1}, y2_own = dinv (.) b_{k+2}
    // (NULL: zero), y_out = dinv (.) b_k, tk_out = b_k (the last application: the signal's gradient).
    // ADJ with PEER (row-sharded): dinv (.) b_k goes to every rank's window as the forward's T_k does.
    const float* cbar;          // [n_rows, S, F]
    const float* tbar;          // [n_rows, F] or NULL
    float c_adj;
};

__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t p;
    asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
// PEER: the operand lives in this rank's exchange window and other GPUs write it while this
// kernel is resident (before its flag wait), so the non-coherent path (.nc: read-only for the
// kernel's lifetime) is not allowed; plain loads, ordered after the wait's fence.sys, are.
template <bool PEER>
__device__ __forceinline__ float4 ld_gather_f4(const float* p, uint64_t pol) {
    float4 v;
    if (PEER)
        asm volatile("ld.global.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                     : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(pol) : "memory");
    else
        asm volatile("ld.global.nc.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                     : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(pol));
    return v;
}
template <bool PEER>
__device__ __forceinline__ float4 ld_operand_f4(const float* p) {
    if (!PEER) return __ldg(reinterpret_cast<const float4*>(p));
    float4 v;
    asm volatile("ld.global.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float4 ld_stream_f4(const float* p, uint64_t pol) {
    float4 v;
    asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ void st_stream_f4(float* p, float4 v, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;"
                 ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(pol) : "memory");
}

// user-visible arrays have row stride F: 16-byte accesses when F % 4 == 0, else per-column
template <bool ALIGNED>
__device__ __forceinline__ void load_user4(const float* base, int64_t off, int ncol, uint64_t pol, float (&v)[4]) {
    if (ALIGNED) {
        const float4 t = ld_stream_f4(base + off, pol);
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = j < ncol ? base[off + j] : 0.f;
    }
}
template <bool ALIGNED>
__device__ __forceinline__ void store_user4(float* base, int64_t off, int ncol, uint64_t pol, const float (&v)[4]) {
    if (ALIGNED) {
        st_stream_f4(base + off, make_float4(v[0], v[1], v[2], v[3]), pol);
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (j < ncol) base[off + j] = v[j];
    }
}

// Fused epilogue of one row tile; `writer` lanes (entry slot 0, column inside
// the padded row) hold the row's sum in acc.  ncol = valid user columns of the lane.
template <bool ALIGNED, bool PEER, bool ADJ>
__device__ __forceinline__ void wide_epilogue(const WideParams& p, int row, int grow, int FL, int fcol, int ncol,
                                              bool writer, float (&acc)[4], uint64_t pol_stream, bool have_own,
                                              const float (&own)[4]) {
    const int F = p.F, ldy = p.ldy;
    float di = 1.f, theta = 0.f;
    if (writer) {
        di = __ldg(p.dinv + grow);
        theta = fmaf(p.a, 1.f - (float)__ldg(p.iso + grow), p.b);
    }
    if (p.delta.n > 0 && writer) {          // edge flips on top of the CSR (UGCA recompute)
        for (int e = 0; e < p.delta.n; ++e) {
            if (p.delta.row[e] == grow && p.delta.col[e] != grow) {
                const float4 x = ld_operand_f4<PEER>(p.ysrc + (int64_t)p.delta.col[e] * ldy + fcol);
                const float w = p.delta.val[e];
                acc[0] = fmaf(w, x.x, acc[0]); acc[1] = fmaf(w, x.y, acc[1]);
                acc[2] = fmaf(w, x.z, acc[2]); acc[3] = fmaf(w, x.w, acc[3]);
            }
        }
    }
    const float nscale = -p.a * di;
    const float inv_di = 1.f / di;
    if constexpr (ADJ) {                    // adjoint epilogue (Clenshaw step): no scale accumulation
        if (!writer) return;
        const int64_t uoff = (int64_t)row * F + fcol;
        const int64_t yoff = (int64_t)row * ldy + fcol;
        float bown[4] = {0.f, 0.f, 0.f, 0.f}, b2[4] = {0.f, 0.f, 0.f, 0.f}, v[4] = {0.f, 0.f, 0.f, 0.f};
        if (theta != 0.f) {                                     // b_{k+1} of the own row = y / dinv
            const float4 t = ld_operand_f4<PEER>(p.ysrc + (int64_t)grow * ldy + fcol);
            bown[0] = t.x * inv_di; bown[1] = t.y * inv_di; bown[2] = t.z * inv_di; bown[3] = t.w * inv_di;
        }
        if (have_own) {
#pragma unroll
            for (int j = 0; j < 4; ++j) b2[j] = own[j] * inv_di;
        } else if (p.y2_own) {
            const float4 t = ld_stream_f4(p.y2_own + yoff, pol_stream);
            b2[0] = t.x * inv_di; b2[1] = t.y * inv_di; b2[2] = t.z * inv_di; b2[3] = t.w * inv_di;
        }
        if (p.tbar) load_user4<ALIGNED>(p.tbar, uoff, ncol, pol_stream, v);
        for (int s = 0; s < p.S; ++s) {
            float t[4];
            load_user4<ALIGNED>(p.cbar, ((int64_t)row * p.S + s) * F + fcol, ncol, pol_stream, t);
#pragma unroll
            for (int j = 0; j < 4; ++j) v[j] = fmaf(p.c_k[s], t[j], v[j]);
        }
        float b[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            b[j] = fmaf(p.c_adj, fmaf(theta, bown[j], nscale * acc[j]), v[j] - b2[j]);
            if (j >= ncol) b[j] = 0.f;                          // padding columns stay zero
        }
        if (p.tk_out) store_user4<ALIGNED>(p.tk_out, uoff, ncol, pol_stream, b);
        if (p.y_out) *reinterpret_cast<float4*>(p.y_out + yoff) = make_float4(di * b[0], di * b[1], di * b[2], di * b[3]);
        if constexpr (PEER) {                                   // row-sharded: dinv (.) b_k into every rank's window
            if (p.peer.has_data) {
                const float4 yv = make_float4(di * b[0], di * b[1], di * b[2], di * b[3]);
                const int64_t goff = (int64_t)grow * ldy + fcol;
                for (int r = 0; r < p.peer.world; ++r) *reinterpret_cast<float4*>(p.peer.dst[r] + goff) = yv;
            }
        }
        return;
    }
    float tk[4] = {0.f, 0.f, 0.f, 0.f}, xprev[4] = {0.f, 0.f, 0.f, 0.f};
    if (writer) {
        const int64_t uoff = (int64_t)row * F + fcol;          // user arrays
        const int64_t yoff = (int64_t)row * ldy + fcol;        // padded slabs
        if (p.first) {
            if (have_own) {
#pragma unroll
                for (int v = 0; v < 4; ++v) xprev[v] = own[v];
            } else {
                load_user4<ALIGNED>(p.x0_own, uoff, ncol, pol_stream, xprev);
            }
        } else if (theta != 0.f) {                              // T_{k-1} of the own row = y / dinv
            const float4 t = ld_operand_f4<PEER>(p.ysrc + (int64_t)grow * ldy + fcol);
            xprev[0] = t.x * inv_di; xprev[1] = t.y * inv_di; xprev[2] = t.z * inv_di; xprev[3] = t.w * inv_di;
        }
        float t2[4] = {0.f, 0.f, 0.f, 0.f};
        if (!p.first) {
            if (have_own) {
#pragma unroll
                for (int v = 0; v < 4; ++v) t2[v] = own[v] * inv_di;
            } else {
                const float4 t = ld_stream_f4(p.y2_own + yoff, pol_stream);
                t2[0] = t.x * inv_di; t2[1] = t.y * inv_di; t2[2] = t.z * inv_di; t2[3] = t.w * inv_di;
            }
        }
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            const float lap = fmaf(theta, xprev[v], nscale * acc[v]);
            tk[v] = p.first ? lap : fmaf(2.f, lap, -t2[v]);
            if (v >= ncol) tk[v] = 0.f;                         // padding columns stay zero
        }
        if (p.tk_out) store_user4<ALIGNED>(p.tk_out, uoff, ncol, pol_stream, tk);
        const float4 yv = make_float4(di * tk[0], di * tk[1], di * tk[2], di * tk[3]);
        if (p.y_out) *reinterpret_cast<float4*>(p.y_out + yoff) = yv;
        if (p.peer.world > 1 && p.peer.has_data) {
            const int64_t goff = (int64_t)grow * ldy + fcol;
            for (int r = 0; r < p.peer.world; ++r) *reinterpret_cast<float4*>(p.peer.dst[r] + goff) = yv;
        }
    }
    for (int s = 0; s < p.S; ++s) {
        float o[4] = {0.f, 0.f, 0.f, 0.f};
        float l1 = 0.f;
        const int64_t ooff = ((int64_t)row * p.S + s) * F + fcol;
        if (writer) {
            if (p.first) {
#pragma unroll
                for (int v = 0; v < 4; ++v) o[v] = fmaf(p.c_k[s], tk[v], p.c_prev[s] * xprev[v]);
            } else {
                float t[4];
                load_user4<ALIGNED>(p.out, ooff, ncol, pol_stream, t);
#pragma unroll
                for (int v = 0; v < 4; ++v) o[v] = fmaf(p.c_k[s], tk[v], t[v]);
            }
#pragma unroll
            for (int v = 0; v < 4; ++v) l1 += v < ncol ? fabsf(o[v]) : 0.f;
        }
        if (p.normalize) {       // uniform branch: every lane takes part in the shuffles
            for (int off = 1; off < FL; off <<= 1) l1 += __shfl_xor_sync(0xffffffffu, l1, off);
            const float inv = 1.f / (l1 + 1e-8f);
#pragma unroll
            for (int v = 0; v < 4; ++v) o[v] *= inv;
        }
        if (writer) store_user4<ALIGNED>(p.out, ooff, ncol, pol_stream, o);
    }
}

// Sum of w_e * y[c_e, tile] over entries q in [qs, qe) taken by this lane's
// entry slot (nzl of NZ), starting from the first index batch already held in
// (pre_c, pre_w) when have_pre.  Full groups of UNR entries per slot run
// branch-free; only the tail is guarded.  Two-level float32 summation: acc is
// folded into hi every 64 entries of a chain.
template <int NZ_LOG2, bool HAS_VALS, bool PEER>
__device__ __forceinline__ void wide_accumulate(const WideParams& p, int qs, int qe, int grow, int lane, int nzl,
                                                const float* ycol, bool have_pre, int pre_c, float pre_w,
                                                uint64_t pol_keep, float (&sum)[4]) {
    constexpr int NZ = 1 << NZ_LOG2;
    constexpr int UNR = NZ <= 4 ? kWideUnroll : 32 / NZ;      // entries in flight per slot; NZ * UNR <= 32
    constexpr int STEP = NZ * UNR;
    const int64_t ldy = p.ldy;
    float acc[4] = {0.f, 0.f, 0.f, 0.f}, hi[4] = {0.f, 0.f, 0.f, 0.f};
    int since_fold = 0;
    for (int b0 = qs; b0 < qe; b0 += 32) {
        const int cnt = min(32, qe - b0);
        int cj = grow;
        float wj = 0.f;
        if (have_pre && b0 == qs) {
            cj = pre_c;
            wj = pre_w;
        } else if (lane < cnt) {
            cj = ld_stream_i32(p.colidx + b0 + lane);
            wj = HAS_VALS ? ld_stream_f32(p.vals + b0 + lane) : 1.f;
        }
        if (lane >= cnt) { cj = grow; wj = 0.f; }
        if (cj == grow) wj = 0.f;                      // stored self loops are not part of L
        int e0 = 0;
        for (; e0 + STEP <= cnt; e0 += STEP) {         // full groups: no guards
            float4 x[UNR];
#pragma unroll
            for (int j = 0; j < UNR; ++j) {
                const int c = __shfl_sync(0xffffffffu, cj, e0 + j * NZ + nzl);
                x[j] = ld_gather_f4<PEER>(ycol + c * ldy, pol_keep);
            }
#pragma unroll
            for (int j = 0; j < UNR; ++j) {
                const float w = __shfl_sync(0xffffffffu, wj, e0 + j * NZ + nzl);
                acc[0] = fmaf(w, x[j].x, acc[0]); acc[1] = fmaf(w, x[j].y, acc[1]);
                acc[2] = fmaf(w, x[j].z, acc[2]); acc[3] = fmaf(w, x[j].w, acc[3]);
            }
        }
        if (e0 < cnt) {                                // tail group (lanes past cnt hold c = own row, w = 0)
            float4 x[UNR];
#pragma unroll
            for (int j = 0; j < UNR; ++j) {
                if (e0 + j * NZ < cnt) {               // warp-uniform
                    const int c = __shfl_sync(0xffffffffu, cj, (e0 + j * NZ + nzl) & 31);
                    x[j] = ld_gather_f4<PEER>(ycol + c * ldy, pol_keep);
                }
            }
#pragma unroll
            for (int j = 0; j < UNR; ++j) {
                if (e0 + j * NZ < cnt) {
                    const float w = __shfl_sync(0xffffffffu, wj, (e0 + j * NZ + nzl) & 31);
                    acc[0] = fmaf(w, x[j].x, acc[0]); acc[1] = fmaf(w, x[j].y, acc[1]);
                    acc[2] = fmaf(w, x[j].z, acc[2]); acc[3] = fmaf(w, x[j].w, acc[3]);
                }
            }
        }
        since_fold += 32;
        if (since_fold >= 64 * NZ) {                   // 64 entries per chain
#pragma unroll
            for (int v = 0; v < 4; ++v) { hi[v] += acc[v]; acc[v] = 0.f; }
            since_fold = 0;
        }
    }
#pragma unroll
    for (int v = 0; v < 4; ++v) sum[v] = hi[v] + acc[v];
}

template <int NZ_LOG2, bool HAS_VALS, bool ALIGNED, bool PEER, bool DYN, bool ADJ = false>
__global__ void __launch_bounds__(kWideBlock, kWideMinBlocks)
cheb_wide_kernel(const __grid_constant__ WideParams p) {
    __shared__ float hub_part[kWideWarps][128];
    constexpr int FL_LOG2 = 5 - NZ_LOG2;
    constexpr int FL = 1 << FL_LOG2;
    const int lane = threadIdx.x & 31;
    const int wid = threadIdx.x >> 5;
    const int fl = lane & (FL - 1);
    const int nzl = lane >> FL_LOG2;
    // the lane's 4 columns; lanes past the padded row width re-read the last column group and never store
    int fcol = blockIdx.y * (FL * 4) + fl * 4;
    const bool col_ok = fcol < p.ldy;
    if (!col_ok) fcol = p.ldy - 4;
    const int ncol = col_ok ? min(4, p.F - fcol) : 0;
    const float* ycol = p.ysrc + fcol;
    const uint64_t pol_keep = l2_policy_evict_last();
    const uint64_t pol_stream = l2_policy_evict_first();
    const int n_rows = (int)p.n_rows;
    int n_hub = p.n_hub ? __ldg(p.n_hub) : 0;
    if (n_hub > n_rows) n_hub = n_rows;
    const bool writer = nzl == 0 && col_ok;
    const float none[4] = {0.f, 0.f, 0.f, 0.f};
    // row-sharded: the operand sits in this rank's exchange window and the other GPUs fill it
    if (PEER) peer_consumer_wait(p.peer.local_flags, p.peer.epoch, p.peer.world, p.peer.rank, p.peer.error);

    // ---- phase A: hub rows, one CTA each, longest first ---------------------
    for (int h = blockIdx.x; h < n_hub; h += gridDim.x) {
        const int row = p.perm ? __ldg(p.perm + h) : h;
        const int grow = (int)p.row0 + row;
        const int start = __ldg(p.rowptr + row), end = __ldg(p.rowptr + row + 1);
        // warp w sums a contiguous run of whole 32-entry batches
        const int n_batches = (end - start + 31) >> 5;
        const int per_warp = (n_batches + kWideWarps - 1) / kWideWarps;
        const int qs = min(end, start + wid * per_warp * 32);
        const int qe = min(end, qs + per_warp * 32);
        float part[4];
        wide_accumulate<NZ_LOG2, HAS_VALS, PEER>(p, qs, qe, grow, lane, nzl, ycol, false, 0, 0.f, pol_keep, part);
#pragma unroll
        for (int o = FL; o < 32; o <<= 1) {
#pragma unroll
            for (int v = 0; v < 4; ++v) part[v] += __shfl_xor_sync(0xffffffffu, part[v], o);
        }
        __syncthreads();                                       // previous hub row's readers are done
        if (nzl == 0) {
#pragma unroll
            for (int v = 0; v < 4; ++v) hub_part[wid][fl * 4 + v] = part[v];
        }
        __syncthreads();
        if (wid == 0) {
            float acc[4];
#pragma unroll
            for (int v = 0; v < 4; ++v) {
                float t = 0.f;
                for (int w = 0; w < kWideWarps; ++w) t += hub_part[w][fl * 4 + v];     // fixed order
                acc[v] = t;
            }
            wide_epilogue<ALIGNED, PEER, ADJ>(p, row, grow, FL, fcol, ncol, writer, acc, pol_stream, false, none);
        }
    }

    // ---- phase B: one row per warp ---------------------------------------------------
    // Rows are taken longest first.  DYN: handed out from a counter (greedy longest-processing-
    // time schedule), which matters on short-row graphs: dealt out cyclically, warp 0 gets the
    // longest row of every round - on the arxiv shape (15 entries per row on average, 660 at
    // most, 36 rounds) the first warps carry twice the work of the last (ncu: slowest SM active
    // 516 k cycles, average 364 k).  The row after next is requested while this one is summed,
    // so the atomic's latency and the next row's pointer loads stay off the critical path.
    // A separate instantiation: the bookkeeping costs the long-row shapes 15-20 % when compiled in.
    const int total_warps = gridDim.x * kWideWarps;
    unsigned* counter = DYN ? p.row_counter + blockIdx.y : nullptr;
    int r = n_hub + blockIdx.x * kWideWarps + wid;             // the first two rows of a warp are fixed
    int r_next = r + total_warps;
    unsigned raw_nn = 0;                                       // row after next: lane 0's pending request
    if (DYN && lane == 0) raw_nn = atomicAdd(counter, 1u);
    int row = 0, start = 0, end = 0, pre_c = 0;
    float pre_w = 0.f;
    float own[4] = {0.f, 0.f, 0.f, 0.f};
    // the own-row operand of the epilogue (T_0 row at order 1, dinv (.) T_{k-2} later; adjoint:
    // dinv (.) b_{k+2} when there is one) is requested a row ahead
    auto load_own = [&](int rw, float (&dst)[4]) {
        if (!writer) return;
        if (ADJ && !p.y2_own) return;
        if (!ADJ && p.first) {
            if (ALIGNED) load_user4<true>(p.x0_own, (int64_t)rw * p.F + fcol, ncol, pol_stream, dst);
        } else {
            const float4 t = ld_stream_f4(p.y2_own + (int64_t)rw * p.ldy + fcol, pol_stream);
            dst[0] = t.x; dst[1] = t.y; dst[2] = t.z; dst[3] = t.w;
        }
    };
    const bool have_own = ADJ ? p.y2_own != nullptr : (!p.first || ALIGNED);
    if (r < n_rows) {
        row = p.perm ? __ldg(p.perm + r) : r;
        start = __ldg(p.rowptr + row);
        end = __ldg(p.rowptr + row + 1);
        if (start + lane < end) {
            pre_c = ld_stream_i32(p.colidx + start + lane);
            pre_w = HAS_VALS ? ld_stream_f32(p.vals + start + lane) : 1.f;
        }
        load_own(row, own);
    }
    while (r < n_rows) {
        // the row after next: static stride without a counter, else what the counter handed out
        // one row ago (a new request goes out now)
        int r_nn = r_next + total_warps;
        if (DYN) {
            r_nn = n_hub + 2 * total_warps + (int)__shfl_sync(0xffffffffu, raw_nn, 0);
            if (lane == 0) raw_nn = atomicAdd(counter, 1u);
        }
        int row_n = 0, start_n = 0, end_n = 0;
        if (r_next < n_rows) {
            row_n = p.perm ? __ldg(p.perm + r_next) : r_next;
            start_n = __ldg(p.rowptr + row_n);
            end_n = __ldg(p.rowptr + row_n + 1);
        }
        const int grow = (int)p.row0 + row;
        float acc[4];
        wide_accumulate<NZ_LOG2, HAS_VALS, PEER>(p, start, end, grow, lane, nzl, ycol, true, pre_c, pre_w, pol_keep, acc);
        int pre_c_n = 0;
        float pre_w_n = 0.f;
        float own_n[4] = {0.f, 0.f, 0.f, 0.f};
        if (r_next < n_rows) {
            if (start_n + lane < end_n) {
                pre_c_n = ld_stream_i32(p.colidx + start_n + lane);
                pre_w_n = HAS_VALS ? ld_stream_f32(p.vals + start_n + lane) : 1.f;
            }
            load_own(row_n, own_n);
        }
#pragma unroll
        for (int o = FL; o < 32; o <<= 1) {
#pragma unroll
            for (int v = 0; v < 4; ++v) acc[v] += __shfl_xor_sync(0xffffffffu, acc[v], o);
        }
        wide_epilogue<ALIGNED, PEER, ADJ>(p, row, grow, FL, fcol, ncol, writer, acc, pol_stream, have_own, own);
        r = r_next; r_next = r_nn; row = row_n; start = start_n; end = end_n; pre_c = pre_c_n; pre_w = pre_w_n;
#pragma unroll
        for (int v = 0; v < 4; ++v) own[v] = own_n[v];
    }
    if (PEER) peer_producer_signal(p.peer);
}

// ---- pre-scaled copy of the input signal into a padded slab ---------------------
// y[r, c] = dinv[row0 + r] * x[r, c] for c < F, 0 for F <= c < ldy
__global__ void __launch_bounds__(256)
prescale_pad_kernel(const float* __restrict__ x, const float* __restrict__ dinv, float* __restrict__ y,
                    int64_t n, int32_t F, int32_t ldy, int64_t row0) {
    const int64_t total = n * ldy;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / ldy;
        const int c = (int)(i - r * ldy);
        y[i] = c < F ? dinv[row0 + r] * x[r * F + c] : 0.f;
    }
}

// ---- processing order ---------------------------------------------------------
// key = ~degree so an ascending radix sort yields the longest rows first
__global__ void __launch_bounds__(256)
row_order_keys_kernel(const int32_t* __restrict__ rowptr, int n, uint32_t* __restrict__ keys,
                      int32_t* __restrict__ ids) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    keys[i] = ~(uint32_t)(rowptr[i + 1] - rowptr[i]);
    ids[i] = i;
}

__global__ void row_order_hubs_kernel(const uint32_t* __restrict__ keys_sorted, int n, int32_t* __restrict__ n_hub) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    int lo = 0, hi = n;                          // first position whose degree < kHubDegree
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if ((int)(~keys_sorted[mid]) >= kHubDegree) lo = mid + 1; else hi = mid;
    }
    *n_hub = lo;
}

}  // namespace egnn

// The narrow (F = 1) Chebyshev step as ONE persistent cooperative kernel:
// all orders k = order_begin .. order_end of
//     T_k = m_k L~ T_{k-1} - T_{k-2},   S_s += c_k(s) T_k
// (calibration/WATS.py:29-37, :55, :65-68, :71-72) over the SELL plan of
// sell.cuh, one CTA per SM, with grid barriers instead of kernel boundaries.
//
// Per order, every CTA
//   1. stages its column block of the operand y = dinv (.) T_{k-1} in shared
//      memory with 1-D TMA bulk copies (cp.async.bulk + mbarrier: no registers
//      or issue slots held while the 190 KB land) - row-sharded: after the
//      flags of the ranks that OWN those columns have arrived;
//   2. sums slices of that block: warps pull slices (longest first) from a
//      per-block counter in global memory, so the ~30 CTAs that serve one
//      column block balance dynamically (ncu on the static split: slowest SM
//      99 k cycles vs 85 k average); each lane streams its virtual row with
//      16-byte index loads, 8 in flight, and gathers from shared memory;
//   3. grid barrier; then runs the fused epilogue for its own rows: partial
//      sums added in float64 in a fixed order (rows with many virtual rows by a
//      whole warp), Laplacian scaling, recurrence, all S scales, L1
//      normalisation on the last order, and the next operand dinv (.) T_k -
//      row-sharded: stored straight into every rank's exchange window;
//   4. grid barrier (row-sharded: one CTA then raises this rank's flag in
//      every window; before a phase stores into the windows it has seen
//      every rank's latest flag, so no buffer is overwritten while a slower
//      rank still stages it).
// Results do not depend on which CTA or warp summed which slice: bitwise
// deterministic.
// Instantiations: PEER (exchange windows of a row-sharded graph) and PATCH
// (UGCA recompute: the vectors passed are the base graph's, the nodes the
// edge flips touch are re-derived in the kernel - one launch per perturbed
// pass); the plain <false, false> one is the benchmarked default.
#pragma once

#include "common.cuh"
#include "peer.cuh"
#include "prep.cuh"
#include "sell.cuh"

namespace egnn {

constexpr int kStepMaxOrders = 16;        // orders per launch (the coefficient window travels as kernel parameters)
constexpr int kSchedBarrier = kSellMaxBlocks * kSellCtrStride;   // sched[c * 32]: next slice of column block c; then the 64-bit barrier counter
constexpr int kEpiWarpRow = kSellEpiWarpRow;           // rows with more partial sums than this are added up by a whole warp
constexpr int kStageChunkFloats = 8192;   // one bulk copy = 32 KB
// partial sums of each of a thread's two epilogue rows requested in the first round trip: a row
// has about one per column block it touches (five blocks on the Reddit shape); 6 or 8 spill at
// 64 registers
constexpr int kEpiFirstParts = 5;

struct SellStepParams {
    // plan
    const uint16_t* idx;
    const int32_t* slice_off;
    const int32_t* blk_slice_ptr;
    const int32_t* vslot;
    const int32_t* cta_info;      // [n_cta] column block (-1: none), [n_cta] rank inside the block, [64] counter start, [n_cta + 1] epilogue rows
    const int32_t* hub;           // [n_cta + 1] + rows: the hub rows of every CTA's epilogue range (sell_cta_hubs_kernel)
    const int32_t* rv_ptr;
    float* vpart;
    unsigned* sched;
    unsigned long long* stamps;   // optional: globaltimer at kernel start and after every grid barrier (CTA 0)
    int32_t trace;                // with stamps: every CTA also records stage-done / barrier-arrival times
    int32_t n_cta, C, CB, n_cols, n_rows, row0;
    // graph vectors and signal
    const float* dinv;            // [n_cols]
    const uint8_t* iso;           // [n_cols]
    const float* x0;              // [n_rows] T_0 of the own rows
    const float* operand_first;   // optional: the operand of order_begin, whole vector, held by the caller
    const float* operand[2];      // operand of order k: operand[(k-1) & 1], indexed by global column
    float* ydst[2][EGNN_MAX_RANKS];   // dinv (.) T_k goes to ydst[k & 1][d][row0 + i], d < n_dst
    int32_t n_dst;
    float* tbuf[2];               // T_k (k >= 1) lives in tbuf[(k-1) & 1] unless t_all is given
    float* t_all;                 // [K+1, n_rows] or NULL
    float* out;                   // [n_rows, S]
    int32_t order_begin, order_end, k_max, S, normalize;
    float a, b;
    float coef[EGNN_MAX_SCALES][kStepMaxOrders + 1];   // coef[s][j] = c_{order_begin-1+j}(s)
    DeltaList delta;
    // PATCH instantiation (UGCA recompute in one launch): dinv / iso / x0 / operand_first are the
    // BASE graph's; the kernel re-derives the entries of the nodes the flips touch from these
    const float* w_base;          // [n_cols] in-degree without self loops
    const float* rowsum_base;     // [n_cols] row sums
    int32_t patch_x0;             // 1: T_0 is the default signal log1p(row sum) and changes with the flips; 0: caller's signal, kept
    // exchange window of this rank (PEER instantiation)
    int32_t world, rank;
    int64_t rows_per;
    unsigned* flag_at[EGNN_MAX_RANKS];    // &flags[rank] in every rank's window
    unsigned* local_flags;
    unsigned* epoch;
    unsigned* error;
};

// ---- small PTX wrappers -------------------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t}"
        ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// 1-D TMA: global -> shared, completion counted in bytes on the mbarrier
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async;" ::: "memory"); }

// Grid barrier of the cooperative launch, split in two halves so that work which does not
// depend on the other CTAs runs between them.  One 64-bit counter that only grows: barrier
// number j of a launch is complete when it reaches base + (j + 1) * n_cta, where base is the
// counter at kernel start rounded down to a multiple of n_cta (no CTA can be more than one
// barrier ahead of the slowest, so every CTA computes the same base).  Thread 0 only.
__device__ __forceinline__ unsigned long long ld_relaxed_gpu_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void grid_arrive(unsigned long long* ctr, bool sys_scope) {
    if (sys_scope) __threadfence_system(); else __threadfence();     // this CTA's stores first
    atomicAdd(ctr, 1ull);
}
__device__ __forceinline__ void grid_wait(const unsigned long long* ctr, unsigned long long target) {
    while ((long long)(ld_relaxed_gpu_u64(ctr) - target) < 0) { }
    __threadfence();                      // acquire; also drops this SM's L1 lines of data other SMs rewrote
}

// Warp 0, every lane: wait until ranks p_lo..p_hi (except this one) have signalled `epoch`
// here - one rank per lane, so the polls of several owners overlap.
__device__ __forceinline__ void peer_wait_ranks(const unsigned* local_flags, int p_lo, int p_hi, int rank,
                                                unsigned epoch, unsigned* error, bool stats, int lane) {
    const unsigned long long t0 = global_timer_ns();
    for (int p = p_lo + lane; p <= p_hi; p += 32) {
        if (p == rank) continue;
        while ((int)(ld_relaxed_sys_u32(local_flags + p) - epoch) < 0) {
            __nanosleep(32);
            if (global_timer_ns() - t0 > kPeerTimeoutNs) {
                atomicExch(error, 1u);
                break;
            }
        }
    }
    __syncwarp();                         // every lane has seen its flag ...
    if (lane == 0) __threadfence_system();    // ... one fence (32 of them cost ~10 us per order): acquire for what follows,
    __syncwarp();                             // in every lane
    if (stats && lane == 0) {
        unsigned long long* stat = reinterpret_cast<unsigned long long*>(
            reinterpret_cast<char*>(const_cast<unsigned*>(local_flags)) - kPeerFlagsOff + kPeerWaitNsOff);
        stat[0] += global_timer_ns() - t0;
        stat[1] += 1ull;
    }
}

struct StepOrderView {            // pointers of one order, resolved once per CTA
    const float* operand;         // dinv (.) T_{k-1}, global columns
    const float* tprev;           // T_{k-1} own rows
    const float* tprev2;          // T_{k-2} own rows (k >= 2)
    float* tk;                    // or NULL
    int k, j;                     // order; index into the coefficient window
    bool first, last, push;
    bool flips_here;              // an edge flip names a row of this CTA's epilogue range
    const float* flip_term;       // shared memory: contribution of every flip (0 for the ones of other CTAs' rows)
    // PATCH: the nodes the flips touch (rows, then columns of the flips) and their re-derived vectors
    bool touched_here;            // one of them is a row of this CTA's epilogue range
    int n_touch;
    const int* pt_node;
    const float* pt_dinv;
    const float* pt_x0;
    const unsigned char* pt_iso;
};

__device__ __forceinline__ int step_patch_find(const int* node, int n, int gi) {
    for (int j = 0; j < n; ++j)
        if (node[j] == gi) return j;
    return -1;
}

__device__ __forceinline__ const float* step_t_ptr(const SellStepParams& p, int j) {
    if (j == 0) return p.x0;
    return p.t_all ? p.t_all + (size_t)j * p.n_rows : p.tbuf[(j - 1) & 1];
}

// What a row's epilogue needs besides its partial sums: requested BEFORE the wait for the
// grid barrier that guards the partial sums, so only the sums are left on the critical path.
struct StepRowPre {
    int t, e;
    float di, theta, xprev, t2, out0;
};

template <bool PATCH>
__device__ __forceinline__ void step_row_patch(const SellStepParams& p, const StepOrderView& v, int gi, StepRowPre& r) {
    if (PATCH && v.touched_here) {        // a node an edge flip touches: its degree changed (uniform per CTA; most skip this)
        const int j = step_patch_find(v.pt_node, v.n_touch, gi);
        if (j >= 0) {
            r.di = v.pt_dinv[j];
            r.theta = fmaf(p.a, 1.f - (float)v.pt_iso[j], p.b);
            if (v.k == 1) r.xprev = v.pt_x0[j];           // T_0 = x0 = log1p(row sum)
            if (v.k == 2) r.t2 = v.pt_x0[j];
        }
    }
}

template <bool PATCH>
__device__ __forceinline__ StepRowPre step_row_prefetch(const SellStepParams& p, const StepOrderView& v, int i) {
    StepRowPre r;
    const int gi = p.row0 + i;
    r.t = __ldg(p.rv_ptr + i);
    r.e = __ldg(p.rv_ptr + i + 1);
    r.di = __ldg(p.dinv + gi);
    r.theta = fmaf(p.a, 1.f - (float)__ldg(p.iso + gi), p.b);
    r.xprev = v.tprev[i];
    r.t2 = v.first ? 0.f : v.tprev2[i];
    r.out0 = v.first ? 0.f : p.out[(size_t)i * p.S];
    step_row_patch<PATCH>(p, v, gi, r);
    return r;
}

// The same words for a row a whole warp sums, spread over the lanes (lane j requests word j:
// t, e, dinv, iso, T_{k-1}, T_{k-2}, S_0) so that the request costs one register, not seven;
// step_hub_gather assembles them (every lane, after the grid barrier's wait)
__device__ __forceinline__ uint32_t step_hub_prefetch(const SellStepParams& p, const StepOrderView& v, int i, int lane) {
    const int gi = p.row0 + i;
    uint32_t w = 0u;
    if (lane == 0) w = (uint32_t)__ldg(p.rv_ptr + i);
    else if (lane == 1) w = (uint32_t)__ldg(p.rv_ptr + i + 1);
    else if (lane == 2) w = __float_as_uint(__ldg(p.dinv + gi));
    else if (lane == 3) w = __ldg(p.iso + gi);
    else if (lane == 4) w = __float_as_uint(v.tprev[i]);
    else if (lane == 5 && !v.first) w = __float_as_uint(v.tprev2[i]);
    else if (lane == 6 && !v.first) w = __float_as_uint(p.out[(size_t)i * p.S]);
    return w;
}
template <bool PATCH>
__device__ __forceinline__ StepRowPre step_hub_gather(const SellStepParams& p, const StepOrderView& v, int i, uint32_t w) {
    StepRowPre r;
    r.t = (int)__shfl_sync(0xffffffffu, w, 0);
    r.e = (int)__shfl_sync(0xffffffffu, w, 1);
    r.di = __uint_as_float(__shfl_sync(0xffffffffu, w, 2));
    r.theta = fmaf(p.a, 1.f - (float)__shfl_sync(0xffffffffu, w, 3), p.b);
    r.xprev = __uint_as_float(__shfl_sync(0xffffffffu, w, 4));
    r.t2 = __uint_as_float(__shfl_sync(0xffffffffu, w, 5));
    r.out0 = __uint_as_float(__shfl_sync(0xffffffffu, w, 6));
    step_row_patch<PATCH>(p, v, p.row0 + i, r);
    return r;
}

// Everything of the row's epilogue that follows the sum of its partials.
__device__ __forceinline__ void step_epilogue_finish(const SellStepParams& p, const StepOrderView& v, int i,
                                                     const StepRowPre& r, double accd) {
    const int gi = p.row0 + i;
    if (v.flips_here)                     // some flip touches a row of this CTA (uniform per CTA; most CTAs skip the list)
        for (int d = 0; d < p.delta.n; ++d)
            if (p.delta.row[d] == gi) accd += (double)v.flip_term[d];     // val * operand[col], fetched before the barrier wait
    const float acc = (float)accd;
    const float lap = fmaf(r.theta, r.xprev, -p.a * r.di * acc);
    const float tk = v.first ? lap : fmaf(2.f, lap, -r.t2);
    if (v.tk) v.tk[i] = tk;
    if (v.push) {
        const float yv = r.di * tk;
        for (int d = 0; d < p.n_dst; ++d) p.ydst[v.k & 1][d][gi] = yv;
    }
    for (int s = 0; s < p.S; ++s) {
        float o = v.first ? fmaf(p.coef[s][v.j + 1], tk, p.coef[s][v.j] * r.xprev)
                          : fmaf(p.coef[s][v.j + 1], tk, s == 0 ? r.out0 : p.out[(size_t)i * p.S + s]);
        if (v.last && p.normalize) o = o / (fabsf(o) + 1e-8f);
        p.out[(size_t)i * p.S + s] = o;
    }
}

// Partial sums of a row with at most kEpiWarpRow virtual rows, added in float64 in storage
// order (always the same order: deterministic).  The first N are requested by the caller (so
// that the loads of several rows are in flight together), the rest eight at a time.
template <int N>
__device__ __forceinline__ void step_row_load(const float* vpart, int t, int e, float (&x)[N]) {
#pragma unroll
    for (int u = 0; u < N; ++u) x[u] = t + u < e ? __ldcg(vpart + t + u) : 0.f;
}
template <int N>
__device__ __forceinline__ double step_row_sum_rest(const float* vpart, int t, int e, const float (&x0)[N]) {
    double a = 0.0;
#pragma unroll
    for (int u = 0; u < N; ++u) a += (double)x0[u];
    for (t += N; t < e; t += 8) {
        float x[8];
        step_row_load(vpart, t, e, x);
#pragma unroll
        for (int u = 0; u < 8; ++u) a += (double)x[u];
    }
    return a;
}
__device__ __forceinline__ double step_row_sum(const float* vpart, int t, int e) {
    float x[8];
    step_row_load(vpart, t, e, x);
    return step_row_sum_rest(vpart, t, e, x);
}

// A row with more than kEpiWarpRow partial sums, by a whole warp: lane-strided float64 sums in a
// fixed shuffle tree; x0 = the lane's first partial (vpart[r.t + lane], 0 past the end).
__device__ __forceinline__ void step_hub_finish(const SellStepParams& p, const StepOrderView& v, int i,
                                                const StepRowPre& r, float x0, int lane) {
    double a = 0.0;
    a += (double)x0;
    for (int t = r.t + lane + 32; t < r.e; t += 32) a += (double)__ldcg(p.vpart + t);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) step_epilogue_finish(p, v, i, r, a);
}
__device__ __forceinline__ float step_hub_first(const float* vpart, int t, int e, int lane) {
    return t + lane < e ? __ldcg(vpart + t + lane) : 0.f;
}

template <bool PEER, bool PATCH>
__global__ void __launch_bounds__(kSellThreads, 1)
sell_step_kernel(const __grid_constant__ SellStepParams p) {
    extern __shared__ __align__(128) float ysm[];
    __shared__ __align__(8) unsigned long long stage_bar;
    __shared__ int hub_first[kSellThreads / 32], hub_span[2];     // the first hub row of every warp (-1: none); CTA's span of the list
    __shared__ float flip_term[EGNN_MAX_DELTA];
    __shared__ int pt_node[PATCH ? 2 * EGNN_MAX_DELTA : 1];
    __shared__ float pt_dinv[PATCH ? 2 * EGNN_MAX_DELTA : 1], pt_x0[PATCH ? 2 * EGNN_MAX_DELTA : 1], pt_y0[PATCH ? 2 * EGNN_MAX_DELTA : 1];
    __shared__ unsigned char pt_iso[PATCH ? 2 * EGNN_MAX_DELTA : 1];
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int wid = tid >> 5;
    constexpr int kWarps = kSellThreads / 32;
    const int g = blockIdx.x;
    const unsigned n_cta = gridDim.x;

    const int c = __ldg(p.cta_info + g);                       // column block this CTA serves (-1: none)
    const int rank_in_block = __ldg(p.cta_info + p.n_cta + g);
    int bs0 = 0, bs1 = 0, ctas_in_block = 1;
    if (c >= 0) {
        bs0 = __ldg(p.blk_slice_ptr + c);
        bs1 = __ldg(p.blk_slice_ptr + c + 1);
        ctas_in_block = __ldg(p.cta_info + 2 * p.n_cta + c) / (kSellThreads / 32);
    }
    const bool has_slices = c >= 0 && bs1 > bs0;
    const int col0 = c >= 0 ? c * p.CB : 0;
    const int cnt = c >= 0 ? min(p.CB, p.n_cols - col0) : 0;
    // rows this CTA owns in the epilogue phases (one or two per thread on the named shapes)
    const int r0 = __ldg(p.cta_info + 2 * p.n_cta + kSellMaxBlocks + g);       // ranges of equal cost (sell_cta_rows_kernel)
    const int r1 = __ldg(p.cta_info + 2 * p.n_cta + kSellMaxBlocks + g + 1);
    // the hub rows of that range (summed by whole warps) are dealt to the warps in turn: warp w
    // takes the w-th, (w + 32)-th, ... of the plan's list
    if (tid < kWarps) {
        const int hb = __ldg(p.hub + g), he = __ldg(p.hub + g + 1);
        hub_first[tid] = hb + tid < he ? __ldg(p.hub + p.n_cta + 1 + hb + tid) : -1;
        if (tid == 0) { hub_span[0] = hb; hub_span[1] = he; }
    }

    unsigned long long* bar_ctr = reinterpret_cast<unsigned long long*>(p.sched + kSchedBarrier);
    // what only thread 0 uses lives in shared memory, not in every thread's registers
    __shared__ unsigned long long bar_base;
    __shared__ int stamp_i, trace_i;
    unsigned epoch_base = 0;
    if (tid == 0) {
        const unsigned long long seen = ld_relaxed_gpu_u64(bar_ctr);
        bar_base = seen - seen % n_cta;
        stamp_i = 1;
        trace_i = 0;
        mbar_init(&stage_bar, 1);
        if (p.stamps && g == 0) p.stamps[0] = global_timer_ns();
    }
    if (PEER) epoch_base = *p.epoch;                           // bumped only by CTA 0 after the first barrier
    unsigned bar_done = 0;                                     // grid barriers completed in this launch (same on every thread)
    unsigned signals = 0;                                      // flags this rank has raised in this launch
    unsigned stage_parity = 0;
    bool pending = false, pending_signal = false;              // a barrier this CTA has arrived at but not yet waited for
    const bool late_done = PEER && p.delta.n > 0;              // the last epilogue reads the window (edge-flip corrections)
    // PATCH: every CTA re-derives dinv / iso / x0 / dinv * x0 of the nodes the flips touch (the
    // arithmetic of patch_nodes_kernel, prep.cuh) into shared memory - no patch / restore launches
    // around the step and no patched copies of the vectors
    const int n_touch = PATCH ? 2 * p.delta.n : 0;
    bool touched_here = false;
    if (PATCH) {
        if (tid < n_touch) {
            const int u = tid < p.delta.n ? p.delta.row[tid] : p.delta.col[tid - p.delta.n];
            float dw = 0.f, dr = 0.f;
            for (int j = 0; j < p.delta.n; ++j) {
                if (p.delta.col[j] == u && p.delta.row[j] != u) dw += p.delta.val[j];     // in-degree (self loops excluded)
                if (p.delta.row[j] == u) dr += p.delta.val[j];                            // row sum (self loops count)
            }
            float dv;
            uint8_t is;
            normaliser_from_w(__ldg(p.w_base + u) + dw, dv, is);
            const int lr = u - p.row0;
            float x = 0.f;                                     // a caller's signal is only ever needed for the own rows
            if (p.patch_x0) x = (float)log1p((double)(__ldg(p.rowsum_base + u) + dr));
            else if (lr >= 0 && lr < p.n_rows) x = __ldg(p.x0 + lr);
            pt_node[tid] = u; pt_dinv[tid] = dv; pt_iso[tid] = is; pt_x0[tid] = x; pt_y0[tid] = dv * x;
            if (p.t_all && p.order_begin == 1 && lr >= r0 && lr < r1) p.t_all[lr] = x;   // T_0 row handed back to the caller
        }
        for (int d = 0; d < p.delta.n; ++d) {
            const int a = p.delta.row[d] - p.row0, b = p.delta.col[d] - p.row0;
            touched_here |= (a >= r0 && a < r1) || (b >= r0 && b < r1);
        }
    }
    __syncthreads();

    // Before a phase stores into the windows: the buffer it writes was last read by the staging
    // of the order before (or of the previous step), and a rank signals only after its grid
    // barrier behind that staging - so every rank's latest signal must be in.  Ranks whose
    // columns this rank's slices never touch are not waited for anywhere else.  Issued by warp 0
    // before a __syncthreads (the flags are long up by then on balanced shards).
    auto wait_windows_free = [&]() {
        if (PEER && wid == 0) peer_wait_ranks(p.local_flags, 0, p.world - 1, p.rank, epoch_base + signals, p.error, false, lane);
    };
    // after a grid barrier that closed a producing phase: CTA 0 raises this rank's flag everywhere
    auto signal_peers = [&]() {
        signals += 1u;
        if (PEER && g == 0 && tid == 0) {
            const unsigned e = epoch_base + signals;
            *p.epoch = e;
            __threadfence_system();                            // release: every CTA's stores (seen through the barrier) first
            for (int q = 0; q < p.world; ++q)
                if (q != p.rank) st_relaxed_sys_u32(p.flag_at[q], e);
        }
    };
    auto stamp = [&]() {
        if (tid == 0) {
            if (p.stamps && g == 0) p.stamps[stamp_i] = global_timer_ns();
            ++stamp_i;
        }
    };
    // per-CTA trace (diagnostic; the stamps buffer then holds 64 + 64 * n_cta words)
    auto trace = [&]() {
        if (tid == 0) {
            if (p.stamps && p.trace && trace_i < 64) p.stamps[64 + (size_t)g * 64 + trace_i] = global_timer_ns();
            ++trace_i;
        }
    };
    // the two halves of a grid barrier (every thread calls both; thread 0 does the work)
    auto bar_arrive = [&](bool sys_scope) {
        __syncthreads();
        if (tid == 0) grid_arrive(bar_ctr, sys_scope);
    };
    auto bar_wait = [&]() {
        if (tid == 0) grid_wait(bar_ctr, bar_base + (unsigned long long)(bar_done + 1u) * n_cta);
        bar_done += 1u;
        __syncthreads();
    };
    // close a producing phase whose barrier is still open: wait, signal the peers, stamp
    auto finish_pending = [&]() {
        if (pending) {
            bar_wait();
            if (pending_signal) signal_peers();
            stamp();
            pending = false;
        }
    };

    // ---- order 0: the first operand y_0 = dinv (.) T_0, unless the caller holds it -------------
    if (p.order_begin == 1 && p.operand_first == nullptr) {
        wait_windows_free();
        __syncthreads();
        for (int i = r0 + tid; i < r1; i += kSellThreads) {
            float yv = __ldg(p.dinv + p.row0 + i) * __ldg(p.x0 + i);
            if (PATCH && touched_here) {
                const int j = step_patch_find(pt_node, n_touch, p.row0 + i);
                if (j >= 0) yv = pt_y0[j];
            }
            for (int d = 0; d < p.n_dst; ++d) p.ydst[0][d][p.row0 + i] = yv;
        }
        bar_arrive(PEER);
        pending = true; pending_signal = true;
    }

    bool flips_here = false;
    for (int d = 0; d < p.delta.n; ++d) flips_here |= p.delta.row[d] - p.row0 >= r0 && p.delta.row[d] - p.row0 < r1;

    for (int k = p.order_begin; k <= p.order_end; ++k) {
        StepOrderView v;
        v.k = k; v.j = k - p.order_begin; v.flips_here = flips_here; v.flip_term = flip_term;
        v.touched_here = touched_here; v.n_touch = n_touch;
        v.pt_node = pt_node; v.pt_dinv = pt_dinv; v.pt_x0 = pt_x0; v.pt_iso = pt_iso;
        v.first = k == 1; v.last = k == p.k_max; v.push = k < p.k_max;
        const bool held = (k == p.order_begin) && p.operand_first != nullptr;
        v.operand = held ? p.operand_first : p.operand[(k - 1) & 1];
        v.tprev = step_t_ptr(p, k - 1);
        v.tprev2 = k >= 2 ? step_t_ptr(p, k - 2) : nullptr;
        v.tk = p.t_all ? p.t_all + (size_t)k * p.n_rows : (v.last ? nullptr : p.tbuf[(k - 1) & 1]);

        // ================= SpMV phase: slices of this CTA's column block ===================
        // what does not depend on the operand comes first: the warp's first slice is fixed
        // (warp w of the block's r-th CTA takes slice w * CTAs + r, so every CTA starts with the
        // same mix of long and short ones - on a row shard these first slices are most of the
        // work; the block's counter starts past them), its metadata and the head of its index
        // stream are requested while the previous phase's barrier completes
        int s = bs1, off = 0, end = 0, slot = -1;
        if (has_slices) {
            s = bs0 + wid * ctas_in_block + rank_in_block;
            if (s < bs1) {
                off = __ldg(p.slice_off + s);
                end = __ldg(p.slice_off + s + 1);
                slot = __ldg(p.vslot + (size_t)s * kSellSliceRows + lane);
                const char* head = reinterpret_cast<const char*>(p.idx + off) + lane * 128;
                if (head < reinterpret_cast<const char*>(p.idx + end)) asm volatile("prefetch.global.L2 [%0];" ::"l"(head));
            }
        }
        finish_pending();                                      // the operand of this order is complete (on this GPU)
        if (has_slices) {
            unsigned raw_next = 0;                             // later slices: requested one slice ahead of their use
            if (lane == 0) raw_next = atomicAdd(p.sched + c * kSellCtrStride, 1u);
            // stage the column block of the operand: bulk copies by one thread, tail and zero slots by the rest
            const float* src = v.operand + col0;
            const int cnt4 = cnt & ~3;
            if (wid == 0) {
                if (PEER && !held) {                           // written by the ranks owning these columns
                    const int p_lo = (int)(col0 / p.rows_per);
                    const int p_hi = (int)((col0 + cnt - 1) / p.rows_per);
                    peer_wait_ranks(p.local_flags, p_lo, min(p_hi, p.world - 1), p.rank, epoch_base + signals, p.error,
                                    g == 0, lane);
                }
                if (lane == 0) {
                    fence_proxy_async();                       // generic-proxy writes (other CTAs / GPUs, acquired above) before the async-proxy reads
                    if (cnt4 > 0) {
                        mbar_expect_tx(&stage_bar, (unsigned)cnt4 * 4u);
                        for (int o = 0; o < cnt4; o += kStageChunkFloats)
                            bulk_g2s(ysm + o, src + o, (unsigned)min(kStageChunkFloats, cnt4 - o) * 4u, &stage_bar);
                    }
                }
            }
            if (PEER && !held) __syncthreads();                // nobody touches the operand before the owners' flags are in
            if (tid >= 32) {                                   // warp 0 is busy issuing; the others fill the rest
                for (int t = cnt4 + tid - 32; t < p.CB + kSellZeroSlots; t += kSellThreads - 32)
                    ysm[t] = t < cnt ? __ldcg(src + t) : 0.f;
            }
            if (cnt4 > 0) mbar_wait(&stage_bar, stage_parity);
            stage_parity ^= (cnt4 > 0) ? 1u : 0u;
            __syncthreads();
            if (PATCH && held && k == 1) {                     // the caller's dinv (.) x0 is the base graph's
                if (tid < n_touch) {
                    const int loc = pt_node[tid] - col0;
                    if (loc >= 0 && loc < cnt) ysm[loc] = pt_y0[tid];
                }
                __syncthreads();
            }
            trace();                                           // operand block staged

            while (s < bs1) {
                // slice after this one: its number arrives from the atomic issued one slice ago;
                // the one after that is requested now
                int s_next = bs0 + (int)__shfl_sync(0xffffffffu, raw_next, 0);
                if (lane == 0) raw_next = atomicAdd(p.sched + c * kSellCtrStride, 1u);
                int off_next = 0, end_next = 0, slot_next = -1;
                if (s_next < bs1) {
                    off_next = __ldg(p.slice_off + s_next);
                    end_next = __ldg(p.slice_off + s_next + 1);
                    slot_next = __ldg(p.vslot + (size_t)s_next * kSellSliceRows + lane);
                }
                const int groups = (end - off) / (kSellGroup * kSellSliceRows);
                const uint4* q0 = reinterpret_cast<const uint4*>(p.idx + off) + lane;
                float acc0 = 0.f, acc1 = 0.f;
                int gq = 0;
                for (; gq + kSellUnroll <= groups; gq += kSellUnroll) {
                    uint4 q[kSellUnroll];
#pragma unroll
                    for (int u = 0; u < kSellUnroll; ++u) q[u] = ld_stream_u32x4(q0 + (size_t)(gq + u) * kSellSliceRows);
#pragma unroll
                    for (int u = 0; u < kSellUnroll; ++u) {
                        if (u & 1) acc1 += sell_gather8(ysm, q[u]);
                        else acc0 += sell_gather8(ysm, q[u]);
                    }
                }
                for (; gq < groups; ++gq) acc0 += sell_gather8(ysm, ld_stream_u32x4(q0 + (size_t)gq * kSellSliceRows));
                if (slot >= 0) p.vpart[slot] = acc0 + acc1;
                s = s_next; off = off_next; end = end_next; slot = slot_next;
            }
        }
        bar_arrive(false);                                     // this CTA's partial sums are in place; shared memory is free
        trace();
        // (measured and dropped: prefetching the head of the next order's index stream into L2
        // while HBM idles here made the step slower for every amount tried, DESIGN.md section 4.2)

        // ================= epilogue phase: the CTA's own rows ================================
        // what a row needs besides its partial sums is requested before the wait for everybody's
        // partial sums: for the thread's rows A and B and for the warp's first hub row
        const int i_a = r0 + tid, i_b = r0 + tid + kSellThreads;
        const int i_h = hub_first[wid];                        // uniform per warp
        StepRowPre pre_a{}, pre_b{};
        if (i_a < r1) pre_a = step_row_prefetch<PATCH>(p, v, i_a);
        if (i_b < r1) pre_b = step_row_prefetch<PATCH>(p, v, i_b);
        const uint32_t wh = i_h >= 0 ? step_hub_prefetch(p, v, i_h, lane) : 0u;
        // (exchange) before this phase stores into the windows, and before a flip's term is read
        // from a column whose owner none of this CTA's waits covered: every rank's latest signal.
        // Polled by warp 0 while the grid barrier completes.
        if (PEER && (v.push || flips_here)) {
            wait_windows_free();
            if (flips_here) __syncthreads();                   // uniform per CTA
        }
        if (flips_here && tid < p.delta.n) {                   // the flips' terms: the operand of this order is complete
            const int lr = p.delta.row[tid] - p.row0, dc = p.delta.col[tid];
            const float yc = (PATCH && held && k == 1) ? pt_y0[p.delta.n + tid] : __ldcg(v.operand + dc);
            flip_term[tid] = (lr >= r0 && lr < r1 && dc != p.delta.row[tid]) ? p.delta.val[tid] * yc : 0.f;
        }
        bar_wait();                                            // every partial sum of every row is in place
        stamp();
        // end-of-step signal: nobody reads the windows any more - unless edge flips are applied,
        // whose corrections the last epilogue still reads from the operand (signalled after it)
        if (PEER && v.last && !late_done) signal_peers();
        if (g == 0 && tid < p.C) p.sched[tid * kSellCtrStride] = (unsigned)__ldg(p.cta_info + 2 * p.n_cta + tid);   // counters for the next SpMV phase
        // the partial sums of rows A and B (the first kEpiFirstParts of each) and of the warp's hub
        // row (the lanes' first ones) are all requested before any is added: one round trip to L2;
        // a hub row is left to its warp by the thread whose row it is
        const bool own_a = i_a < r1 && pre_a.e - pre_a.t <= kEpiWarpRow;
        const bool own_b = i_b < r1 && pre_b.e - pre_b.t <= kEpiWarpRow;
        float xa[kEpiFirstParts], xb[kEpiFirstParts];
        step_row_load(p.vpart, pre_a.t, own_a ? pre_a.e : pre_a.t, xa);
        step_row_load(p.vpart, pre_b.t, own_b ? pre_b.e : pre_b.t, xb);
        const float xh = i_h >= 0 ? step_hub_first(p.vpart, (int)__shfl_sync(0xffffffffu, wh, 0),
                                                   (int)__shfl_sync(0xffffffffu, wh, 1), lane) : 0.f;
        if (own_a) step_epilogue_finish(p, v, i_a, pre_a, step_row_sum_rest(p.vpart, pre_a.t, pre_a.e, xa));
        if (own_b) step_epilogue_finish(p, v, i_b, pre_b, step_row_sum_rest(p.vpart, pre_b.t, pre_b.e, xb));
        for (int i = i_b + kSellThreads; i < r1; i += kSellThreads) {      // ranges of more than 2048 rows
            const StepRowPre r = step_row_prefetch<PATCH>(p, v, i);
            if (r.e - r.t <= kEpiWarpRow) step_epilogue_finish(p, v, i, r, step_row_sum(p.vpart, r.t, r.e));
        }
        if (i_h >= 0) {
            step_hub_finish(p, v, i_h, step_hub_gather<PATCH>(p, v, i_h, wh), xh, lane);
            for (int h = hub_span[0] + wid + kWarps; h < hub_span[1]; h += kWarps) {   // more hub rows than warps
                const int i = __ldg(p.hub + p.n_cta + 1 + h);
                const StepRowPre r = step_row_prefetch<PATCH>(p, v, i);
                step_hub_finish(p, v, i, r, step_hub_first(p.vpart, r.t, r.e, lane), lane);
            }
        }
        // the next order (or a peer) reads what this phase wrote
        if (k < p.order_end || (PEER && (v.push || (v.last && late_done)))) {
            bar_arrive(PEER && v.push);
            pending = true; pending_signal = v.push || (v.last && late_done);
        }
        trace();                                               // this CTA's rows are done
    }
    finish_pending();
    if (p.stamps && g == 0 && tid == 0) p.stamps[stamp_i] = global_timer_ns();
}

}  // namespace egnn

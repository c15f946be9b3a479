// extern "C" surface of libegnn_b200.so (declared in include/egnn_b200.h).
// Host-side driver logic only: argument checks, kernel selection, launches on
// the caller's stream.  No allocation, no synchronisation, no global state.
#include <stdarg.h>
#include <stdlib.h>

#include "adjoint.cuh"
#include "cheb.cuh"
#include "common.cuh"
#include "head.cuh"
#include "metrics.cuh"
#include "peer.cuh"
#include "prep.cuh"
#include "sell.cuh"
#include "sell_step.cuh"
#include "shard_grad.cuh"
#include "structure_grad.cuh"
#include "surrogate.cuh"
#include "blocked.cuh"
#include "wide.cuh"

namespace egnn {

static thread_local char g_err[512] = {0};
char* last_error_buf() { return g_err; }
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

static int device_sm_count();
constexpr int kWideMinF = 8;             // narrower signals keep the multi-row-per-warp kernel (cheb.cuh)
constexpr int64_t kBlockedMinNnz = int64_t(1) << 22;   // below this the CSR is L2-resident: the generic kernel is as fast
constexpr int kWideDynamicMaxDegree = 64;   // mean entries per row below which the wide kernel hands rows out dynamically

static int pow2_ceil_log2(int64_t x) {
    int l = 0;
    while ((int64_t(1) << l) < x) ++l;
    return l;
}

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Caller arrays of row stride f are read and written with 16-byte vector accesses when
// f % 4 == 0 (FeatVec<4>, load_user4<true>), so their base addresses must be 16-byte aligned then.
static inline bool vec_aligned(const void* p, int32_t f) {
    return f % 4 != 0 || p == nullptr || ((uintptr_t)p & 15) == 0;
}

// The caller's edge flips into `d`.  Every index must address a node below `bound`: n, or the
// global node count of a row shard.
static int fill_delta(DeltaList& d, const int32_t* r, const int32_t* c, const float* v, int32_t n, int64_t bound) {
    EGNN_REQUIRE(n >= 0 && n <= EGNN_MAX_DELTA, "n_delta out of range");
    EGNN_REQUIRE(n == 0 || (r && c && v), "delta arrays missing");
    d.n = n;
    for (int i = 0; i < n; ++i) {
        EGNN_REQUIRE(r[i] >= 0 && r[i] < bound && c[i] >= 0 && c[i] < bound, "delta index out of range");
        d.row[i] = r[i]; d.col[i] = c[i]; d.val[i] = v[i];
    }
    return EGNN_OK;
}

// `what` names the workspace in the message ("sell workspace", "transpose workspace", ...)
static int require_workspace(const void* ws, size_t bytes, size_t need, const char* what) {
    if (ws && bytes >= need) return EGNN_OK;
    set_error("%s too small: need %zu bytes, got %zu", what, need, bytes);
    return EGNN_ERR_WORKSPACE;
}

// Event i of the caller's per-order timing list (two per order: before and after), if it gave one.
static int record_event(void* const* events, int i, cudaStream_t st) {
    return events ? check_cuda(cudaEventRecord((cudaEvent_t)events[i], st), "event record") : EGNN_OK;
}

// Coefficient of order m of every scale, from the caller's [S, k + 1] host table.
static void order_coefs(float* dst, const float* coeffs_host, int k, int S, int m) {
    for (int s = 0; s < S; ++s) dst[s] = coeffs_host[s * (k + 1) + m];
}
static CoefRow coef_row(const float* coeffs_host, int k, int S, int m) {
    CoefRow c{};
    order_coefs(c.c, coeffs_host, k, S, m);
    return c;
}

// Row width of the wide kernel's operand slabs and exchange windows: F padded to 16 bytes.
static inline int wide_ldy(int32_t f) { return (f + 3) / 4 * 4; }

// Slab m of a [*, rows, F] stack, or NULL without one.
template <typename T>
static inline T* slab_of(T* stack, size_t slab_elems, int m) {
    return stack ? stack + (size_t)m * slab_elems : nullptr;
}

// Lane layout and instantiation for one order launch.
struct OrderConfig {
    int vec, u, fl_log2, nz_log2, tile, grid_y;
    bool prescaled;
};

static OrderConfig choose_config(int64_t n_rows, int64_t nnz, int32_t F) {
    OrderConfig c{};
    if (F % 4 == 0) { c.vec = 4; c.u = 1; }
    else if (F <= 32) { c.vec = 1; c.u = 1; }
    else { c.vec = 1; c.u = 4; }
    const int per_lane = c.vec * c.u;
    int fl = pow2_ceil_log2((F + per_lane - 1) / per_lane);
    if (c.vec == 1 && c.u == 4) fl = 5;           // u-strided layout wants the full warp
    if (fl > 5) fl = 5;
    c.fl_log2 = fl;
    c.tile = (1 << fl) * per_lane;
    c.grid_y = (F + c.tile - 1) / c.tile;
    // non-zeros in parallel: about half the mean row length, within the warp
    const double mean = n_rows > 0 ? double(nnz) / double(n_rows) : 1.0;
    int nz = 0;
    while (nz < 5 - fl && double(1 << (nz + 1)) <= mean * 0.75) ++nz;
    c.nz_log2 = nz;
    c.prescaled = (F <= 4);
    return c;
}

template <int VEC, int U, bool ADJ>
static void launch_order_vu(const OrderParams& p, bool has_vals, bool prescaled, dim3 grid,
                            cudaStream_t st) {
    if (has_vals) {
        if (prescaled) cheb_order_kernel<VEC, U, true, true, ADJ><<<grid, kOrderBlock, 0, st>>>(p);
        else cheb_order_kernel<VEC, U, true, false, ADJ><<<grid, kOrderBlock, 0, st>>>(p);
    } else {
        if (prescaled) cheb_order_kernel<VEC, U, false, true, ADJ><<<grid, kOrderBlock, 0, st>>>(p);
        else cheb_order_kernel<VEC, U, false, false, ADJ><<<grid, kOrderBlock, 0, st>>>(p);
    }
}

// ADJ: the adjoint instantiation (an application of M^T in the backward pass)
template <bool ADJ = false>
static int launch_order(const OrderParams& p, const OrderConfig& c, cudaStream_t st) {
    if (p.n_rows == 0) return EGNN_OK;
    const int rows_per_block = (kOrderBlock / 32) * (32 >> (c.fl_log2 + c.nz_log2));
    dim3 grid((unsigned)ceil_div64(p.n_rows, rows_per_block), (unsigned)c.grid_y, 1);
    const bool has_vals = p.vals != nullptr;
    if (c.vec == 4) launch_order_vu<4, 1, ADJ>(p, has_vals, c.prescaled, grid, st);
    else if (c.u == 1) launch_order_vu<1, 1, ADJ>(p, has_vals, c.prescaled, grid, st);
    else launch_order_vu<1, 4, ADJ>(p, has_vals, c.prescaled, grid, st);
    EGNN_LAUNCH_CHECK("cheb_order_kernel launch");
    return EGNN_OK;
}

// Lane layout of the wide kernel for a padded row width ldy (multiple of 4):
// FL feature lanes x NZ entry slots, tiles of FL * 4 columns in gridDim.y.
struct RingConfig { int nz_log2, grid_y; };
static RingConfig ring_config(int ldy) {
    int fl_log2 = pow2_ceil_log2((ldy + 3) / 4);
    if (fl_log2 > 5) fl_log2 = 5;
    RingConfig c;
    c.nz_log2 = 5 - fl_log2;
    const int tile = (1 << fl_log2) * 4;
    c.grid_y = (ldy + tile - 1) / tile;
    return c;
}

template <int NZ_LOG2, bool PEER, bool DYN, bool ADJ>
static int launch_wide_npd(const WideParams& p, dim3 grid, cudaStream_t st) {
    const bool aligned = (p.F % 4) == 0;
    if (p.vals) {
        if (aligned) cheb_wide_kernel<NZ_LOG2, true, true, PEER, DYN, ADJ><<<grid, kWideBlock, 0, st>>>(p);
        else cheb_wide_kernel<NZ_LOG2, true, false, PEER, DYN, ADJ><<<grid, kWideBlock, 0, st>>>(p);
    } else {
        if (aligned) cheb_wide_kernel<NZ_LOG2, false, true, PEER, DYN, ADJ><<<grid, kWideBlock, 0, st>>>(p);
        else cheb_wide_kernel<NZ_LOG2, false, false, PEER, DYN, ADJ><<<grid, kWideBlock, 0, st>>>(p);
    }
    EGNN_LAUNCH_CHECK("cheb_wide_kernel launch");
    return EGNN_OK;
}

// DYN instantiation (single GPU only): rows handed out from p.row_counter
template <int NZ_LOG2, bool PEER, bool ADJ>
static int launch_wide_np(const WideParams& p, dim3 grid, cudaStream_t st) {
    if (!PEER && p.row_counter) return launch_wide_npd<NZ_LOG2, false, true, ADJ>(p, grid, st);
    return launch_wide_npd<NZ_LOG2, PEER, false, ADJ>(p, grid, st);
}

// PEER instantiation: operand in the exchange window, written by the other GPUs (world > 1),
// for the forward orders and the adjoint applications alike.
template <int NZ_LOG2, bool ADJ>
static int launch_wide_n(const WideParams& p, dim3 grid, cudaStream_t st) {
    return p.peer.world > 1 ? launch_wide_np<NZ_LOG2, true, ADJ>(p, grid, st)
                            : launch_wide_np<NZ_LOG2, false, ADJ>(p, grid, st);
}

// (Measured and dropped: pinning the gather operand in L2 with an access-policy window and the
// persisting set-aside - arxiv F = 128 0.283 -> 0.276 ms per order, Reddit F = 64 2.13 -> 2.28,
// Physics F = 8415 2.77 -> 3.6: the set-aside shrinks the L2 left for the other four slabs.)
// Wide kernel: persistent grid of kWideMinBlocks CTAs per SM per feature tile.
template <bool ADJ = false>
static int launch_wide(const WideParams& p, const RingConfig& c, int sm_count, cudaStream_t st) {
    dim3 grid((unsigned)(sm_count * kWideMinBlocks), (unsigned)c.grid_y, 1);
    switch (c.nz_log2) {
        case 0: return launch_wide_n<0, ADJ>(p, grid, st);
        case 1: return launch_wide_n<1, ADJ>(p, grid, st);
        case 2: return launch_wide_n<2, ADJ>(p, grid, st);
        case 3: return launch_wide_n<3, ADJ>(p, grid, st);
        default: return launch_wide_n<4, ADJ>(p, grid, st);
    }
}

static int grid_for(int64_t work_items, int threads) {
    int64_t b = ceil_div64(work_items, threads);
    const int64_t cap = (int64_t)kSmCountB200 * 16;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (int)b;
}

// Row L1 normalisation of `rows` x S feature vectors of width f, after the last order.
static int launch_l1_normalize(float* out, int64_t rows, int32_t S, int32_t f, cudaStream_t st) {
    l1_normalize_kernel<<<grid_for(rows * S * 32, 256), 256, 0, st>>>(out, rows * S, f);
    EGNN_LAUNCH_CHECK("l1_normalize_kernel launch");
    return EGNN_OK;
}

// Grid of a kernel that pushes `items` floats into the peer windows with 1024 threads per CTA:
// at most one CTA per SM, since each CTA issues one system-scope fence.
static unsigned push_grid(int64_t items) {
    const int64_t blocks = ceil_div64(items > 0 ? items : 1, 1024);
    const int sms = device_sm_count();
    return (unsigned)(blocks > sms ? sms : blocks);
}

static int launch_degree(const int32_t* rowptr, const int32_t* colidx, const float* vals_or_null, int64_t rows,
                         float* rowsum, float* diag, double* colsum, int32_t* unsorted_flag_or_null, int64_t row0,
                         cudaStream_t st) {
    const auto kernel = vals_or_null ? degree_kernel<true> : degree_kernel<false>;
    kernel<<<grid_for(rows * 32, 256), 256, 0, st>>>(rowptr, colidx, vals_or_null, rows, rowsum, diag, colsum,
                                                      unsorted_flag_or_null, row0);
    EGNN_LAUNCH_CHECK("degree_kernel launch");
    return EGNN_OK;
}

// Column blocks of the shared-memory staged narrow paths (SELL plan and plan-free blocked kernel)
static void narrow_geometry(int64_t n, int* n_blocks, int* col_block) {
    const int64_t cb_max = 49152;                     // 192 KB of float32 operand per CTA
    const int64_t c = ceil_div64(n, cb_max);
    int64_t cb = ceil_div64(ceil_div64(n, c), 32) * 32;
    if (cb > 65504) cb = 65504;
    *n_blocks = (int)ceil_div64(n, cb);
    *col_block = (int)cb;
}

// ---- Chebyshev workspace layout (egnn_cheb_workspace_bytes; forward and adjoint) ---------------
// f < 8: two T slabs, ping-pong for T_{k-1} / T_{k-2} (the adjoint's b vectors), and for f <= 4
// two pre-scaled operand slabs dinv (.) T.  f >= 8: two operand slabs with rows padded to 16 bytes
// and one row counter per (order, feature tile) for the wide kernel's dynamic row schedule.
// f == 1 adds the segment table, partial sums and counters of the plan-free blocked kernel.
struct ChebWs {
    float* t[2];
    float* y[2];
    unsigned* row_counters;
    int C, CB;                   // blocked kernel: column blocks the next three are sized for
    int32_t* seg;
    float* part;
    unsigned* blk_counters;
    size_t total_bytes;
};

static ChebWs cheb_ws_layout(void* base, int64_t n, int32_t f) {
    ChebWs w{};
    size_t off = 0;
    char* b = (char*)align_up((size_t)base, 256);
    auto take = [&](size_t bytes) { void* ptr = b + off; off += align_up(bytes, 256); return ptr; };
    if (f >= kWideMinF) {
        const size_t ldy = (size_t)wide_ldy(f);
        w.y[0] = (float*)take(sizeof(float) * (size_t)n * ldy);
        w.y[1] = (float*)take(sizeof(float) * (size_t)n * ldy);
        w.row_counters = (unsigned*)take(sizeof(unsigned) * (size_t)EGNN_MAX_ORDER * ((ldy + 127) / 128));
    } else {
        const size_t slab = sizeof(float) * (size_t)n * (size_t)f;
        w.t[0] = (float*)take(slab);
        w.t[1] = (float*)take(slab);
        if (f <= 4) {
            w.y[0] = (float*)take(slab);
            w.y[1] = (float*)take(slab);
        }
        if (f == 1) {
            narrow_geometry(n > 0 ? n : 1, &w.C, &w.CB);
            w.seg = (int32_t*)take(4 * (size_t)(w.C + 1) * (size_t)n);
            w.part = (float*)take(4 * (size_t)w.C * (size_t)n);
            w.blk_counters = (unsigned*)take(4 * (size_t)EGNN_MAX_ORDER * (size_t)w.C);
        }
    }
    w.total_bytes = off + 256;
    return w;
}

// ---- one pass of the Chebyshev recurrence, forward or adjoint ------------------------------------
// The rows a pass runs over (all n, or one row shard: local row r is node row0 + r), their CSR (of the
// transposed graph for the adjoint), the operator a * L_sym + b * I and the [S, k + 1] coefficients.
struct ChebArgs {
    const int32_t* rowptr;
    const int32_t* colidx;
    const float* vals;           // NULL: binary adjacency
    const int32_t* row_order;    // wide kernel: degree-descending row order and hub count, or NULL
    const float* dinv;
    const uint8_t* iso;
    int64_t rows, row0, nnz;
    int32_t f, k, S;
    const float* coeffs;         // host
    float a, b;
    DeltaList delta;
    void* const* events;         // two per order (application), or NULL
    cudaStream_t st;
};

static WideParams wide_params(const ChebArgs& c) {
    WideParams wp{};
    wp.delta = c.delta;
    wp.rowptr = c.rowptr; wp.colidx = c.colidx; wp.vals = c.vals;
    wp.perm = c.row_order; wp.n_hub = c.row_order ? c.row_order + c.rows : nullptr;
    wp.dinv = c.dinv; wp.iso = c.iso; wp.n_rows = c.rows; wp.row0 = c.row0;
    wp.F = c.f; wp.ldy = wide_ldy(c.f); wp.S = c.S; wp.a = c.a; wp.b = c.b;
    return wp;
}

static OrderParams order_params(const ChebArgs& c, const OrderConfig& cfg) {
    OrderParams p{};
    p.delta = c.delta;
    p.rowptr = c.rowptr; p.colidx = c.colidx; p.vals = c.vals; p.dinv = c.dinv; p.iso = c.iso;
    p.n_rows = c.rows; p.row0 = c.row0; p.F = c.f; p.S = c.S; p.a = c.a; p.b = c.b;
    p.fl_log2 = cfg.fl_log2; p.nz_log2 = cfg.nz_log2;
    return p;
}


// ---- SELL plan workspace layout (shared by prepare and fill) -----------------
struct SellWs {
    int32_t *seg_start, *seg_cnt, *nv, *u_off, *nvrow, *rv_ptr, *uval, *perm, *vsrc, *vslot, *vrow;
    uint32_t *key, *key_sorted;
    int32_t *q_ptr, *vp_ptr, *bsp, *bstride, *slice_sz, *slice_off;
    int64_t* totals;
    void* cub_temp;
    size_t cub_bytes;
    size_t total_bytes;
    int64_t umax, smax;
};

static size_t sell_cub_bytes(int64_t cn1, int64_t n1, int64_t umax, int64_t smax1) {
    size_t a = 0, b = 0, c = 0, d = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, a, (int32_t*)nullptr, (int32_t*)nullptr, (int)cn1);
    cub::DeviceScan::ExclusiveSum(nullptr, b, (int32_t*)nullptr, (int32_t*)nullptr, (int)n1);
    cub::DeviceScan::ExclusiveSum(nullptr, c, (int32_t*)nullptr, (int32_t*)nullptr, (int)smax1);
    cub::DeviceRadixSort::SortPairs(nullptr, d, (uint32_t*)nullptr, (uint32_t*)nullptr, (int32_t*)nullptr,
                                    (int32_t*)nullptr, (int)umax);
    size_t m = a > b ? a : b;
    m = m > c ? m : c;
    m = m > d ? m : d;
    return m + 256;
}

static SellWs sell_ws_layout(void* base, int64_t n, int64_t nnz, int C, int lmax) {
    SellWs w{};
    const int64_t cn = (int64_t)C * n;
    w.umax = cn + nnz / lmax + 1;
    w.smax = (w.umax + (int64_t)kSellSliceRows * C) / kSellSliceRows + 1;
    size_t off = 0;
    char* b = (char*)align_up((size_t)base, 256);
    auto take = [&](size_t bytes) { void* ptr = b + off; off += align_up(bytes, 256); return ptr; };
    w.seg_start = (int32_t*)take(4 * cn);
    w.seg_cnt = (int32_t*)take(4 * cn);
    w.nv = (int32_t*)take(4 * (cn + 1));
    w.u_off = (int32_t*)take(4 * (cn + 1));
    w.nvrow = (int32_t*)take(4 * (n + 1));
    w.rv_ptr = (int32_t*)take(4 * (n + 1));
    w.key = (uint32_t*)take(4 * w.umax);
    w.key_sorted = (uint32_t*)take(4 * w.umax);
    w.uval = (int32_t*)take(4 * w.umax);
    w.perm = (int32_t*)take(4 * w.umax);
    w.vsrc = (int32_t*)take(4 * w.umax);
    w.vslot = (int32_t*)take(4 * w.umax);
    w.vrow = (int32_t*)take(4 * w.umax);
    w.q_ptr = (int32_t*)take(4 * (C + 1));
    w.vp_ptr = (int32_t*)take(4 * (C + 1));
    w.bsp = (int32_t*)take(4 * (C + 1));
    w.bstride = (int32_t*)take(4 * (C + 1));
    w.slice_sz = (int32_t*)take(4 * (w.smax + 1));
    w.slice_off = (int32_t*)take(4 * (w.smax + 1));
    w.totals = (int64_t*)take(8 * 8);
    w.cub_bytes = sell_cub_bytes(cn + 1, n + 1, w.umax, w.smax + 1);
    w.cub_temp = take(w.cub_bytes);
    w.total_bytes = off + 256;
    return w;
}

static int sell_check_geometry(int64_t n, int64_t nnz, const egnn_sell_plan* plan) {
    EGNN_REQUIRE(plan != nullptr, "null plan");
    EGNN_REQUIRE(plan->n_cols >= 1 && plan->row0 >= 0 && (int64_t)plan->row0 + n <= plan->n_cols,
                 "row shard [row0, row0 + n) must lie inside n_cols");
    EGNN_REQUIRE(n >= 1 && n < (int64_t(1) << 31) && nnz >= 0 && nnz < (int64_t(1) << 31), "n/nnz out of range");
    EGNN_REQUIRE(plan->n_blocks >= 1 && plan->n_blocks <= kSellMaxBlocks, "n_blocks out of range");
    EGNN_REQUIRE(plan->col_block >= 32 && plan->col_block % 32 == 0 && plan->col_block + kSellZeroSlots <= 65536,
                 "col_block must be a multiple of 32 that leaves room for the zero slots in 16-bit local indices");
    EGNN_REQUIRE((int64_t)plan->col_block * plan->n_blocks >= plan->n_cols, "column blocks do not cover n_cols");
    EGNN_REQUIRE(plan->lmax >= 8 && plan->lmax <= kSellLmaxCap && plan->lmax % 8 == 0, "lmax must be a multiple of 8 in [8, 256]");
    EGNN_REQUIRE((int64_t)plan->n_blocks * n < (int64_t(1) << 30), "n_blocks * n too large");
    return EGNN_OK;
}

static inline size_t peer_slab_stride(const egnn_peer_window* w) {
    return align_up(sizeof(float) * (size_t)w->world * (size_t)w->rows_per * (size_t)w->f, 256);
}
static inline float* peer_operand(const egnn_peer_window* w, int r, int which) {
    return (float*)((char*)w->base[r] + kPeerHeaderBytes + (size_t)which * peer_slab_stride(w));
}
static int peer_check(const egnn_peer_window* w) {
    EGNN_REQUIRE(w->world >= 1 && w->world <= EGNN_MAX_RANKS && w->rank >= 0 && w->rank < w->world, "bad rank/world");
    EGNN_REQUIRE(w->rows_per >= 1 && w->f >= 1, "bad window shape");
    for (int r = 0; r < w->world; ++r) EGNN_REQUIRE(w->base[r] != nullptr, "window of a rank is not mapped");
    return EGNN_OK;
}
static void fill_peer_push(PeerPush& pp, const egnn_peer_window* w, int which, bool has_data, bool wait_first) {
    pp.world = w->world; pp.rank = w->rank; pp.wait_first = wait_first; pp.has_data = has_data;
    char* own = (char*)w->base[w->rank];
    for (int r = 0; r < w->world; ++r) {
        pp.dst[r] = peer_operand(w, r, which);
        pp.flag[r] = (unsigned*)((char*)w->base[r] + kPeerFlagsOff) + w->rank;
    }
    pp.local_flags = (unsigned*)(own + kPeerFlagsOff);
    pp.epoch = (unsigned*)(own + kPeerEpochOff);
    pp.done_ctr = (unsigned*)(own + kPeerDoneOff);
    pp.error = (unsigned*)(own + kPeerErrorOff);
}

// ---- the narrow-path step kernel (sell_step.cuh) ------------------------------
static void step_fill_plan(SellStepParams& sp, const egnn_sell_plan* pl) {
    sp.idx = pl->idx; sp.slice_off = pl->slice_off; sp.blk_slice_ptr = pl->blk_slice_ptr; sp.vslot = pl->vslot;
    sp.cta_info = pl->cta_info; sp.hub = pl->hub; sp.rv_ptr = pl->rv_ptr; sp.vpart = pl->vpart; sp.sched = pl->sched;
    sp.stamps = (unsigned long long*)pl->stamps;
    sp.trace = pl->reserved;          // diagnostic: per-CTA trace behind the stamps (scripts/time_step.py)
    sp.n_cta = pl->n_cta; sp.C = pl->n_blocks; sp.CB = pl->col_block; sp.n_cols = pl->n_cols;
    sp.n_rows = pl->n; sp.row0 = pl->row0;
}

static void step_fill_peer(SellStepParams& sp, const egnn_peer_window* w) {
    sp.world = w->world; sp.rank = w->rank; sp.rows_per = w->rows_per;
    char* own = (char*)w->base[w->rank];
    for (int r = 0; r < w->world; ++r) sp.flag_at[r] = (unsigned*)((char*)w->base[r] + kPeerFlagsOff) + w->rank;
    sp.local_flags = (unsigned*)(own + kPeerFlagsOff);
    sp.epoch = (unsigned*)(own + kPeerEpochOff);
    sp.error = (unsigned*)(own + kPeerErrorOff);
}

// One cooperative launch: every CTA must be resident (grid barriers, and - row-sharded - flag
// waits on the other GPUs), one CTA per SM.
static int launch_sell_step(const SellStepParams& sp, bool peer, cudaStream_t st) {
    const size_t smem = sizeof(float) * ((size_t)sp.CB + kSellZeroSlots);
    const bool patch = sp.w_base != nullptr && sp.delta.n > 0;     // flips on top of the base graph's vectors
    const void* fn = peer ? (patch ? (const void*)sell_step_kernel<true, true> : (const void*)sell_step_kernel<true, false>)
                          : (patch ? (const void*)sell_step_kernel<false, true> : (const void*)sell_step_kernel<false, false>);
    int rc = check_cuda(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                        "cudaFuncSetAttribute(sell_step_kernel)");
    if (rc) return rc;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)sp.n_cta, 1, 1);
    cfg.blockDim = dim3(kSellThreads, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;
    attr[0].val.cooperative = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    void* args[1] = {(void*)&sp};
    return check_cuda(cudaLaunchKernelExC(&cfg, fn, args), "sell_step_kernel launch");
}

// Launches the orders order_begin..order_end (default 1..k) of one step in chunks of
// kStepMaxOrders.  `sp` carries everything but the order window.
static int run_sell_step(SellStepParams sp, int k, int n_scales, const float* coeffs_host, bool peer, cudaStream_t st,
                         int order_begin = 1, int order_end = -1) {
    if (order_end < 0) order_end = k;
    const float* held = sp.operand_first;
    for (int ob = order_begin; ob <= order_end; ob += kStepMaxOrders) {
        const int oe = ob + kStepMaxOrders - 1 < order_end ? ob + kStepMaxOrders - 1 : order_end;
        sp.order_begin = ob; sp.order_end = oe; sp.k_max = k; sp.S = n_scales;
        sp.operand_first = ob == order_begin ? held : nullptr;
        for (int s = 0; s < n_scales; ++s)
            for (int j = 0; j <= oe - ob + 1; ++j) sp.coef[s][j] = coeffs_host[s * (k + 1) + ob - 1 + j];
        int rc = launch_sell_step(sp, peer, st);
        if (rc) return rc;
    }
    return EGNN_OK;
}

static int device_sm_count() {
    int dev = 0, sms = kSmCountB200;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms;
}

}  // namespace egnn

using namespace egnn;

extern "C" {

int egnn_abi_version(void) { return 13; }

const char* egnn_last_error(void) { return last_error_buf(); }

int egnn_device_info(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor) {
    int dev = 0;
    int rc = check_cuda(cudaGetDevice(&dev), "cudaGetDevice");
    if (rc) return rc;
    cudaDeviceProp prop;
    rc = check_cuda(cudaGetDeviceProperties(&prop, dev), "cudaGetDeviceProperties");
    if (rc) return rc;
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    if (prop.major != 10) {
        set_error("libegnn_b200 is built for sm_100a only; device is sm_%d%d", prop.major, prop.minor);
        return EGNN_ERR_UNSUPPORTED_ARCH;
    }
    return EGNN_OK;
}

int egnn_dense_to_csr_count(const float* adj, int64_t n, int64_t ld, int32_t* rowptr,
                            int32_t* nonbinary, egnn_stream_t stream) {
    EGNN_REQUIRE(adj && rowptr && nonbinary, "null pointer");
    EGNN_REQUIRE(n >= 0 && ld >= n, "bad shape");
    cudaStream_t st = (cudaStream_t)stream;
    int rc = check_cuda(cudaMemsetAsync(nonbinary, 0, sizeof(int32_t), st), "memset nonbinary");
    if (rc) return rc;
    if (n > 0) {
        dense_count_kernel<<<grid_for(n * 32, 256), 256, 0, st>>>(adj, n, ld, rowptr + 1, nonbinary);
        EGNN_LAUNCH_CHECK("dense_count_kernel launch");
    }
    rowptr_scan_kernel<<<1, 1024, 0, st>>>(rowptr, n);
    EGNN_LAUNCH_CHECK("rowptr_scan_kernel launch");
    return EGNN_OK;
}

int egnn_dense_to_csr_fill(const float* adj, int64_t n, int64_t ld, const int32_t* rowptr,
                           int32_t* colidx, float* vals_or_null, egnn_stream_t stream) {
    EGNN_REQUIRE(adj && rowptr, "null pointer");
    EGNN_REQUIRE(n >= 0 && ld >= n, "bad shape");
    if (n == 0) return EGNN_OK;
    EGNN_REQUIRE(colidx != nullptr, "null colidx");
    dense_fill_kernel<<<grid_for(n * 32, 256), 256, 0, (cudaStream_t)stream>>>(adj, n, ld, rowptr, colidx,
                                                                               vals_or_null);
    EGNN_LAUNCH_CHECK("dense_fill_kernel launch");
    return EGNN_OK;
}

int egnn_degree_rows(const int32_t* rowptr, const int32_t* colidx, const float* vals_or_null, int64_t n,
                     int64_t row_begin, int64_t row_end, float* rowsum, float* diag, double* colsum,
                     int32_t* unsorted_flag_or_null, egnn_stream_t stream) {
    EGNN_REQUIRE(rowptr && rowsum && diag && colsum, "null pointer");
    EGNN_REQUIRE(n >= 0 && row_begin >= 0 && row_begin <= row_end && row_end <= n, "bad row range");
    const int64_t rows = row_end - row_begin;
    if (rows == 0) return EGNN_OK;
    // rowptr values are absolute positions in colidx, so a row range is the same kernel on shifted row arrays
    return launch_degree(rowptr + row_begin, colidx, vals_or_null, rows, rowsum + row_begin, diag + row_begin, colsum,
                         unsorted_flag_or_null, row_begin, (cudaStream_t)stream);
}

int egnn_graph_prep_finish(const double* colsum, const float* diag, const float* rowsum, int64_t n, float* dinv,
                           uint8_t* iso, float* x0_logdeg, float* w_out_or_null, egnn_stream_t stream) {
    EGNN_REQUIRE(colsum && diag && rowsum && dinv && iso, "null pointer");
    EGNN_REQUIRE(n >= 0, "bad shape");
    if (n == 0) return EGNN_OK;
    normaliser_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, (cudaStream_t)stream>>>(colsum, diag, rowsum, n, dinv, iso,
                                                                                    x0_logdeg, w_out_or_null);
    EGNN_LAUNCH_CHECK("normaliser_kernel launch");
    return EGNN_OK;
}

int egnn_graph_prep(const int32_t* rowptr, const int32_t* colidx, const float* vals_or_null, int64_t n,
                    float* dinv, uint8_t* iso, float* x0_logdeg, float* w_out_or_null,
                    float* rowsum_out, float* diag_ws, double* colsum_ws, int32_t* unsorted_flag_or_null,
                    egnn_stream_t stream) {
    EGNN_REQUIRE(rowptr && dinv && iso && rowsum_out && diag_ws && colsum_ws, "null pointer");
    EGNN_REQUIRE(n >= 0, "bad shape");
    if (n == 0) return EGNN_OK;
    cudaStream_t st = (cudaStream_t)stream;
    int rc = check_cuda(cudaMemsetAsync(colsum_ws, 0, sizeof(double) * n, st), "memset colsum");
    if (rc) return rc;
    if (unsorted_flag_or_null) {
        rc = check_cuda(cudaMemsetAsync(unsorted_flag_or_null, 0, sizeof(int32_t), st), "memset flag");
        if (rc) return rc;
    }
    rc = egnn_degree_rows(rowptr, colidx, vals_or_null, n, 0, n, rowsum_out, diag_ws, colsum_ws, unsorted_flag_or_null,
                          stream);
    if (rc) return rc;
    return egnn_graph_prep_finish(colsum_ws, diag_ws, rowsum_out, n, dinv, iso, x0_logdeg, w_out_or_null, stream);
}

int egnn_patch_degrees(const float* w_base, const float* rowsum_base, const float* dinv_base,
                       const uint8_t* iso_base, const float* x0_base, int64_t n,
                       const int32_t* delta_row_host, const int32_t* delta_col_host,
                       const float* delta_val_host, int32_t n_delta, float* dinv_out, uint8_t* iso_out,
                       float* x0_out, int64_t row_begin, int64_t n_rows, egnn_stream_t stream) {
    EGNN_REQUIRE(w_base && dinv_base && iso_base && dinv_out && iso_out, "null pointer");
    EGNN_REQUIRE(row_begin >= 0 && n_rows >= 0 && row_begin + n_rows <= n, "bad row range");
    EGNN_REQUIRE(n_rows == 0 || (rowsum_base && x0_base && x0_out), "null pointer");
    DeltaList d;
    int rc = fill_delta(d, delta_row_host, delta_col_host, delta_val_host, n_delta, n);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    rc = check_cuda(cudaMemcpyAsync(dinv_out, dinv_base, sizeof(float) * n, cudaMemcpyDeviceToDevice, st), "copy dinv");
    if (rc) return rc;
    rc = check_cuda(cudaMemcpyAsync(iso_out, iso_base, sizeof(uint8_t) * n, cudaMemcpyDeviceToDevice, st), "copy iso");
    if (rc) return rc;
    if (n_rows > 0) {
        rc = check_cuda(cudaMemcpyAsync(x0_out, x0_base, sizeof(float) * n_rows, cudaMemcpyDeviceToDevice, st), "copy x0");
        if (rc) return rc;
    }
    if (n_delta > 0) {
        patch_degrees_kernel<<<1, EGNN_MAX_DELTA, 0, st>>>(w_base, rowsum_base, d, dinv_out, iso_out, x0_out, row_begin, n_rows);
        EGNN_LAUNCH_CHECK("patch_degrees_kernel launch");
    }
    return EGNN_OK;
}

int egnn_patch_nodes(const float* w_base, const float* rowsum_base, const float* dinv_base, const uint8_t* iso_base,
                     const float* x0_base, const float* y0_base, int64_t n, const int32_t* delta_row_host,
                     const int32_t* delta_col_host, const float* delta_val_host, int32_t n_delta, float* dinv_io,
                     uint8_t* iso_io, float* x0_io, float* y0_io, int32_t restore, egnn_stream_t stream) {
    EGNN_REQUIRE(w_base && rowsum_base && dinv_base && iso_base && x0_base && y0_base && dinv_io && iso_io && x0_io && y0_io,
                 "null pointer");
    DeltaList d;
    int rc = fill_delta(d, delta_row_host, delta_col_host, delta_val_host, n_delta, n);
    if (rc) return rc;
    if (n_delta == 0) return EGNN_OK;
    patch_nodes_kernel<<<1, 2 * EGNN_MAX_DELTA, 0, (cudaStream_t)stream>>>(w_base, rowsum_base, dinv_base, iso_base, x0_base,
                                                                          y0_base, d, dinv_io, iso_io, x0_io, y0_io,
                                                                          restore ? 1 : 0);
    EGNN_LAUNCH_CHECK("patch_nodes_kernel launch");
    return EGNN_OK;
}

static size_t row_order_cub_bytes(int64_t n) {
    size_t b = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, b, (uint32_t*)nullptr, (uint32_t*)nullptr, (int32_t*)nullptr,
                                    (int32_t*)nullptr, (int)n);
    return b + 256;
}

size_t egnn_row_order_ws_bytes(int64_t n) {
    if (n < 1) return 256;
    return 3 * align_up(4 * (size_t)n, 256) + row_order_cub_bytes(n) + 256;
}

int egnn_row_order(const int32_t* rowptr, int64_t n, int32_t* order_out, void* workspace, size_t workspace_bytes,
                   egnn_stream_t stream) {
    EGNN_REQUIRE(rowptr && order_out, "null pointer");
    EGNN_REQUIRE(n >= 0 && n < (int64_t(1) << 31), "bad shape");
    cudaStream_t st = (cudaStream_t)stream;
    if (n == 0) return check_cuda(cudaMemsetAsync(order_out, 0, sizeof(int32_t), st), "memset n_hub");
    int rc = require_workspace(workspace, workspace_bytes, egnn_row_order_ws_bytes(n), "row-order workspace");
    if (rc) return rc;
    const size_t arr = align_up(4 * (size_t)n, 256);
    char* ws = (char*)align_up((size_t)workspace, 256);
    uint32_t* keys = (uint32_t*)ws;
    uint32_t* keys_sorted = (uint32_t*)(ws + arr);
    int32_t* ids = (int32_t*)(ws + 2 * arr);
    void* cub_temp = ws + 3 * arr;
    size_t cub_bytes = row_order_cub_bytes(n);
    row_order_keys_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, st>>>(rowptr, (int)n, keys, ids);
    EGNN_LAUNCH_CHECK("row_order_keys_kernel launch");
    rc = check_cuda(cub::DeviceRadixSort::SortPairs(cub_temp, cub_bytes, keys, keys_sorted, ids, order_out, (int)n, 0, 32,
                                                    st), "sort rows by degree");
    if (rc) return rc;
    row_order_hubs_kernel<<<1, 32, 0, st>>>(keys_sorted, (int)n, order_out + n);
    EGNN_LAUNCH_CHECK("row_order_hubs_kernel launch");
    return EGNN_OK;
}

}  // extern "C"

// ---- the wavelet pass: one static function per path of egnn_cheb_wavelet -------------------------
// Where order `order` of the forward writes T_k: its slab of t_all; nowhere on the last order (T_K
// is never read again); else the two T slabs for orders 1 and 2, and in place over T_{k-2} after.
static float* t_slot(const ChebArgs& c, const ChebWs& ws, float* t_all, int order, const float* t_prev2) {
    if (t_all) return slab_of(t_all, (size_t)c.rows * (size_t)c.f, order);
    if (order == c.k) return nullptr;
    if (order <= 2) return ws.t[order - 1];
    return const_cast<float*>(t_prev2);
}

static int wavelet_order0(const ChebArgs& c, const float* x0, float* out, float* t_all, int32_t normalize_l1) {
    const size_t slab_elems = (size_t)c.rows * (size_t)c.f;
    OrderParams p{};
    p.delta = c.delta;
    order_coefs(p.c_prev, c.coeffs, 0, c.S, 0);
    order0_kernel<<<grid_for((int64_t)slab_elems * c.S, 256), 256, 0, c.st>>>(x0, out, c.rows, c.f, c.S, p);
    EGNN_LAUNCH_CHECK("order0_kernel launch");
    if (t_all) {
        int rc = check_cuda(cudaMemcpyAsync(t_all, x0, sizeof(float) * slab_elems, cudaMemcpyDeviceToDevice, c.st), "copy T0");
        if (rc) return rc;
    }
    return normalize_l1 ? launch_l1_normalize(out, c.rows, c.S, c.f, c.st) : EGNN_OK;
}

// All K orders in one persistent launch (sell_step.cuh); the first operand dinv (.) T_0 is computed
// inside it unless the caller keeps it (y0: fixed per graph for the default signal).
static int wavelet_sell(const ChebArgs& c, const ChebWs& ws, const egnn_sell_plan* plan, const float* x0,
                        const float* y0, float* out, float* t_all, int32_t normalize_l1, const float* w_base,
                        const float* rowsum_base, int32_t default_signal) {
    EGNN_REQUIRE(c.f == 1 && c.vals == nullptr, "the SELL plan serves F = 1 on a binary adjacency");
    EGNN_REQUIRE(plan->n == c.rows && plan->n_cols == c.rows && plan->row0 == 0 && plan->vpart && plan->slice_off && plan->blk_slice_ptr &&
                 plan->rv_ptr && plan->vslot && plan->cta_info && plan->hub && plan->sched, "SELL plan does not match the graph or is not filled");
    SellStepParams sp{};
    step_fill_plan(sp, plan);
    sp.delta = c.delta;
    sp.w_base = w_base; sp.rowsum_base = rowsum_base; sp.patch_x0 = default_signal ? 1 : 0;
    sp.dinv = c.dinv; sp.iso = c.iso; sp.x0 = x0;
    sp.operand_first = y0;
    sp.operand[0] = ws.y[0]; sp.operand[1] = ws.y[1];
    sp.ydst[0][0] = ws.y[0]; sp.ydst[1][0] = ws.y[1]; sp.n_dst = 1;
    sp.tbuf[0] = ws.t[0]; sp.tbuf[1] = ws.t[1]; sp.t_all = t_all; sp.out = out;
    sp.normalize = normalize_l1; sp.a = c.a; sp.b = c.b;
    sp.world = 1; sp.rank = 0; sp.rows_per = c.rows;
    int rc = record_event(c.events, 0, c.st);
    if (rc) return rc;
    rc = run_sell_step(sp, c.k, c.S, c.coeffs, false, c.st);
    if (rc) return rc;
    for (int e = 1; e < 2 * c.k; ++e) {           // one launch: events 0 and 1 bracket the whole step, the rest follow it
        rc = record_event(c.events, e, c.st);
        if (rc) return rc;
    }
    return EGNN_OK;
}

// First use of a large graph at F = 1 (no SELL plan yet): plan-free column-blocked kernel (blocked.cuh)
static int wavelet_blocked(const ChebArgs& c, const ChebWs& ws, const float* x0, float* out, float* t_all,
                           int32_t normalize_l1) {
    const int64_t n = c.rows;
    const int C = ws.C, CB = ws.CB;
    int rc = check_cuda(cudaMemsetAsync(ws.blk_counters, 0, sizeof(unsigned) * (size_t)c.k * (size_t)C, c.st),
                        "memset batch counters");
    if (rc) return rc;
    blocked_bounds_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, c.st>>>(c.rowptr, c.colidx, (int)n, C, CB, ws.seg);
    EGNN_LAUNCH_CHECK("blocked_bounds_kernel launch");
    const size_t smem = sizeof(float) * (size_t)CB;
    const void* fn = c.vals ? (const void*)blocked_spmv_kernel<true> : (const void*)blocked_spmv_kernel<false>;
    rc = check_cuda(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                    "cudaFuncSetAttribute(blocked_spmv_kernel)");
    if (rc) return rc;
    BlockedParams bp{};
    bp.colidx = c.colidx; bp.vals = c.vals; bp.seg = ws.seg; bp.part = ws.part;
    bp.n = (int32_t)n; bp.C = C; bp.CB = CB; bp.n_cta = device_sm_count();
    if (bp.n_cta < C) bp.n_cta = C;
    BlockedEpilogueParams ep{};
    ep.delta = c.delta;
    ep.part = ws.part; ep.dinv = c.dinv; ep.iso = c.iso; ep.out = out; ep.n = (int32_t)n; ep.C = C; ep.S = c.S;
    ep.a = c.a; ep.b = c.b;
    const float* t_prev = x0;
    const float* t_prev2 = nullptr;
    for (int order = 1; order <= c.k; ++order) {
        const bool last = order == c.k;
        float* t_out = t_slot(c, ws, t_all, order, t_prev2);
        rc = record_event(c.events, 2 * (order - 1), c.st);
        if (rc) return rc;
        bp.y = ws.y[(order - 1) & 1];
        bp.counter = ws.blk_counters + (size_t)(order - 1) * C;
        if (c.vals) blocked_spmv_kernel<true><<<bp.n_cta, kBlockedThreads, smem, c.st>>>(bp);
        else blocked_spmv_kernel<false><<<bp.n_cta, kBlockedThreads, smem, c.st>>>(bp);
        EGNN_LAUNCH_CHECK("blocked_spmv_kernel launch");
        ep.y_prev = bp.y; ep.tprev = t_prev; ep.tprev2 = t_prev2; ep.tk = t_out;
        ep.y_out = last ? nullptr : ws.y[order & 1];
        ep.first = order == 1; ep.normalize = last && normalize_l1;
        order_coefs(ep.c_prev, c.coeffs, c.k, c.S, order - 1);
        order_coefs(ep.c_k, c.coeffs, c.k, c.S, order);
        blocked_epilogue_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, c.st>>>(ep);
        EGNN_LAUNCH_CHECK("blocked_epilogue_kernel launch");
        rc = record_event(c.events, 2 * (order - 1) + 1, c.st);
        if (rc) return rc;
        t_prev2 = t_prev;
        t_prev = t_out;
    }
    return EGNN_OK;
}

static int wavelet_wide(const ChebArgs& c, const ChebWs& ws, const float* x0, float* out, float* t_all,
                        int32_t normalize_l1) {
    const int64_t n = c.rows;
    const int ldy = wide_ldy(c.f);
    const RingConfig rcfg = ring_config(ldy);
    WideParams wp = wide_params(c);
    wp.out = out;
    // ws.y[] hold dinv (.) T_k, rows padded to 16 bytes
    prescale_pad_kernel<<<grid_for(n * ldy, 256), 256, 0, c.st>>>(x0, c.dinv, ws.y[0], n, c.f, ldy, 0);
    EGNN_LAUNCH_CHECK("prescale_pad_kernel launch");
    int rc = check_cuda(cudaMemsetAsync(ws.row_counters, 0, sizeof(unsigned) * (size_t)c.k * (size_t)rcfg.grid_y, c.st),
                        "memset row counters");
    if (rc) return rc;
    const bool fuse_norm = normalize_l1 && rcfg.grid_y == 1;
    // dynamic rows pay off where rows are short and one feature tile covers the signal (arxiv
    // shape F = 128: 0.283 -> 0.23 ms per order); measured slower on long rows (Reddit shape
    // F = 64: 2.13 -> 2.48) and on many feature tiles (Physics F = 8415: 2.77 -> 3.3)
    const bool dynamic_rows = rcfg.grid_y == 1 && c.nnz < (int64_t)kWideDynamicMaxDegree * n;
    const int sms = device_sm_count();
    for (int order = 1; order <= c.k; ++order) {
        const bool last = order == c.k;
        wp.first = order == 1;
        wp.normalize = last && fuse_norm;
        wp.row_counter = dynamic_rows ? ws.row_counters + (size_t)(order - 1) * (size_t)rcfg.grid_y : nullptr;
        wp.ysrc = ws.y[(order - 1) & 1];
        wp.x0_own = order == 1 ? x0 : nullptr;
        wp.y2_own = order == 1 ? nullptr : ws.y[order & 1];
        wp.y_out = last ? nullptr : ws.y[order & 1];      // in place over dinv (.) T_{k-2} (own row only)
        wp.tk_out = slab_of(t_all, (size_t)n * (size_t)c.f, order);
        order_coefs(wp.c_prev, c.coeffs, c.k, c.S, order - 1);
        order_coefs(wp.c_k, c.coeffs, c.k, c.S, order);
        rc = record_event(c.events, 2 * (order - 1), c.st);
        if (rc) return rc;
        rc = launch_wide(wp, rcfg, sms, c.st);
        if (rc) return rc;
        rc = record_event(c.events, 2 * (order - 1) + 1, c.st);
        if (rc) return rc;
    }
    return normalize_l1 && !fuse_norm ? launch_l1_normalize(out, n, c.S, c.f, c.st) : EGNN_OK;
}

static int wavelet_generic(const ChebArgs& c, const ChebWs& ws, const OrderConfig& cfg, const float* x0, float* out,
                           float* t_all, int32_t normalize_l1) {
    OrderParams p = order_params(c, cfg);
    p.out = out;
    const bool fuse_norm = normalize_l1 && cfg.grid_y == 1;
    const float* t_prev = x0;         // T_{k-1}
    const float* t_prev2 = nullptr;   // T_{k-2}
    for (int order = 1; order <= c.k; ++order) {
        const bool last = order == c.k;
        float* t_out = t_slot(c, ws, t_all, order, t_prev2);
        p.first = order == 1;
        p.normalize = last && fuse_norm;
        p.tprev_own = t_prev;
        p.tprev2_own = t_prev2;
        p.tk_own = t_out;
        p.gsrc = cfg.prescaled ? ws.y[(order - 1) & 1] : t_prev;
        p.y_own = (cfg.prescaled && !last) ? ws.y[order & 1] : nullptr;
        order_coefs(p.c_prev, c.coeffs, c.k, c.S, order - 1);
        order_coefs(p.c_k, c.coeffs, c.k, c.S, order);
        int rc = record_event(c.events, 2 * (order - 1), c.st);
        if (rc) return rc;
        rc = launch_order(p, cfg, c.st);
        if (rc) return rc;
        rc = record_event(c.events, 2 * (order - 1) + 1, c.st);
        if (rc) return rc;
        t_prev2 = t_prev;
        t_prev = t_out;
    }
    return normalize_l1 && !fuse_norm ? launch_l1_normalize(out, c.rows, c.S, c.f, c.st) : EGNN_OK;
}

extern "C" {

size_t egnn_cheb_workspace_bytes(int64_t n, int32_t f) {
    return cheb_ws_layout(nullptr, n, f).total_bytes;
}

int egnn_cheb_wavelet(const int32_t* rowptr, const int32_t* colidx, const float* vals_or_null,
                      const float* dinv, const uint8_t* iso, const float* x0, int64_t n, int64_t nnz,
                      int32_t f, int32_t k, int32_t n_scales, const float* coeffs_host, float op_scale, float op_shift,
                      float* out, float* t_all_or_null, int32_t normalize_l1,
                      const int32_t* delta_row_host, const int32_t* delta_col_host,
                      const float* delta_val_host, int32_t n_delta, void* workspace,
                      size_t workspace_bytes, egnn_stream_t stream, void* const* order_events_host,
                      const egnn_sell_plan* sell_plan, const int32_t* row_order_or_null,
                      const float* y0_or_null, int32_t rows_sorted,
                      const float* w_base_or_null, const float* rowsum_base_or_null, int32_t default_signal) {
    EGNN_REQUIRE(rowptr && dinv && iso && x0 && out && coeffs_host, "null pointer");
    EGNN_REQUIRE((w_base_or_null == nullptr) == (rowsum_base_or_null == nullptr), "w_base and rowsum_base come together");
    EGNN_REQUIRE(w_base_or_null == nullptr || n_delta == 0 || sell_plan, "in-kernel degree patches need the SELL plan path");
    EGNN_REQUIRE(nnz == 0 || colidx, "null colidx");
    EGNN_REQUIRE(n >= 0 && n < (int64_t(1) << 31) && nnz >= 0 && nnz < (int64_t(1) << 31), "n/nnz out of int32 range");
    EGNN_REQUIRE(f >= 1, "f must be >= 1");
    EGNN_REQUIRE(k >= 0 && k <= EGNN_MAX_ORDER, "k out of range");
    EGNN_REQUIRE(n_scales >= 1 && n_scales <= EGNN_MAX_SCALES, "n_scales out of range");
    EGNN_REQUIRE(vec_aligned(x0, f) && vec_aligned(out, f) && vec_aligned(t_all_or_null, f),
                 "x0, out and t_all must be 16-byte aligned when f % 4 == 0");
    if (n == 0) return EGNN_OK;
    ChebArgs c{};
    c.rowptr = rowptr; c.colidx = colidx; c.vals = vals_or_null; c.row_order = row_order_or_null;
    c.dinv = dinv; c.iso = iso; c.rows = n; c.nnz = nnz; c.f = f; c.k = k; c.S = n_scales;
    c.coeffs = coeffs_host; c.a = op_scale; c.b = op_shift; c.events = order_events_host; c.st = (cudaStream_t)stream;
    int rc = fill_delta(c.delta, delta_row_host, delta_col_host, delta_val_host, n_delta, n);
    if (rc) return rc;
    if (k == 0) return wavelet_order0(c, x0, out, t_all_or_null, normalize_l1);

    const OrderConfig cfg = choose_config(n, nnz, f);
    rc = require_workspace(workspace, workspace_bytes, egnn_cheb_workspace_bytes(n, f), "workspace");
    if (rc) return rc;
    const ChebWs ws = cheb_ws_layout(workspace, n, f);
    const size_t slab_elems = (size_t)n * (size_t)f;
    if (t_all_or_null) {
        rc = check_cuda(cudaMemcpyAsync(t_all_or_null, x0, sizeof(float) * slab_elems, cudaMemcpyDeviceToDevice, c.st), "copy T0");
        if (rc) return rc;
    }
    if (cfg.prescaled && !sell_plan) {
        prescale_kernel<<<grid_for((int64_t)slab_elems, 256), 256, 0, c.st>>>(x0, dinv, ws.y[0], n, f, 0);
        EGNN_LAUNCH_CHECK("prescale_kernel launch");
    }
    if (sell_plan)
        return wavelet_sell(c, ws, sell_plan, x0, y0_or_null, out, t_all_or_null, normalize_l1, w_base_or_null,
                            rowsum_base_or_null, default_signal);
    if (f == 1 && rows_sorted && (nnz >= kBlockedMinNnz || rows_sorted == 2) && nnz > 0)
        return wavelet_blocked(c, ws, x0, out, t_all_or_null, normalize_l1);
    if (f >= kWideMinF) return wavelet_wide(c, ws, x0, out, t_all_or_null, normalize_l1);
    return wavelet_generic(c, ws, cfg, x0, out, t_all_or_null, normalize_l1);
}

}  // extern "C"

// ---- backward of the wavelet pass (csrc/adjoint.cuh) ------------------------------------------------
// Application j = 1..K produces b_m, m = K - j (b_0 = the signal's gradient).  b_all: [K+1, n, f]
// receives Xbar (slab 0) and every Clenshaw vector b_m (slab m); the generic path then keeps its
// b vectors there instead of the workspace ping-pong slabs.
static int adjoint_wide(const ChebArgs& c, const ChebWs& ws, const float* cbar, const float* tbar, float* xbar,
                        float* b_all) {
    const int64_t n = c.rows;
    const int k = c.k;
    const size_t slab_elems = (size_t)n * (size_t)c.f;
    const int ldy = wide_ldy(c.f);
    const RingConfig rcfg = ring_config(ldy);
    int rc = check_cuda(cudaMemsetAsync(ws.row_counters, 0, sizeof(unsigned) * (size_t)k * (size_t)rcfg.grid_y, c.st),
                        "memset row counters");
    if (rc) return rc;
    // ws.y[] hold dinv (.) b, rows padded to 16 bytes
    adjoint_prologue_kernel<<<grid_for(n * ldy, 256), 256, 0, c.st>>>(
        cbar, slab_of(tbar, slab_elems, k), c.dinv, slab_of(b_all, slab_elems, k), ws.y[0], n, c.f, c.S, ldy,
        coef_row(c.coeffs, k, c.S, k));
    EGNN_LAUNCH_CHECK("adjoint_prologue_kernel launch");
    WideParams wp = wide_params(c);
    wp.cbar = cbar;
    const bool dynamic_rows = rcfg.grid_y == 1 && c.nnz < (int64_t)kWideDynamicMaxDegree * n;   // as the forward
    const int sms = device_sm_count();
    for (int j = 1; j <= k; ++j) {
        const int m = k - j;
        wp.row_counter = dynamic_rows ? ws.row_counters + (size_t)(j - 1) * (size_t)rcfg.grid_y : nullptr;
        wp.ysrc = ws.y[(j - 1) & 1];
        wp.y2_own = j == 1 ? nullptr : ws.y[j & 1];
        wp.y_out = m == 0 ? nullptr : ws.y[j & 1];           // in place over dinv (.) b_{m+2} (own row only)
        wp.tk_out = m == 0 ? xbar : slab_of(b_all, slab_elems, m);
        wp.tbar = slab_of(tbar, slab_elems, m);
        wp.c_adj = m == 0 ? 1.f : 2.f;
        order_coefs(wp.c_k, c.coeffs, k, c.S, m);
        rc = record_event(c.events, 2 * (j - 1), c.st);
        if (rc) return rc;
        rc = launch_wide<true>(wp, rcfg, sms, c.st);
        if (rc) return rc;
        rc = record_event(c.events, 2 * (j - 1) + 1, c.st);
        if (rc) return rc;
    }
    return EGNN_OK;
}

static int adjoint_generic(const ChebArgs& c, const ChebWs& ws, const float* cbar, const float* tbar, float* xbar,
                           float* b_all) {
    const int64_t n = c.rows;
    const int k = c.k;
    const size_t slab_elems = (size_t)n * (size_t)c.f;
    const OrderConfig cfg = choose_config(n, c.nnz, c.f);
    // b_m of application j: ws.t[j & 1] (in place over b_{m+2}), or slab m of b_all
    auto b_vec = [&](int j) { return b_all ? slab_of(b_all, slab_elems, k - j) : ws.t[j & 1]; };
    adjoint_prologue_kernel<<<grid_for((int64_t)slab_elems, 256), 256, 0, c.st>>>(
        cbar, slab_of(tbar, slab_elems, k), c.dinv, b_vec(0), cfg.prescaled ? ws.y[0] : nullptr, n, c.f, c.S, c.f,
        coef_row(c.coeffs, k, c.S, k));
    EGNN_LAUNCH_CHECK("adjoint_prologue_kernel launch");
    OrderParams p = order_params(c, cfg);
    p.cbar = cbar;
    for (int j = 1; j <= k; ++j) {
        const int m = k - j;
        p.tprev_own = b_vec(j - 1);
        p.tprev2_own = j == 1 ? nullptr : b_vec(j - 2);
        p.tk_own = m == 0 ? xbar : b_vec(j);
        p.gsrc = cfg.prescaled ? ws.y[(j - 1) & 1] : b_vec(j - 1);
        p.y_own = (cfg.prescaled && m > 0) ? ws.y[j & 1] : nullptr;
        p.tbar = slab_of(tbar, slab_elems, m);
        p.c_adj = m == 0 ? 1.f : 2.f;
        order_coefs(p.c_k, c.coeffs, k, c.S, m);
        int rc = record_event(c.events, 2 * (j - 1), c.st);
        if (rc) return rc;
        rc = launch_order<true>(p, cfg, c.st);
        if (rc) return rc;
        rc = record_event(c.events, 2 * (j - 1) + 1, c.st);
        if (rc) return rc;
    }
    return EGNN_OK;
}

static int cheb_adjoint_impl(const int32_t* rowptr_t, const int32_t* colidx_t, const float* vals_t_or_null,
                             const float* dinv, const uint8_t* iso, int64_t n, int64_t nnz, int32_t f, int32_t k,
                             int32_t n_scales, const float* coeffs_host, float op_scale, float op_shift,
                             const float* cbar, const float* tbar_or_null, float* xbar,
                             const int32_t* delta_row_host, const int32_t* delta_col_host,
                             const float* delta_val_host, int32_t n_delta, void* workspace,
                             size_t workspace_bytes, egnn_stream_t stream, void* const* app_events_host,
                             const int32_t* row_order_or_null, float* b_all_or_null) {
    EGNN_REQUIRE(rowptr_t && dinv && iso && cbar && xbar && coeffs_host, "null pointer");
    EGNN_REQUIRE(nnz == 0 || colidx_t, "null colidx");
    EGNN_REQUIRE(n >= 0 && n < (int64_t(1) << 31) && nnz >= 0 && nnz < (int64_t(1) << 31), "n/nnz out of int32 range");
    EGNN_REQUIRE(f >= 1, "f must be >= 1");
    EGNN_REQUIRE(k >= 0 && k <= EGNN_MAX_ORDER, "k out of range");
    EGNN_REQUIRE(n_scales >= 1 && n_scales <= EGNN_MAX_SCALES, "n_scales out of range");
    EGNN_REQUIRE(vec_aligned(cbar, f) && vec_aligned(tbar_or_null, f) && vec_aligned(xbar, f) &&
                 vec_aligned(b_all_or_null, f), "cbar, tbar, xbar and b_all must be 16-byte aligned when f % 4 == 0");
    if (n == 0) return EGNN_OK;
    ChebArgs c{};
    c.rowptr = rowptr_t; c.colidx = colidx_t; c.vals = vals_t_or_null; c.row_order = row_order_or_null;
    c.dinv = dinv; c.iso = iso; c.rows = n; c.nnz = nnz; c.f = f; c.k = k; c.S = n_scales;
    c.coeffs = coeffs_host; c.a = op_scale; c.b = op_shift; c.events = app_events_host; c.st = (cudaStream_t)stream;
    int rc = fill_delta(c.delta, delta_row_host, delta_col_host, delta_val_host, n_delta, n);
    if (rc) return rc;
    const size_t slab_elems = (size_t)n * (size_t)f;
    if (k == 0) {
        adjoint_prologue_kernel<<<grid_for((int64_t)slab_elems, 256), 256, 0, c.st>>>(
            cbar, tbar_or_null, dinv, xbar, nullptr, n, f, n_scales, f, coef_row(coeffs_host, 0, n_scales, 0));
        EGNN_LAUNCH_CHECK("adjoint_prologue_kernel launch");
    } else {
        rc = require_workspace(workspace, workspace_bytes, egnn_cheb_workspace_bytes(n, f), "workspace");
        if (rc) return rc;
        const ChebWs ws = cheb_ws_layout(workspace, n, f);
        rc = f >= kWideMinF ? adjoint_wide(c, ws, cbar, tbar_or_null, xbar, b_all_or_null)
                            : adjoint_generic(c, ws, cbar, tbar_or_null, xbar, b_all_or_null);
        if (rc) return rc;
    }
    return b_all_or_null ? check_cuda(cudaMemcpyAsync(b_all_or_null, xbar, sizeof(float) * slab_elems,
                                                      cudaMemcpyDeviceToDevice, c.st), "copy Xbar")
                         : EGNN_OK;
}

// ---- one order (adjoint application) of a row shard ----------------------------------------------
// Generic kernel, split over the rank's local and remote columns: phase 0 sums the local columns
// into p.acc_ws, phase 1 adds the remote columns from the gathered operand and runs the epilogue,
// phase 2 is one launch over the unsplit rows.  The edge flips ride with the launch that gathers
// from the exchanged operand, so phase 0 does not look at them.  p comes filled for the local CSR.
// Weighted shards: p.vals holds the local half's (or the unsplit rows') values, vals_remote the remote half's.
template <bool ADJ>
static int order_sharded_phase(OrderParams& p, const OrderConfig& cfg, int32_t phase, const int32_t* rowptr_remote,
                               const int32_t* colidx_remote, const float* vals_remote, const float* gathered,
                               const char* gathered_missing, const int32_t* delta_row_host,
                               const int32_t* delta_col_host, const float* delta_val_host, int32_t n_delta, int64_t n,
                               cudaStream_t st) {
    if (phase == 0) {                 // local columns: gathers hit the rank's own slab
        EGNN_REQUIRE(p.rowptr && p.acc_ws, "local half missing");
        p.gsrc = p.tprev_own - p.row0 * (int64_t)p.F;      // indexed by global column, only own rows touched
        p.mode = 1;
        p.normalize = 0;
        return launch_order<ADJ>(p, cfg, st);
    }
    int rc = fill_delta(p.delta, delta_row_host, delta_col_host, delta_val_host, n_delta, n);
    if (rc) return rc;
    EGNN_REQUIRE(gathered != nullptr, gathered_missing);
    p.gsrc = gathered;
    if (phase == 1) {                 // remote columns + epilogue
        EGNN_REQUIRE(rowptr_remote && p.acc_ws, "remote half missing");
        p.rowptr = rowptr_remote; p.colidx = colidx_remote; p.vals = vals_remote; p.mode = 2;
    } else {                          // one launch over the unsplit rows
        EGNN_REQUIRE(p.rowptr != nullptr, "csr missing");
    }
    return launch_order<ADJ>(p, cfg, st);
}

// Wide kernel with the exchange fused: order (application) `step` reads buffer (step - 1) & 1 of
// the own window - the full operand, global rows - and, unless it is the last, stores the next
// operand into buffer step & 1 of every rank's window (a plain store into the own rows at world 1).
template <bool ADJ>
static int wide_sharded_step(WideParams& wp, const RingConfig& rcfg, const egnn_peer_window* win, int step, bool last,
                             cudaStream_t st) {
    wp.ysrc = peer_operand(win, win->rank, (step - 1) & 1);
    float* own_next = peer_operand(win, win->rank, step & 1) + wp.row0 * (int64_t)wp.ldy;
    wp.y2_own = step == 1 ? nullptr : own_next;                  // dinv (.) T_{k-2} (b_{m+2}) of the own rows
    wp.y_out = (!last && win->world == 1) ? own_next : nullptr;
    fill_peer_push(wp.peer, win, step & 1, !last, false);
    return launch_wide<ADJ>(wp, rcfg, device_sm_count(), st);
}

extern "C" {

int egnn_cheb_adjoint(const int32_t* rowptr_t, const int32_t* colidx_t, const float* vals_t_or_null,
                      const float* dinv, const uint8_t* iso, int64_t n, int64_t nnz, int32_t f, int32_t k,
                      int32_t n_scales, const float* coeffs_host, float op_scale, float op_shift,
                      const float* cbar, const float* tbar_or_null, float* xbar,
                      const int32_t* delta_row_host, const int32_t* delta_col_host,
                      const float* delta_val_host, int32_t n_delta, void* workspace,
                      size_t workspace_bytes, egnn_stream_t stream, void* const* app_events_host,
                      const int32_t* row_order_or_null) {
    return cheb_adjoint_impl(rowptr_t, colidx_t, vals_t_or_null, dinv, iso, n, nnz, f, k, n_scales, coeffs_host,
                             op_scale, op_shift, cbar, tbar_or_null, xbar, delta_row_host, delta_col_host,
                             delta_val_host, n_delta, workspace, workspace_bytes, stream, app_events_host,
                             row_order_or_null, nullptr);
}

int egnn_cheb_adjoint_all(const int32_t* rowptr_t, const int32_t* colidx_t, const float* vals_t_or_null,
                          const float* dinv, const uint8_t* iso, int64_t n, int64_t nnz, int32_t f, int32_t k,
                          int32_t n_scales, const float* coeffs_host, float op_scale, float op_shift,
                          const float* cbar, const float* tbar_or_null, float* xbar,
                          const int32_t* delta_row_host, const int32_t* delta_col_host,
                          const float* delta_val_host, int32_t n_delta, void* workspace,
                          size_t workspace_bytes, egnn_stream_t stream, void* const* app_events_host,
                          const int32_t* row_order_or_null, float* b_all) {
    EGNN_REQUIRE(b_all, "null b_all");
    return cheb_adjoint_impl(rowptr_t, colidx_t, vals_t_or_null, dinv, iso, n, nnz, f, k, n_scales, coeffs_host,
                             op_scale, op_shift, cbar, tbar_or_null, xbar, delta_row_host, delta_col_host,
                             delta_val_host, n_delta, workspace, workspace_bytes, stream, app_events_host,
                             row_order_or_null, b_all);
}

int egnn_l1_normalize(const float* c, float* h, int64_t n_vec, int32_t f, egnn_stream_t stream) {
    EGNN_REQUIRE(c && h, "null pointer");
    EGNN_REQUIRE(n_vec >= 0 && f >= 1, "bad shape");
    if (n_vec == 0) return EGNN_OK;
    l1_normalize_out_kernel<<<grid_for(n_vec * 32, 256), 256, 0, (cudaStream_t)stream>>>(c, h, n_vec, f);
    EGNN_LAUNCH_CHECK("l1_normalize_out_kernel launch");
    return EGNN_OK;
}

int egnn_l1_normalize_backward(const float* c, const float* hbar, const float* cbar_in_or_null, float* cbar_out,
                               int64_t n_vec, int32_t f, egnn_stream_t stream) {
    EGNN_REQUIRE(c && hbar && cbar_out, "null pointer");
    EGNN_REQUIRE(n_vec >= 0 && f >= 1, "bad shape");
    if (n_vec == 0) return EGNN_OK;
    l1_normalize_backward_kernel<<<grid_for(n_vec * 32, 256), 256, 0, (cudaStream_t)stream>>>(
        c, hbar, cbar_in_or_null, cbar_out, n_vec, f);
    EGNN_LAUNCH_CHECK("l1_normalize_backward_kernel launch");
    return EGNN_OK;
}

size_t egnn_cheb_coeff_grad_ws_bytes(int32_t k, int32_t n_scales) {
    const int64_t q = (int64_t)(k > 0 ? k + 1 : 1) * (n_scales > 0 ? n_scales : 1);
    return align_up(sizeof(double) * (size_t)kCoefGradBlocks * (size_t)q, 256) + 256;
}

int egnn_cheb_coeff_grad(const float* cbar, const float* t_all, int64_t n, int32_t f, int32_t k, int32_t n_scales,
                         double* grad_out, void* workspace, size_t workspace_bytes, egnn_stream_t stream) {
    EGNN_REQUIRE(cbar && t_all && grad_out, "null pointer");
    EGNN_REQUIRE(n >= 0 && n < (int64_t(1) << 31) && f >= 1, "bad shape");
    EGNN_REQUIRE(k >= 0 && k <= EGNN_MAX_ORDER, "k out of range");
    EGNN_REQUIRE(n_scales >= 1 && n_scales <= EGNN_MAX_SCALES, "n_scales out of range");
    int rc = require_workspace(workspace, workspace_bytes, egnn_cheb_coeff_grad_ws_bytes(k, n_scales),
                               "coefficient-gradient workspace");
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    double* partial = (double*)align_up((size_t)workspace, 256);
    coeff_grad_partial_kernel<<<kCoefGradBlocks, kCoefGradThreads, 0, st>>>(cbar, t_all, n, f, k, n_scales, partial);
    EGNN_LAUNCH_CHECK("coeff_grad_partial_kernel launch");
    const int n_out = n_scales * (k + 1);
    coeff_grad_finish_kernel<<<(unsigned)ceil_div64(n_out, 128), 128, 0, st>>>(partial, kCoefGradBlocks, n_out, grad_out);
    EGNN_LAUNCH_CHECK("coeff_grad_finish_kernel launch");
    return EGNN_OK;
}

static size_t transpose_cub_bytes(int64_t n, int64_t nnz) {
    size_t a = 0, b = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, a, (const uint32_t*)nullptr, (uint32_t*)nullptr, (const int32_t*)nullptr,
                                    (int32_t*)nullptr, (int)nnz);
    cub::DeviceScan::ExclusiveSum(nullptr, b, (int32_t*)nullptr, (int32_t*)nullptr, (int)(n + 1));
    return (a > b ? a : b) + 256;
}

size_t egnn_csr_transpose_ws_bytes(int64_t n, int64_t nnz) {
    if (n < 0 || nnz < 0) return 256;
    return 3 * align_up(4 * (size_t)(nnz > 0 ? nnz : 1), 256) + align_up(4 * (size_t)(n + 1), 256) +
           transpose_cub_bytes(n, nnz) + 256;
}

int egnn_csr_transpose(const int32_t* rowptr, const int32_t* colidx, const float* vals_or_null, int64_t n,
                       int64_t nnz, int32_t* rowptr_t, int32_t* colidx_t, float* vals_t_or_null, void* workspace,
                       size_t workspace_bytes, egnn_stream_t stream) {
    EGNN_REQUIRE(rowptr && rowptr_t, "null pointer");
    EGNN_REQUIRE(nnz == 0 || (colidx && colidx_t), "null colidx");
    EGNN_REQUIRE((vals_or_null == nullptr) == (vals_t_or_null == nullptr), "vals and vals_t come together");
    EGNN_REQUIRE(n >= 0 && n < (int64_t(1) << 31) && nnz >= 0 && nnz < (int64_t(1) << 31), "n/nnz out of int32 range");
    int rc = require_workspace(workspace, workspace_bytes, egnn_csr_transpose_ws_bytes(n, nnz), "transpose workspace");
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t arr = align_up(4 * (size_t)(nnz > 0 ? nnz : 1), 256);
    char* ws = (char*)align_up((size_t)workspace, 256);
    uint32_t* keys_sorted = (uint32_t*)ws;
    int32_t* ids = (int32_t*)(ws + arr);
    int32_t* ids_sorted = (int32_t*)(ws + 2 * arr);
    int32_t* counts = (int32_t*)(ws + 3 * arr);
    void* cub_temp = ws + 3 * arr + align_up(4 * (size_t)(n + 1), 256);
    size_t cub_bytes = transpose_cub_bytes(n, nnz);
    rc = check_cuda(cudaMemsetAsync(counts, 0, sizeof(int32_t) * (size_t)(n + 1), st), "memset column counts");
    if (rc) return rc;
    if (nnz > 0) {
        transpose_count_kernel<<<grid_for(nnz, 256), 256, 0, st>>>(colidx, nnz, ids, counts);
        EGNN_LAUNCH_CHECK("transpose_count_kernel launch");
        // stable: entries of one column keep their CSR (row-major) order, so the rows come out sorted
        const int end_bit = pow2_ceil_log2(n > 1 ? n : 2);
        rc = check_cuda(cub::DeviceRadixSort::SortPairs(cub_temp, cub_bytes, (const uint32_t*)colidx, keys_sorted, ids,
                                                        ids_sorted, (int)nnz, 0, end_bit, st), "sort entries by column");
        if (rc) return rc;
        transpose_fill_kernel<<<grid_for(nnz, 256), 256, 0, st>>>(rowptr, n, vals_or_null, ids_sorted, nnz, colidx_t,
                                                                 vals_t_or_null);
        EGNN_LAUNCH_CHECK("transpose_fill_kernel launch");
    }
    return check_cuda(cub::DeviceScan::ExclusiveSum(cub_temp, cub_bytes, counts, rowptr_t, (int)(n + 1), st),
                      "scan column counts");
}

// ---- gradient w.r.t. the adjacency (csrc/structure_grad.cuh) ---------------------------------------
// lanes across the K*F products of one entry: the next power of two, at most a warp
static int stack_fl_log2(int32_t f, int32_t k) {
    const int64_t kf = (int64_t)f * k;
    const int l = pow2_ceil_log2(kf > 1 ? kf : 1);
    return l > 5 ? 5 : l;
}

size_t egnn_adj_grad_degree_ws_bytes(int64_t n) {
    return 2 * align_up(sizeof(double) * (size_t)(n > 0 ? n : 1), 256) + 256;
}

int egnn_adj_grad_degree(const int32_t* rowptr, const int32_t* colidx, const float* vals_or_null,
                         const int32_t* rowptr_t, const int32_t* colidx_t, const float* vals_t_or_null,
                         const float* dinv, const uint8_t* iso, int64_t n, int64_t nnz, int32_t f, int32_t k,
                         float op_scale, const float* lam, const float* t, const float* xbar_or_null,
                         const float* rowsum_or_null, float* gw, float* grho, void* workspace,
                         size_t workspace_bytes, egnn_stream_t stream) {
    return egnn_adj_grad_degree_flips(rowptr, colidx, vals_or_null, rowptr_t, colidx_t, vals_t_or_null, dinv, iso, n,
                                      nnz, f, k, op_scale, lam, t, xbar_or_null, rowsum_or_null, nullptr, nullptr,
                                      nullptr, 0, gw, grho, workspace, workspace_bytes, stream);
}

int egnn_adj_grad_degree_flips(const int32_t* rowptr, const int32_t* colidx, const float* vals_or_null,
                               const int32_t* rowptr_t, const int32_t* colidx_t, const float* vals_t_or_null,
                               const float* dinv, const uint8_t* iso, int64_t n, int64_t nnz, int32_t f,
                               int32_t k, float op_scale, const float* lam, const float* t,
                               const float* xbar_or_null, const float* rowsum_or_null,
                               const int32_t* delta_row_host, const int32_t* delta_col_host,
                               const float* delta_val_host, int32_t n_delta, float* gw, float* grho,
                               void* workspace, size_t workspace_bytes, egnn_stream_t stream) {
    DeltaList d;
    int rc = fill_delta(d, delta_row_host, delta_col_host, delta_val_host, n_delta, n);
    if (rc) return rc;
    EGNN_REQUIRE(rowptr && rowptr_t && dinv && iso && gw && grho, "null pointer");
    EGNN_REQUIRE(nnz == 0 || (colidx && colidx_t), "null colidx");
    EGNN_REQUIRE((vals_or_null == nullptr) == (vals_t_or_null == nullptr), "vals and vals_t come together");
    EGNN_REQUIRE(k == 0 || (lam && t), "null lambda / T stacks");
    EGNN_REQUIRE((xbar_or_null == nullptr) || rowsum_or_null, "xbar needs rowsum");
    EGNN_REQUIRE(n >= 0 && n < (int64_t(1) << 31) && nnz >= 0 && nnz < (int64_t(1) << 31), "n/nnz out of int32 range");
    EGNN_REQUIRE(f >= 1 && k >= 0 && k <= EGNN_MAX_ORDER, "bad f / k");
    rc = require_workspace(workspace, workspace_bytes, egnn_adj_grad_degree_ws_bytes(n),
                           "adjacency-gradient workspace");
    if (rc) return rc;
    if (n == 0) return EGNN_OK;
    cudaStream_t st = (cudaStream_t)stream;
    double* r = (double*)align_up((size_t)workspace, 256);
    double* q = (double*)((char*)r + align_up(sizeof(double) * (size_t)n, 256));
    const int fl = stack_fl_log2(f, k);
    const int blocks = grid_for(n * 32, 256);
    adj_grad_degree_kernel<<<blocks, 256, 0, st>>>(rowptr, colidx, vals_or_null, dinv, lam, t, n, f, k, fl, r);
    EGNN_LAUNCH_CHECK("adj_grad_degree_kernel launch");
    adj_grad_degree_kernel<<<blocks, 256, 0, st>>>(rowptr_t, colidx_t, vals_t_or_null, dinv, t, lam, n, f, k, fl, q);
    EGNN_LAUNCH_CHECK("adj_grad_degree_kernel launch");
    if (d.n > 0) {
        adj_grad_flip_terms_kernel<<<1, 32 * kFlipWarps, 0, st>>>(d, dinv, lam, t, n, f, k, fl, r, q);
        EGNN_LAUNCH_CHECK("adj_grad_flip_terms_kernel launch");
    }
    adj_grad_finish_kernel<<<grid_for(n, 256), 256, 0, st>>>(r, q, dinv, iso, xbar_or_null, rowsum_or_null, n,
                                                             op_scale, gw, grho);
    EGNN_LAUNCH_CHECK("adj_grad_finish_kernel launch");
    return EGNN_OK;
}

int egnn_adj_grad_pairs(const int32_t* rows, const int32_t* cols, int64_t n_pairs, const float* dinv,
                        const float* lam, const float* t, const float* gw, const float* grho, int64_t n, int32_t f,
                        int32_t k, float op_scale, float* out, egnn_stream_t stream) {
    EGNN_REQUIRE(n_pairs >= 0 && n >= 0 && n < (int64_t(1) << 31) && f >= 1 && k >= 0 && k <= EGNN_MAX_ORDER,
                 "bad shape");
    if (n_pairs == 0) return EGNN_OK;
    EGNN_REQUIRE(rows && cols && dinv && gw && grho && out, "null pointer");
    EGNN_REQUIRE(k == 0 || (lam && t), "null lambda / T stacks");
    const int fl = stack_fl_log2(f, k);
    adj_grad_pairs_kernel<<<grid_for(ceil_div64(n_pairs, 32 >> fl) * 32, 256), 256, 0, (cudaStream_t)stream>>>(
        rows, cols, n_pairs, dinv, lam, t, gw, grho, n, f, k, fl, op_scale, out);
    EGNN_LAUNCH_CHECK("adj_grad_pairs_kernel launch");
    return EGNN_OK;
}

int egnn_adj_grad_dense(const float* dinv, const float* lam, const float* t, const float* gw, const float* grho,
                        int64_t n, int32_t f, int32_t k, float op_scale, float* out, int64_t ld,
                        egnn_stream_t stream) {
    EGNN_REQUIRE(n >= 0 && n < (int64_t(1) << 31) && f >= 1 && k >= 0 && k <= EGNN_MAX_ORDER, "bad shape");
    EGNN_REQUIRE(ld >= n, "ld must be >= n");
    if (n == 0) return EGNN_OK;
    EGNN_REQUIRE(dinv && gw && grho && out, "null pointer");
    EGNN_REQUIRE(k == 0 || (lam && t), "null lambda / T stacks");
    const int64_t tiles = ceil_div64(n, kDenseTile);
    EGNN_REQUIRE(tiles <= 65535, "n too large for the dense gradient");
    const int vec_ok = (ld % 4 == 0) && ((uintptr_t)out & 15) == 0;
    adj_grad_dense_kernel<<<dim3((unsigned)tiles, (unsigned)tiles, 1), kDenseThreads, 0, (cudaStream_t)stream>>>(
        lam, t, dinv, gw, grho, n, f, k, op_scale, out, ld, vec_ok);
    EGNN_LAUNCH_CHECK("adj_grad_dense_kernel launch");
    return EGNN_OK;
}

}  // extern "C"

// One order of a row shard, binary (vals_local == vals_remote == NULL) or weighted (both given).
static int cheb_order_sharded_impl(const int32_t* rowptr_local, const int32_t* colidx_local, const float* vals_local,
                                   const int32_t* rowptr_remote, const int32_t* colidx_remote,
                                   const float* vals_remote, const float* dinv_full, const uint8_t* iso_full,
                                   const float* t_prev_full, const float* t_prev_local, const float* t_prev2_local,
                                   float* t_out_local, float* out_local, float* acc_ws, int64_t n, int64_t nnz_hint,
                                   int64_t row_begin, int64_t row_end, int32_t f, int32_t order, int32_t k_max,
                                   int32_t n_scales, const float* coeffs_host, float op_scale, float op_shift,
                                   int32_t normalize_l1, int32_t phase, const int32_t* delta_row_host,
                                   const int32_t* delta_col_host, const float* delta_val_host, int32_t n_delta,
                                   egnn_stream_t stream) {
    EGNN_REQUIRE(dinv_full && iso_full && out_local && coeffs_host && t_prev_local, "null pointer");
    EGNN_REQUIRE(row_begin >= 0 && row_end >= row_begin && row_end <= n, "bad row range");
    EGNN_REQUIRE(order >= 1 && order <= k_max && k_max <= EGNN_MAX_ORDER, "bad order");
    EGNN_REQUIRE(n_scales >= 1 && n_scales <= EGNN_MAX_SCALES, "n_scales out of range");
    EGNN_REQUIRE(phase >= 0 && phase <= 2, "bad phase");
    EGNN_REQUIRE(order == 1 || t_prev2_local, "T_{k-2} missing");
    EGNN_REQUIRE((vals_local == nullptr) == (vals_remote == nullptr), "values of the local and remote halves come together");
    const int64_t rows = row_end - row_begin;
    if (rows == 0) return EGNN_OK;
    cudaStream_t st = (cudaStream_t)stream;
    ChebArgs c{};
    c.rowptr = rowptr_local; c.colidx = colidx_local; c.vals = vals_local; c.dinv = dinv_full; c.iso = iso_full;
    c.rows = rows; c.row0 = row_begin; c.nnz = nnz_hint; c.f = f; c.k = k_max; c.S = n_scales;
    c.coeffs = coeffs_host; c.a = op_scale; c.b = op_shift; c.st = st;
    OrderConfig cfg = choose_config(rows, nnz_hint, f);
    cfg.prescaled = false;            // sharded slabs carry plain T_k (what the exchange moves)
    OrderParams p = order_params(c, cfg);
    p.tprev_own = t_prev_local; p.tprev2_own = t_prev2_local; p.tk_own = t_out_local;
    p.out = out_local; p.acc_ws = acc_ws; p.first = order == 1;
    order_coefs(p.c_prev, coeffs_host, k_max, n_scales, order - 1);
    order_coefs(p.c_k, coeffs_host, k_max, n_scales, order);
    const bool last = order == k_max;
    const bool fuse_norm = normalize_l1 && cfg.grid_y == 1;
    p.normalize = last && fuse_norm;
    int rc = order_sharded_phase<false>(p, cfg, phase, rowptr_remote, colidx_remote, vals_remote, t_prev_full,
                                        "gathered T_{k-1} missing", delta_row_host, delta_col_host, delta_val_host,
                                        n_delta, n, st);
    if (rc) return rc;
    if (phase != 0 && last && normalize_l1 && !fuse_norm) return launch_l1_normalize(out_local, rows, n_scales, f, st);
    return EGNN_OK;
}

extern "C" {

int egnn_cheb_order_sharded(const int32_t* rowptr_local, const int32_t* colidx_local,
                            const int32_t* rowptr_remote, const int32_t* colidx_remote,
                            const float* dinv_full, const uint8_t* iso_full, const float* t_prev_full,
                            const float* t_prev_local, const float* t_prev2_local, float* t_out_local,
                            float* out_local, float* acc_ws, int64_t n, int64_t nnz_hint,
                            int64_t row_begin, int64_t row_end, int32_t f, int32_t order, int32_t k_max,
                            int32_t n_scales, const float* coeffs_host, float op_scale, float op_shift,
                            int32_t normalize_l1, int32_t phase,
                            const int32_t* delta_row_host, const int32_t* delta_col_host,
                            const float* delta_val_host, int32_t n_delta, egnn_stream_t stream) {
    return cheb_order_sharded_impl(rowptr_local, colidx_local, nullptr, rowptr_remote, colidx_remote, nullptr,
                                   dinv_full, iso_full, t_prev_full, t_prev_local, t_prev2_local, t_out_local,
                                   out_local, acc_ws, n, nnz_hint, row_begin, row_end, f, order, k_max, n_scales,
                                   coeffs_host, op_scale, op_shift, normalize_l1, phase, delta_row_host,
                                   delta_col_host, delta_val_host, n_delta, stream);
}

int egnn_cheb_order_sharded_vals(const int32_t* rowptr_local, const int32_t* colidx_local, const float* vals_local,
                                 const int32_t* rowptr_remote, const int32_t* colidx_remote, const float* vals_remote,
                                 const float* dinv_full, const uint8_t* iso_full, const float* t_prev_full,
                                 const float* t_prev_local, const float* t_prev2_local, float* t_out_local,
                                 float* out_local, float* acc_ws, int64_t n, int64_t nnz_hint,
                                 int64_t row_begin, int64_t row_end, int32_t f, int32_t order, int32_t k_max,
                                 int32_t n_scales, const float* coeffs_host, float op_scale, float op_shift,
                                 int32_t normalize_l1, int32_t phase,
                                 const int32_t* delta_row_host, const int32_t* delta_col_host,
                                 const float* delta_val_host, int32_t n_delta, egnn_stream_t stream) {
    return cheb_order_sharded_impl(rowptr_local, colidx_local, vals_local, rowptr_remote, colidx_remote, vals_remote,
                                   dinv_full, iso_full, t_prev_full, t_prev_local, t_prev2_local, t_out_local,
                                   out_local, acc_ws, n, nnz_hint, row_begin, row_end, f, order, k_max, n_scales,
                                   coeffs_host, op_scale, op_shift, normalize_l1, phase, delta_row_host,
                                   delta_col_host, delta_val_host, n_delta, stream);
}

int egnn_sell_geometry(int64_t n, int64_t nnz, int32_t* n_blocks, int32_t* col_block, int32_t* lmax) {
    EGNN_REQUIRE(n_blocks && col_block && lmax, "null pointer");
    EGNN_REQUIRE(n >= 1, "bad shape");
    int nb = 1, cb = 32;
    narrow_geometry(n, &nb, &cb);
    *n_blocks = nb;
    *col_block = cb;
    *lmax = 256;
    (void)nnz;
    return EGNN_OK;
}

size_t egnn_sell_ws_bytes(int64_t n, int64_t nnz, int32_t n_blocks, int32_t lmax) {
    if (n < 1 || n_blocks < 1 || lmax < 8) return 0;
    return sell_ws_layout(nullptr, n, nnz, n_blocks, lmax).total_bytes;
}

int egnn_sell_prepare(const int32_t* rowptr, const int32_t* colidx, int64_t n, int64_t nnz,
                      egnn_sell_plan* plan, void* workspace, size_t workspace_bytes, egnn_stream_t stream) {
    int rc = sell_check_geometry(n, nnz, plan);
    if (rc) return rc;
    EGNN_REQUIRE(rowptr && (colidx || nnz == 0), "null pointer");
    const int C = plan->n_blocks, CB = plan->col_block, lmax = plan->lmax;
    SellWs w = sell_ws_layout(workspace, n, nnz, C, lmax);
    rc = require_workspace(workspace, workspace_bytes, w.total_bytes, "sell workspace");
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t cn = (int64_t)C * n;
    rc = check_cuda(cudaMemsetAsync(w.nv + cn, 0, 4, st), "memset"); if (rc) return rc;
    rc = check_cuda(cudaMemsetAsync(w.nvrow + n, 0, 4, st), "memset"); if (rc) return rc;
    rc = check_cuda(cudaMemsetAsync(w.key, 0xff, 4 * w.umax, st), "memset"); if (rc) return rc;
    rc = check_cuda(cudaMemsetAsync(w.slice_sz, 0, 4 * (w.smax + 1), st), "memset"); if (rc) return rc;
    rc = check_cuda(cudaMemsetAsync(w.totals, 0, 64, st), "memset"); if (rc) return rc;
    sell_count_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, st>>>(rowptr, colidx, (int)n, C, CB, lmax, w.seg_start,
                                                                   w.seg_cnt, w.nv, w.nvrow);
    EGNN_LAUNCH_CHECK("sell_count_kernel launch");
    size_t tb = w.cub_bytes;
    rc = check_cuda(cub::DeviceScan::ExclusiveSum(w.cub_temp, tb, w.nv, w.u_off, (int)(cn + 1), st), "scan nv"); if (rc) return rc;
    tb = w.cub_bytes;
    rc = check_cuda(cub::DeviceScan::ExclusiveSum(w.cub_temp, tb, w.nvrow, w.rv_ptr, (int)(n + 1), st), "scan nvrow"); if (rc) return rc;
    sell_emit_kernel<<<(unsigned)ceil_div64(cn, 256), 256, 0, st>>>((int)n, C, lmax, w.seg_start, w.seg_cnt, w.nv, w.u_off,
                                                                   w.rv_ptr, w.key, w.uval, w.vsrc, w.vslot, w.vrow);
    EGNN_LAUNCH_CHECK("sell_emit_kernel launch");
    tb = w.cub_bytes;
    rc = check_cuda(cub::DeviceRadixSort::SortPairs(w.cub_temp, tb, w.key, w.key_sorted, w.uval, w.perm, (int)w.umax, 0, 32, st), "sort vrows");
    if (rc) return rc;
    sell_blocks_kernel<<<1, 32, 0, st>>>((int)n, C, w.u_off, w.q_ptr, w.vp_ptr, w.bsp, w.bstride, w.totals);
    EGNN_LAUNCH_CHECK("sell_blocks_kernel launch");
    sell_slice_kernel<<<(unsigned)ceil_div64(w.smax, 256), 256, 0, st>>>(C, lmax, w.key_sorted, w.q_ptr, w.bsp, w.bstride, w.totals, w.slice_sz);
    EGNN_LAUNCH_CHECK("sell_slice_kernel launch");
    tb = w.cub_bytes;
    rc = check_cuda(cub::DeviceScan::ExclusiveSum(w.cub_temp, tb, w.slice_sz, w.slice_off, (int)(w.smax + 1), st), "scan slices"); if (rc) return rc;
    sell_totals_kernel<<<1, 32, 0, st>>>(w.slice_off, w.rv_ptr, (int)n, w.totals);
    EGNN_LAUNCH_CHECK("sell_totals_kernel launch");
    sell_hub_count_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, st>>>(w.rv_ptr, (int)n, w.totals);
    EGNN_LAUNCH_CHECK("sell_hub_count_kernel launch");
    int64_t tot[8];
    rc = check_cuda(cudaMemcpyAsync(tot, w.totals, 64, cudaMemcpyDeviceToHost, st), "copy totals"); if (rc) return rc;
    rc = check_cuda(cudaStreamSynchronize(st), "sync"); if (rc) return rc;
    plan->n = (int32_t)n;
    plan->n_cta = device_sm_count();               // persistent grid of the hot kernel: one CTA per SM
    plan->n_vrows = tot[kTotV];
    plan->n_slices = tot[kTotSlices];
    plan->n_entries = tot[kTotEntries];
    plan->n_rowv = tot[kTotRowV];
    plan->n_hub = tot[kTotHub];
    return EGNN_OK;
}

int egnn_sell_fill(const int32_t* rowptr, const int32_t* colidx, int64_t n, int64_t nnz,
                   const egnn_sell_plan* plan, void* workspace, size_t workspace_bytes, egnn_stream_t stream) {
    int rc = sell_check_geometry(n, nnz, plan);
    if (rc) return rc;
    (void)rowptr;
    EGNN_REQUIRE(plan->slice_off && plan->blk_slice_ptr && plan->rv_ptr && plan->cta_info && plan->sched && plan->hub,
                 "plan buffers not allocated");
    EGNN_REQUIRE(plan->n_hub >= 0 && plan->n_hub <= n, "n_hub out of range");
    EGNN_REQUIRE(plan->n_cta >= 1 && plan->n_cta <= 4096, "n_cta out of range");
    EGNN_REQUIRE(plan->n_entries == 0 || plan->idx, "plan idx not allocated");
    EGNN_REQUIRE(plan->n_vrows == 0 || plan->vslot, "plan vslot not allocated");
    const int C = plan->n_blocks, CB = plan->col_block, lmax = plan->lmax;
    SellWs w = sell_ws_layout(workspace, n, nnz, C, lmax);
    rc = require_workspace(workspace, workspace_bytes, w.total_bytes, "sell workspace");
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    rc = check_cuda(cudaMemcpyAsync(plan->slice_off, w.slice_off, 4 * (plan->n_slices + 1), cudaMemcpyDeviceToDevice, st), "copy slice_off"); if (rc) return rc;
    rc = check_cuda(cudaMemcpyAsync(plan->blk_slice_ptr, w.bsp, 4 * (C + 1), cudaMemcpyDeviceToDevice, st), "copy blk_slice_ptr"); if (rc) return rc;
    rc = check_cuda(cudaMemcpyAsync(plan->rv_ptr, w.rv_ptr, 4 * (n + 1), cudaMemcpyDeviceToDevice, st), "copy rv_ptr"); if (rc) return rc;
    sell_cta_blocks_kernel<<<1, 32, 0, st>>>(w.slice_off, w.bsp, C, plan->n_cta, plan->cta_info, plan->sched);
    EGNN_LAUNCH_CHECK("sell_cta_blocks_kernel launch");
    // epilogue row ranges balanced by cost, and the hub rows of every range (nvrow / nv / u_off / key
    // of the workspace are free again: reused for the costs, the hub flags and their prefixes)
    int32_t* hub_flag = w.u_off;
    int32_t* hub_prefix = reinterpret_cast<int32_t*>(w.key);
    int32_t* cta_rows = plan->cta_info + 2 * plan->n_cta + kSellMaxBlocks;
    sell_row_cost_kernel<<<(unsigned)ceil_div64(n + 1, 256), 256, 0, st>>>(w.rv_ptr, (int)n, w.nvrow, hub_flag);
    EGNN_LAUNCH_CHECK("sell_row_cost_kernel launch");
    size_t tb = w.cub_bytes;
    rc = check_cuda(cub::DeviceScan::ExclusiveSum(w.cub_temp, tb, w.nvrow, w.nv, (int)(n + 1), st), "scan row costs"); if (rc) return rc;
    sell_cta_rows_kernel<<<(unsigned)ceil_div64(plan->n_cta + 1, 128), 128, 0, st>>>(w.nv, (int)n, plan->n_cta, cta_rows);
    EGNN_LAUNCH_CHECK("sell_cta_rows_kernel launch");
    tb = w.cub_bytes;
    rc = check_cuda(cub::DeviceScan::ExclusiveSum(w.cub_temp, tb, hub_flag, hub_prefix, (int)(n + 1), st), "scan hub flags"); if (rc) return rc;
    sell_cta_hubs_kernel<<<(unsigned)ceil_div64(n > plan->n_cta ? n : plan->n_cta + 1, 256), 256, 0, st>>>(
        hub_flag, hub_prefix, cta_rows, (int)n, plan->n_cta, plan->hub);
    EGNN_LAUNCH_CHECK("sell_cta_hubs_kernel launch");
    if (plan->n_slices > 0) {
        rc = check_cuda(cudaFuncSetAttribute(sell_fill_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSellFillSmem),
                        "cudaFuncSetAttribute(sell_fill_kernel)");
        if (rc) return rc;
        sell_fill_kernel<<<(unsigned)ceil_div64(plan->n_slices, kSellFillWarps), kSellFillWarps * 32, kSellFillSmem, st>>>(
            colidx, C, CB, lmax, (int)plan->n_slices, w.key_sorted, w.perm, w.vsrc, w.vslot, w.vrow, w.q_ptr, w.vp_ptr,
            w.bsp, w.bstride, w.slice_off, plan->idx, plan->vslot, plan->row0);
        EGNN_LAUNCH_CHECK("sell_fill_kernel launch");
    }
    return EGNN_OK;
}

int egnn_sell_step_sharded(const egnn_sell_plan* plan, const float* dinv_full, const uint8_t* iso_full,
                           const float* x0_local, const float* y_first_full, float* y_slab0, float* y_slab1,
                           float* tbuf0, float* tbuf1, float* t_all_or_null, float* out_local,
                           int32_t order_begin, int32_t order_end, int32_t k_max, int32_t n_scales,
                           const float* coeffs_host, float op_scale, float op_shift, int32_t normalize_l1,
                           const int32_t* delta_row_host, const int32_t* delta_col_host,
                           const float* delta_val_host, int32_t n_delta,
                           const float* w_base_or_null, const float* rowsum_base_or_null, int32_t default_signal,
                           const egnn_peer_window* win, egnn_stream_t stream) {
    EGNN_REQUIRE(plan && dinv_full && iso_full && out_local && coeffs_host, "null pointer");
    EGNN_REQUIRE((w_base_or_null == nullptr) == (rowsum_base_or_null == nullptr), "w_base and rowsum_base come together");
    EGNN_REQUIRE(plan->vpart && plan->slice_off && plan->blk_slice_ptr && plan->rv_ptr && plan->vslot && plan->cta_info && plan->hub && plan->sched,
                 "SELL plan is not filled");
    EGNN_REQUIRE(order_begin >= 1 && order_begin <= order_end && order_end <= k_max && k_max <= EGNN_MAX_ORDER, "bad order range");
    EGNN_REQUIRE(n_scales >= 1 && n_scales <= EGNN_MAX_SCALES, "n_scales out of range");
    EGNN_REQUIRE(plan->n == 0 || x0_local, "T_0 rows missing");
    EGNN_REQUIRE(t_all_or_null || k_max == 1 || (tbuf0 && tbuf1), "T buffers missing");
    const bool fused = win && win->world > 1;
    if (win) {
        int rc = peer_check(win);
        if (rc) return rc;
        EGNN_REQUIRE(win->f == 1 && (int64_t)win->world * win->rows_per >= plan->n_cols &&
                     (int64_t)plan->row0 + plan->n <= (int64_t)win->world * win->rows_per, "window does not fit the plan");
    } else {
        // without a window one launch covers one order: the caller exchanges the operand in between
        EGNN_REQUIRE(plan->n == plan->n_cols || (order_begin == order_end && y_first_full),
                     "a row shard without an exchange window runs one order per call on a gathered operand");
        EGNN_REQUIRE(order_end == k_max || (y_slab0 && y_slab1), "operand slabs missing");
    }
    SellStepParams sp{};
    int rc = fill_delta(sp.delta, delta_row_host, delta_col_host, delta_val_host, n_delta, plan->n_cols);
    if (rc) return rc;
    step_fill_plan(sp, plan);
    sp.w_base = w_base_or_null; sp.rowsum_base = rowsum_base_or_null; sp.patch_x0 = default_signal ? 1 : 0;
    sp.dinv = dinv_full; sp.iso = iso_full; sp.x0 = x0_local; sp.operand_first = y_first_full;
    sp.tbuf[0] = tbuf0; sp.tbuf[1] = tbuf1; sp.t_all = t_all_or_null; sp.out = out_local;
    sp.normalize = normalize_l1; sp.a = op_scale; sp.b = op_shift;
    sp.world = 1; sp.rank = 0; sp.rows_per = plan->n_cols;
    if (win) {
        // operand buffers live in the exchange windows: order k reads buffer (k-1)&1 of the own
        // window, its epilogue stores dinv (.) T_k into buffer k&1 of EVERY rank's window
        step_fill_peer(sp, win);
        for (int b = 0; b < 2; ++b) {
            sp.operand[b] = peer_operand(win, win->rank, b);
            for (int r = 0; r < win->world; ++r) sp.ydst[b][r] = peer_operand(win, r, b);
        }
        sp.n_dst = win->world;
    } else {
        // operand slabs hold only the own rows: shifted so that the global row index lands in them
        float* slab[2] = {y_slab0, y_slab1};
        for (int b = 0; b < 2; ++b) {
            sp.operand[b] = nullptr;
            sp.ydst[b][0] = slab[b] ? (float*)((uintptr_t)slab[b] - sizeof(float) * (size_t)plan->row0) : nullptr;
        }
        if (plan->n == plan->n_cols) { sp.operand[0] = y_slab0; sp.operand[1] = y_slab1; }
        sp.n_dst = 1;
    }
    return run_sell_step(sp, k_max, n_scales, coeffs_host, fused, (cudaStream_t)stream, order_begin, order_end);
}

size_t egnn_calibration_metrics_ws_bytes(int32_t n_classes, int32_t n_bins) {
    if (n_classes < 1 || n_bins < 1 || n_bins > kEceMaxBins) return 0;
    return 3 * align_up(8 * (size_t)n_classes * n_bins, 256) + 256 + 256;
}

int egnn_calibration_metrics(const float* x, int32_t is_log, const int64_t* labels, const uint8_t* mask_or_null,
                             int64_t n, int32_t n_classes, int32_t n_bins, double* out3, void* workspace,
                             size_t workspace_bytes, egnn_stream_t stream) {
    EGNN_REQUIRE(x && labels && out3, "null pointer");
    EGNN_REQUIRE(n >= 0 && n_classes >= 1 && n_bins >= 1 && n_bins <= kEceMaxBins, "bad shape");
    int rc = require_workspace(workspace, workspace_bytes, egnn_calibration_metrics_ws_bytes(n_classes, n_bins),
                               "metrics workspace");
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    char* base = (char*)align_up((size_t)workspace, 256);
    const size_t arr = align_up(8 * (size_t)n_classes * n_bins, 256);
    EceWs ws;
    ws.sum_p = (double*)base;
    ws.count = (unsigned long long*)(base + arr);
    ws.hits = (unsigned long long*)(base + 2 * arr);
    ws.scalars = (double*)(base + 3 * arr);
    rc = check_cuda(cudaMemsetAsync(base, 0, 3 * arr + 64, st), "memset metrics workspace");
    if (rc) return rc;
    if (n > 0) {
        ece_accumulate_kernel<<<grid_for(n * 32, 256), 256, 0, st>>>(x, is_log, labels, mask_or_null, n, n_classes, n_bins, ws);
        EGNN_LAUNCH_CHECK("ece_accumulate_kernel launch");
    }
    ece_finalize_kernel<<<1, 256, 0, st>>>(n_classes, n_bins, ws, out3);
    EGNN_LAUNCH_CHECK("ece_finalize_kernel launch");
    return EGNN_OK;
}

int egnn_temperature_head(const float* feats, const float* w1, const float* b1, const float* w2, const float* b2,
                          const float* logits, float* out, float* temps_out_or_null, int64_t n, int32_t f,
                          int32_t hidden, int32_t n_classes, egnn_stream_t stream) {
    EGNN_REQUIRE(feats && w1 && b1 && w2 && b2 && logits && out, "null pointer");
    EGNN_REQUIRE(n >= 0 && n_classes >= 1, "bad shape");
    EGNN_REQUIRE(f >= 1 && f <= kHeadMaxFeat && hidden >= 1 && hidden <= kHeadMaxHidden, "head too large (f, hidden <= 64)");
    if (n == 0) return EGNN_OK;
    temperature_head_kernel<<<grid_for(n * 32, 256), 256, 0, (cudaStream_t)stream>>>(feats, w1, b1, w2, b2, logits, out,
                                                                                   temps_out_or_null, n, f, hidden,
                                                                                   n_classes);
    EGNN_LAUNCH_CHECK("temperature_head_kernel launch");
    return EGNN_OK;
}

size_t egnn_peer_window_bytes(int64_t rows_per, int32_t world, int32_t f) {
    if (rows_per < 1 || world < 1 || f < 1) return 0;
    egnn_peer_window w{};
    w.world = world; w.rows_per = rows_per; w.f = f;
    return kPeerHeaderBytes + 2 * peer_slab_stride(&w);
}

int egnn_peer_alloc(size_t bytes, void** dev_ptr, void* ipc_handle_out) {
    EGNN_REQUIRE(dev_ptr && ipc_handle_out && bytes >= kPeerHeaderBytes, "bad arguments");
    static_assert(sizeof(cudaIpcMemHandle_t) == EGNN_IPC_HANDLE_BYTES, "IPC handle size");
    void* ptr = nullptr;
    int rc = check_cuda(cudaMalloc(&ptr, bytes), "cudaMalloc(exchange window)");
    if (rc) return rc;
    rc = check_cuda(cudaMemset(ptr, 0, bytes), "cudaMemset(exchange window)");
    if (rc) { cudaFree(ptr); return rc; }
    cudaIpcMemHandle_t h;
    rc = check_cuda(cudaIpcGetMemHandle(&h, ptr), "cudaIpcGetMemHandle");
    if (rc) { cudaFree(ptr); return rc; }
    memcpy(ipc_handle_out, &h, sizeof(h));
    *dev_ptr = ptr;
    return EGNN_OK;
}

int egnn_peer_open(const void* ipc_handle, void** dev_ptr) {
    EGNN_REQUIRE(ipc_handle && dev_ptr, "null pointer");
    cudaIpcMemHandle_t h;
    memcpy(&h, ipc_handle, sizeof(h));
    void* ptr = nullptr;
    int rc = check_cuda(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess), "cudaIpcOpenMemHandle");
    if (rc) return rc;
    *dev_ptr = ptr;
    return EGNN_OK;
}

int egnn_peer_close(void* dev_ptr) {
    EGNN_REQUIRE(dev_ptr != nullptr, "null pointer");
    return check_cuda(cudaIpcCloseMemHandle(dev_ptr), "cudaIpcCloseMemHandle");
}

int egnn_peer_free(void* dev_ptr) {
    EGNN_REQUIRE(dev_ptr != nullptr, "null pointer");
    return check_cuda(cudaFree(dev_ptr), "cudaFree(exchange window)");
}

void* egnn_peer_operand(const egnn_peer_window* win, int32_t which) {
    if (!win || which < 0 || which > 1 || win->rank < 0 || win->rank >= EGNN_MAX_RANKS || !win->base[win->rank]) return nullptr;
    return peer_operand(win, win->rank, which);
}

int egnn_peer_error(const egnn_peer_window* win, int32_t* error_out, egnn_stream_t stream) {
    EGNN_REQUIRE(win && error_out, "null pointer");
    int rc = peer_check(win);
    if (rc) return rc;
    unsigned v = 0;
    rc = check_cuda(cudaMemcpyAsync(&v, (char*)win->base[win->rank] + kPeerErrorOff, 4, cudaMemcpyDeviceToHost,
                                    (cudaStream_t)stream), "copy error word");
    if (rc) return rc;
    rc = check_cuda(cudaStreamSynchronize((cudaStream_t)stream), "sync");
    if (rc) return rc;
    *error_out = (int32_t)v;
    return EGNN_OK;
}

int egnn_peer_wait_stats(const egnn_peer_window* win, uint64_t* total_ns, uint64_t* waits, int32_t reset,
                         egnn_stream_t stream) {
    EGNN_REQUIRE(win && total_ns && waits, "null pointer");
    int rc = peer_check(win);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long v[2] = {0, 0};
    char* stat = (char*)win->base[win->rank] + kPeerWaitNsOff;
    rc = check_cuda(cudaMemcpyAsync(v, stat, 16, cudaMemcpyDeviceToHost, st), "copy wait stats");
    if (rc) return rc;
    rc = check_cuda(cudaStreamSynchronize(st), "sync");
    if (rc) return rc;
    if (reset) {
        rc = check_cuda(cudaMemsetAsync(stat, 0, 16, st), "reset wait stats");
        if (rc) return rc;
    }
    *total_ns = v[0];
    *waits = v[1];
    return EGNN_OK;
}

int egnn_peer_prescale_push(const float* x_local, const float* dinv_full, int64_t n_rows, int64_t row0, int32_t f,
                            const egnn_peer_window* win, egnn_stream_t stream) {
    EGNN_REQUIRE(dinv_full && win, "null pointer");
    EGNN_REQUIRE(n_rows >= 0 && row0 >= 0 && f >= 1 && (n_rows == 0 || x_local), "bad shape");
    int rc = peer_check(win);
    if (rc) return rc;
    EGNN_REQUIRE(win->f == (f >= kWideMinF ? wide_ldy(f) : f) && row0 + n_rows <= (int64_t)win->world * win->rows_per,
                 "window does not fit the signal");
    PeerPush pp{};
    fill_peer_push(pp, win, 0, true, true);
    peer_prescale_push_kernel<<<push_grid(n_rows * win->f), 1024, 0, (cudaStream_t)stream>>>(x_local, dinv_full, n_rows,
                                                                                            row0, f, win->f, pp);
    EGNN_LAUNCH_CHECK("peer_prescale_push_kernel launch");
    return EGNN_OK;
}

int egnn_wide_order_sharded(const int32_t* rowptr_local, const int32_t* colidx_local, const float* vals_or_null,
                            const int32_t* row_order_or_null, const float* dinv_full, const uint8_t* iso_full,
                            const float* x0_local, float* t_out_local_or_null, float* out_local, int64_t n_global,
                            int64_t row_begin, int64_t row_end, int32_t f, int32_t order, int32_t k_max,
                            int32_t n_scales, const float* coeffs_host, float op_scale, float op_shift,
                            int32_t normalize_l1, const int32_t* delta_row_host, const int32_t* delta_col_host,
                            const float* delta_val_host, int32_t n_delta, const egnn_peer_window* win,
                            egnn_stream_t stream) {
    EGNN_REQUIRE(rowptr_local && dinv_full && iso_full && out_local && coeffs_host && win, "null pointer");
    EGNN_REQUIRE(row_begin >= 0 && row_end >= row_begin && row_end <= n_global, "bad row range");
    EGNN_REQUIRE(f >= kWideMinF, "the wide sharded order serves f >= 8");
    EGNN_REQUIRE(order >= 1 && order <= k_max && k_max <= EGNN_MAX_ORDER, "bad order");
    EGNN_REQUIRE(n_scales >= 1 && n_scales <= EGNN_MAX_SCALES, "n_scales out of range");
    EGNN_REQUIRE(order > 1 || x0_local || row_end == row_begin, "T_0 rows missing");
    int rc = peer_check(win);
    if (rc) return rc;
    EGNN_REQUIRE(win->f == wide_ldy(f) && (int64_t)win->world * win->rows_per >= n_global, "window does not fit the signal");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t rows = row_end - row_begin;
    ChebArgs c{};
    c.rowptr = rowptr_local; c.colidx = colidx_local; c.vals = vals_or_null; c.row_order = row_order_or_null;
    c.dinv = dinv_full; c.iso = iso_full; c.rows = rows; c.row0 = row_begin; c.f = f; c.k = k_max; c.S = n_scales;
    c.coeffs = coeffs_host; c.a = op_scale; c.b = op_shift; c.st = st;
    rc = fill_delta(c.delta, delta_row_host, delta_col_host, delta_val_host, n_delta, n_global);
    if (rc) return rc;
    const RingConfig rcfg = ring_config(wide_ldy(f));
    const bool last = order == k_max;
    const bool fuse_norm = normalize_l1 && rcfg.grid_y == 1;
    WideParams wp = wide_params(c);
    wp.out = out_local;
    wp.first = order == 1;
    wp.normalize = last && fuse_norm;
    wp.x0_own = order == 1 ? x0_local : nullptr;
    wp.tk_out = t_out_local_or_null;
    order_coefs(wp.c_prev, coeffs_host, k_max, n_scales, order - 1);
    order_coefs(wp.c_k, coeffs_host, k_max, n_scales, order);
    rc = wide_sharded_step<false>(wp, rcfg, win, order, last, st);
    if (rc) return rc;
    if (last && normalize_l1 && !fuse_norm && rows > 0) return launch_l1_normalize(out_local, rows, n_scales, f, st);
    return EGNN_OK;
}

// ---- backward of the row-sharded pass ------------------------------------------------------------
// Application app = 1..K of the adjoint produces b_m, m = K - app, on the rank's rows (b_0: the
// signal's gradient); app 0 is the prologue b_K = v_K.  tbar_or_null is the whole [K+1, rows, f] stack.
static int adjoint_sharded_check(int64_t n, int64_t row_begin, int64_t row_end, int32_t f, int32_t app, int32_t k_max,
                                 int32_t n_scales) {
    EGNN_REQUIRE(n >= 0 && n < (int64_t(1) << 31) && row_begin >= 0 && row_end >= row_begin && row_end <= n,
                 "bad row range");
    EGNN_REQUIRE(f >= 1, "f must be >= 1");
    EGNN_REQUIRE(k_max >= 0 && k_max <= EGNN_MAX_ORDER && app >= 0 && app <= k_max, "bad application");
    EGNN_REQUIRE(n_scales >= 1 && n_scales <= EGNN_MAX_SCALES, "n_scales out of range");
    return EGNN_OK;
}

// Binary (vals_local == vals_remote == NULL) or weighted (both given) shard of the transposed adjacency.
static int cheb_adjoint_sharded_impl(const int32_t* rowptr_local, const int32_t* colidx_local, const float* vals_local,
                                     const int32_t* rowptr_remote, const int32_t* colidx_remote,
                                     const float* vals_remote, const float* dinv_full, const uint8_t* iso_full,
                                     const float* b_prev_full, const float* b_prev_local,
                                     const float* b_prev2_local_or_null, float* b_out_local, const float* cbar_local,
                                     const float* tbar_local_or_null, float* acc_ws, int64_t n, int64_t nnz_hint,
                                     int64_t row_begin, int64_t row_end, int32_t f, int32_t app, int32_t k_max,
                                     int32_t n_scales, const float* coeffs_host, float op_scale, float op_shift,
                                     int32_t phase, const int32_t* delta_row_host, const int32_t* delta_col_host,
                                     const float* delta_val_host, int32_t n_delta, egnn_stream_t stream) {
    EGNN_REQUIRE(dinv_full && iso_full && b_out_local && cbar_local && coeffs_host, "null pointer");
    int rc = adjoint_sharded_check(n, row_begin, row_end, f, app, k_max, n_scales);
    if (rc) return rc;
    EGNN_REQUIRE(phase >= 0 && phase <= 2, "bad phase");
    EGNN_REQUIRE(app == 0 || b_prev_local, "b_{m+1} rows missing");
    EGNN_REQUIRE((vals_local == nullptr) == (vals_remote == nullptr), "values of the local and remote halves come together");
    EGNN_REQUIRE(vec_aligned(b_prev_full, f) && vec_aligned(b_prev_local, f) && vec_aligned(b_prev2_local_or_null, f) &&
                 vec_aligned(b_out_local, f) && vec_aligned(cbar_local, f) && vec_aligned(tbar_local_or_null, f) &&
                 vec_aligned(acc_ws, f), "b, cbar, tbar and acc_ws must be 16-byte aligned when f % 4 == 0");
    const int64_t rows = row_end - row_begin;
    if (rows == 0) return EGNN_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t slab_elems = (size_t)rows * (size_t)f;
    const int m = k_max - app;
    const float* tbar_m = slab_of(tbar_local_or_null, slab_elems, m);
    if (app == 0) {
        adjoint_prologue_kernel<<<grid_for((int64_t)slab_elems, 256), 256, 0, st>>>(
            cbar_local, tbar_m, dinv_full + row_begin, b_out_local, nullptr, rows, f, n_scales, f,
            coef_row(coeffs_host, k_max, n_scales, k_max));
        EGNN_LAUNCH_CHECK("adjoint_prologue_kernel launch");
        return EGNN_OK;
    }
    ChebArgs c{};
    c.rowptr = rowptr_local; c.colidx = colidx_local; c.vals = vals_local; c.dinv = dinv_full; c.iso = iso_full;
    c.rows = rows; c.row0 = row_begin; c.nnz = nnz_hint; c.f = f; c.k = k_max; c.S = n_scales;
    c.coeffs = coeffs_host; c.a = op_scale; c.b = op_shift; c.st = st;
    OrderConfig cfg = choose_config(rows, nnz_hint, f);
    cfg.prescaled = false;            // sharded slabs carry plain b (what the exchange moves)
    OrderParams p = order_params(c, cfg);
    p.tprev_own = b_prev_local; p.tprev2_own = b_prev2_local_or_null; p.tk_own = b_out_local; p.acc_ws = acc_ws;
    p.cbar = cbar_local; p.tbar = tbar_m; p.c_adj = m == 0 ? 1.f : 2.f;
    order_coefs(p.c_k, coeffs_host, k_max, n_scales, m);
    return order_sharded_phase<true>(p, cfg, phase, rowptr_remote, colidx_remote, vals_remote, b_prev_full,
                                     "gathered b_{m+1} missing", delta_row_host, delta_col_host, delta_val_host,
                                     n_delta, n, st);
}

int egnn_cheb_adjoint_sharded(const int32_t* rowptr_local, const int32_t* colidx_local,
                              const int32_t* rowptr_remote, const int32_t* colidx_remote,
                              const float* dinv_full, const uint8_t* iso_full, const float* b_prev_full,
                              const float* b_prev_local, const float* b_prev2_local_or_null, float* b_out_local,
                              const float* cbar_local, const float* tbar_local_or_null, float* acc_ws,
                              int64_t n, int64_t nnz_hint, int64_t row_begin, int64_t row_end, int32_t f,
                              int32_t app, int32_t k_max, int32_t n_scales, const float* coeffs_host,
                              float op_scale, float op_shift, int32_t phase,
                              const int32_t* delta_row_host, const int32_t* delta_col_host,
                              const float* delta_val_host, int32_t n_delta, egnn_stream_t stream) {
    return cheb_adjoint_sharded_impl(rowptr_local, colidx_local, nullptr, rowptr_remote, colidx_remote, nullptr,
                                     dinv_full, iso_full, b_prev_full, b_prev_local, b_prev2_local_or_null,
                                     b_out_local, cbar_local, tbar_local_or_null, acc_ws, n, nnz_hint, row_begin,
                                     row_end, f, app, k_max, n_scales, coeffs_host, op_scale, op_shift, phase,
                                     delta_row_host, delta_col_host, delta_val_host, n_delta, stream);
}

int egnn_cheb_adjoint_sharded_vals(const int32_t* rowptr_local, const int32_t* colidx_local, const float* vals_local,
                                   const int32_t* rowptr_remote, const int32_t* colidx_remote,
                                   const float* vals_remote, const float* dinv_full, const uint8_t* iso_full,
                                   const float* b_prev_full, const float* b_prev_local,
                                   const float* b_prev2_local_or_null, float* b_out_local, const float* cbar_local,
                                   const float* tbar_local_or_null, float* acc_ws, int64_t n, int64_t nnz_hint,
                                   int64_t row_begin, int64_t row_end, int32_t f, int32_t app, int32_t k_max,
                                   int32_t n_scales, const float* coeffs_host, float op_scale, float op_shift,
                                   int32_t phase, const int32_t* delta_row_host, const int32_t* delta_col_host,
                                   const float* delta_val_host, int32_t n_delta, egnn_stream_t stream) {
    return cheb_adjoint_sharded_impl(rowptr_local, colidx_local, vals_local, rowptr_remote, colidx_remote,
                                     vals_remote, dinv_full, iso_full, b_prev_full, b_prev_local,
                                     b_prev2_local_or_null, b_out_local, cbar_local, tbar_local_or_null, acc_ws, n,
                                     nnz_hint, row_begin, row_end, f, app, k_max, n_scales, coeffs_host, op_scale,
                                     op_shift, phase, delta_row_host, delta_col_host, delta_val_host, n_delta, stream);
}

// Fused wide adjoint of a binary or weighted shard; b_out_local_or_null [rows, f] receives b_m of every
// application m >= 1 (app 0: b_K), as egnn_cheb_adjoint_all keeps them on one GPU.
static int wide_adjoint_sharded_impl(const int32_t* rowptr_local, const int32_t* colidx_local,
                                     const float* vals_or_null, const int32_t* row_order_or_null,
                                     const float* dinv_full, const uint8_t* iso_full, const float* cbar_local,
                                     const float* tbar_local_or_null, float* xbar_local, float* b_out_local_or_null,
                                     int64_t n_global, int64_t row_begin, int64_t row_end, int32_t f, int32_t app,
                                     int32_t k_max, int32_t n_scales, const float* coeffs_host, float op_scale,
                                     float op_shift, const int32_t* delta_row_host, const int32_t* delta_col_host,
                                     const float* delta_val_host, int32_t n_delta, const egnn_peer_window* win,
                                     egnn_stream_t stream) {
    EGNN_REQUIRE(rowptr_local && dinv_full && iso_full && cbar_local && coeffs_host && win, "null pointer");
    int rc = adjoint_sharded_check(n_global, row_begin, row_end, f, app, k_max, n_scales);
    if (rc) return rc;
    EGNN_REQUIRE(f >= kWideMinF, "the wide sharded adjoint serves f >= 8");
    EGNN_REQUIRE(k_max >= 1, "k_max = 0 has no application to exchange");
    EGNN_REQUIRE(app < k_max || xbar_local || row_end == row_begin, "xbar rows missing");
    EGNN_REQUIRE(vec_aligned(cbar_local, f) && vec_aligned(tbar_local_or_null, f) && vec_aligned(xbar_local, f) &&
                 vec_aligned(b_out_local_or_null, f),
                 "cbar, tbar, xbar and b_out must be 16-byte aligned when f % 4 == 0");
    rc = peer_check(win);
    if (rc) return rc;
    const int ldy = wide_ldy(f);
    EGNN_REQUIRE(win->f == ldy && (int64_t)win->world * win->rows_per >= n_global, "window does not fit the signal");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t rows = row_end - row_begin;
    const size_t slab_elems = (size_t)rows * (size_t)f;
    const int m = k_max - app;
    const float* tbar_m = slab_of(tbar_local_or_null, slab_elems, m);
    if (app == 0) {                   // b_K = v_K, its operand into buffer 0 of every window
        PeerPush pp{};
        fill_peer_push(pp, win, 0, true, true);
        adjoint_prologue_push_kernel<<<push_grid(rows * ldy), 1024, 0, st>>>(
            cbar_local, tbar_m, dinv_full, rows, row_begin, f, n_scales, ldy, coef_row(coeffs_host, k_max, n_scales, k_max),
            pp);
        EGNN_LAUNCH_CHECK("adjoint_prologue_push_kernel launch");
        if (b_out_local_or_null && rows > 0) {        // and b_K itself into the caller's rows
            adjoint_prologue_kernel<<<grid_for((int64_t)slab_elems, 256), 256, 0, st>>>(
                cbar_local, tbar_m, dinv_full + row_begin, b_out_local_or_null, nullptr, rows, f, n_scales, f,
                coef_row(coeffs_host, k_max, n_scales, k_max));
            EGNN_LAUNCH_CHECK("adjoint_prologue_kernel launch");
        }
        return EGNN_OK;
    }
    ChebArgs c{};
    c.rowptr = rowptr_local; c.colidx = colidx_local; c.vals = vals_or_null; c.row_order = row_order_or_null;
    c.dinv = dinv_full; c.iso = iso_full; c.rows = rows; c.row0 = row_begin; c.f = f; c.k = k_max; c.S = n_scales;
    c.coeffs = coeffs_host; c.a = op_scale; c.b = op_shift; c.st = st;
    rc = fill_delta(c.delta, delta_row_host, delta_col_host, delta_val_host, n_delta, n_global);
    if (rc) return rc;
    WideParams wp = wide_params(c);
    wp.tk_out = m == 0 ? xbar_local : b_out_local_or_null;
    wp.cbar = cbar_local; wp.tbar = tbar_m; wp.c_adj = m == 0 ? 1.f : 2.f;
    order_coefs(wp.c_k, coeffs_host, k_max, n_scales, m);
    return wide_sharded_step<true>(wp, ring_config(ldy), win, app, m == 0, st);
}

int egnn_wide_adjoint_sharded(const int32_t* rowptr_local, const int32_t* colidx_local,
                              const int32_t* row_order_or_null, const float* dinv_full, const uint8_t* iso_full,
                              const float* cbar_local, const float* tbar_local_or_null, float* xbar_local,
                              int64_t n_global, int64_t row_begin, int64_t row_end, int32_t f, int32_t app,
                              int32_t k_max, int32_t n_scales, const float* coeffs_host, float op_scale,
                              float op_shift, const int32_t* delta_row_host, const int32_t* delta_col_host,
                              const float* delta_val_host, int32_t n_delta, const egnn_peer_window* win,
                              egnn_stream_t stream) {
    return wide_adjoint_sharded_impl(rowptr_local, colidx_local, nullptr, row_order_or_null, dinv_full, iso_full,
                                     cbar_local, tbar_local_or_null, xbar_local, nullptr, n_global, row_begin, row_end,
                                     f, app, k_max, n_scales, coeffs_host, op_scale, op_shift, delta_row_host,
                                     delta_col_host, delta_val_host, n_delta, win, stream);
}

int egnn_wide_adjoint_sharded_all(const int32_t* rowptr_local, const int32_t* colidx_local, const float* vals_or_null,
                                  const int32_t* row_order_or_null, const float* dinv_full, const uint8_t* iso_full,
                                  const float* cbar_local, const float* tbar_local_or_null, float* xbar_local,
                                  float* b_out_local_or_null, int64_t n_global, int64_t row_begin, int64_t row_end,
                                  int32_t f, int32_t app, int32_t k_max, int32_t n_scales, const float* coeffs_host,
                                  float op_scale, float op_shift, const int32_t* delta_row_host,
                                  const int32_t* delta_col_host, const float* delta_val_host, int32_t n_delta,
                                  const egnn_peer_window* win, egnn_stream_t stream) {
    return wide_adjoint_sharded_impl(rowptr_local, colidx_local, vals_or_null, row_order_or_null, dinv_full, iso_full,
                                     cbar_local, tbar_local_or_null, xbar_local, b_out_local_or_null, n_global,
                                     row_begin, row_end, f, app, k_max, n_scales, coeffs_host, op_scale, op_shift,
                                     delta_row_host, delta_col_host, delta_val_host, n_delta, win, stream);
}

// ---- gradient w.r.t. the edge weights of a row shard (csrc/shard_grad.cuh) ---------------------------
// Lanes across the K*F / vec vectors of one entry: the next power of two, at most a warp.
static int shard_fl_log2(int64_t kf, int vec) {
    const int64_t nv = kf / vec;
    const int l = pow2_ceil_log2(nv > 1 ? nv : 1);
    return l > 5 ? 5 : l;
}

int egnn_adj_grad_stacks_sharded(const float* lam_all, int64_t lam_slab_rows, const float* t_all, int64_t t_slab_rows,
                                 const float* dinv_full, int64_t n_global, int64_t row_begin, int64_t row_end,
                                 int32_t f, int32_t k, float* pl_local, float* pt_local, egnn_stream_t stream) {
    EGNN_REQUIRE(n_global >= 0 && n_global < (int64_t(1) << 31) && row_begin >= 0 && row_end >= row_begin &&
                 row_end <= n_global, "bad row range");
    EGNN_REQUIRE(f >= 1 && k >= 0 && k <= EGNN_MAX_ORDER, "bad f / k");
    const int64_t rows = row_end - row_begin;
    EGNN_REQUIRE(lam_slab_rows >= rows && t_slab_rows >= rows, "slabs shorter than the rank's rows");
    if (rows == 0 || k == 0) return EGNN_OK;
    EGNN_REQUIRE(lam_all && t_all && dinv_full && pl_local && pt_local, "null pointer");
    shard_grad_stacks_kernel<<<grid_for(rows * k * f, 256), 256, 0, (cudaStream_t)stream>>>(
        lam_all, lam_slab_rows * f, t_all, t_slab_rows * f, dinv_full + row_begin, rows, f, k, pl_local, pt_local);
    EGNN_LAUNCH_CHECK("shard_grad_stacks_kernel launch");
    return EGNN_OK;
}

size_t egnn_adj_grad_degree_sharded_ws_bytes(int64_t rows) {
    return 2 * align_up(sizeof(double) * (size_t)(rows > 0 ? rows : 1), 256) + 256;
}

static int launch_shard_dot(const int32_t* rowptr, const int32_t* colidx, const float* vals, const int32_t* perm,
                            const float* own, const float* gath, int64_t rows, int64_t row0, int32_t kf,
                            double* out, float* g_out, cudaStream_t st) {
    const int vec = kf % 4 == 0 ? 4 : 1;
    const int fl = shard_fl_log2(kf, vec);
    const int blocks = grid_for(rows * 32, 256);
    if (vec == 4)
        shard_grad_dot_kernel<4><<<blocks, 256, 0, st>>>(rowptr, colidx, vals, perm, own, gath, rows, row0, kf, fl,
                                                          out, g_out);
    else
        shard_grad_dot_kernel<1><<<blocks, 256, 0, st>>>(rowptr, colidx, vals, perm, own, gath, rows, row0, kf, fl,
                                                          out, g_out);
    EGNN_LAUNCH_CHECK("shard_grad_dot_kernel launch");
    return EGNN_OK;
}

int egnn_adj_grad_degree_sharded(const int32_t* rowptr, const int32_t* colidx, const float* vals_or_null,
                                 const int32_t* row_order_or_null, const int32_t* rowptr_t, const int32_t* colidx_t,
                                 const float* vals_t_or_null, const int32_t* row_order_t_or_null,
                                 const float* dinv_full, const uint8_t* iso_full, int64_t n_global, int64_t row_begin,
                                 int64_t row_end, int32_t f, int32_t k, float op_scale, const float* pl_full,
                                 const float* pt_full, const float* xbar_local_or_null,
                                 const float* rowsum_local_or_null, float* g_out, float* gw_local, float* grho_local,
                                 void* workspace, size_t workspace_bytes, egnn_stream_t stream) {
    return egnn_adj_grad_degree_sharded_flips(rowptr, colidx, vals_or_null, row_order_or_null, rowptr_t, colidx_t,
                                              vals_t_or_null, row_order_t_or_null, dinv_full, iso_full, n_global,
                                              row_begin, row_end, f, k, op_scale, pl_full, pt_full,
                                              xbar_local_or_null, rowsum_local_or_null, nullptr, nullptr, nullptr, 0,
                                              nullptr, g_out, gw_local, grho_local, workspace, workspace_bytes,
                                              stream);
}

int egnn_adj_grad_degree_sharded_flips(const int32_t* rowptr, const int32_t* colidx, const float* vals_or_null,
                                       const int32_t* row_order_or_null, const int32_t* rowptr_t,
                                       const int32_t* colidx_t, const float* vals_t_or_null,
                                       const int32_t* row_order_t_or_null, const float* dinv_full,
                                       const uint8_t* iso_full, int64_t n_global, int64_t row_begin, int64_t row_end,
                                       int32_t f, int32_t k, float op_scale, const float* pl_full,
                                       const float* pt_full, const float* xbar_local_or_null,
                                       const float* rowsum_local_or_null, const int32_t* delta_row_host,
                                       const int32_t* delta_col_host, const float* delta_val_host, int32_t n_delta,
                                       float* g_flips_out, float* g_out, float* gw_local, float* grho_local,
                                       void* workspace, size_t workspace_bytes, egnn_stream_t stream) {
    DeltaList d;
    int rc = fill_delta(d, delta_row_host, delta_col_host, delta_val_host, n_delta, n_global);
    if (rc) return rc;
    EGNN_REQUIRE(d.n == 0 || g_flips_out, "null g_flips_out");
    EGNN_REQUIRE(rowptr && rowptr_t && dinv_full && iso_full && g_out && gw_local && grho_local, "null pointer");
    EGNN_REQUIRE(n_global >= 0 && n_global < (int64_t(1) << 31) && row_begin >= 0 && row_end >= row_begin &&
                 row_end <= n_global, "bad row range");
    EGNN_REQUIRE(f >= 1 && k >= 0 && k <= EGNN_MAX_ORDER, "bad f / k");
    EGNN_REQUIRE((vals_or_null == nullptr) == (vals_t_or_null == nullptr), "vals and vals_t come together");
    EGNN_REQUIRE(k == 0 || (pl_full && pt_full), "null lambda / T stacks");
    EGNN_REQUIRE((xbar_local_or_null == nullptr) || rowsum_local_or_null, "xbar needs rowsum");
    const int64_t kf = (int64_t)k * f;
    EGNN_REQUIRE(kf < (int64_t(1) << 31), "k * f out of int32 range");
    EGNN_REQUIRE(vec_aligned(pl_full, (int32_t)(kf % 4 == 0 ? 4 : 1)) && vec_aligned(pt_full, (int32_t)(kf % 4 == 0 ? 4 : 1)),
                 "the lambda / T stacks must be 16-byte aligned when k * f % 4 == 0");
    const int64_t rows = row_end - row_begin;
    rc = require_workspace(workspace, workspace_bytes, egnn_adj_grad_degree_sharded_ws_bytes(rows),
                           "adjacency-gradient workspace");
    if (rc) return rc;
    if (rows == 0) return EGNN_OK;    // a rank without rows: no term of its own (its flip values are all 0)
    cudaStream_t st = (cudaStream_t)stream;
    double* r = (double*)align_up((size_t)workspace, 256);
    double* q = (double*)((char*)r + align_up(sizeof(double) * (size_t)rows, 256));
    if (k == 0) {                     // no operator in the pass: g = 0, R = Q = 0, only grho
        rc = check_cuda(cudaMemsetAsync(r, 0, 2 * align_up(sizeof(double) * (size_t)rows, 256), st), "memset R, Q");
        if (rc) return rc;
        if (d.n > 0) {
            rc = check_cuda(cudaMemsetAsync(g_flips_out, 0, sizeof(float) * (size_t)d.n, st), "memset g_flips");
            if (rc) return rc;
        }
    } else {
        rc = launch_shard_dot(rowptr, colidx, vals_or_null, row_order_or_null, pl_full, pt_full, rows, row_begin,
                              (int32_t)kf, r, g_out, st);
        if (rc) return rc;
        rc = launch_shard_dot(rowptr_t, colidx_t, vals_t_or_null, row_order_t_or_null, pt_full, pl_full, rows,
                              row_begin, (int32_t)kf, q, nullptr, st);
        if (rc) return rc;
        if (d.n > 0) {
            const int vec = kf % 4 == 0 ? 4 : 1;
            const int fl = shard_fl_log2(kf, vec);
            if (vec == 4)
                shard_grad_flip_terms_kernel<4><<<1, 32 * kShardFlipWarps, 0, st>>>(d, pl_full, pt_full, rows,
                                                                                     row_begin, (int32_t)kf, fl,
                                                                                     g_flips_out, r, q);
            else
                shard_grad_flip_terms_kernel<1><<<1, 32 * kShardFlipWarps, 0, st>>>(d, pl_full, pt_full, rows,
                                                                                     row_begin, (int32_t)kf, fl,
                                                                                     g_flips_out, r, q);
            EGNN_LAUNCH_CHECK("shard_grad_flip_terms_kernel launch");
        }
    }
    adj_grad_finish_kernel<<<grid_for(rows, 256), 256, 0, st>>>(r, q, dinv_full + row_begin, iso_full + row_begin,
                                                                xbar_local_or_null, rowsum_local_or_null, rows,
                                                                op_scale, gw_local, grho_local);
    EGNN_LAUNCH_CHECK("adj_grad_finish_kernel launch");
    return EGNN_OK;
}

int egnn_adj_grad_entries_sharded(const int32_t* rowptr, const int32_t* colidx, int64_t n_global, int64_t row_begin,
                                  int64_t row_end, int32_t k, const float* g, const float* gw_full,
                                  const float* grho_local, float op_scale, float* out, egnn_stream_t stream) {
    EGNN_REQUIRE(n_global >= 0 && n_global < (int64_t(1) << 31) && row_begin >= 0 && row_end >= row_begin &&
                 row_end <= n_global, "bad row range");
    EGNN_REQUIRE(k >= 0 && k <= EGNN_MAX_ORDER, "bad k");
    const int64_t rows = row_end - row_begin;
    if (rows == 0) return EGNN_OK;   // a rank without rows: nothing to write (its buffers may be empty)
    EGNN_REQUIRE(rowptr && gw_full && grho_local && out, "null pointer");
    EGNN_REQUIRE(k == 0 || g, "null g");
    shard_grad_entries_kernel<<<grid_for(rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(
        rowptr, colidx, k == 0 ? nullptr : g, gw_full, grho_local, rows, row_begin, op_scale, out);
    EGNN_LAUNCH_CHECK("shard_grad_entries_kernel launch");
    return EGNN_OK;
}

int egnn_adj_grad_flips_sharded(const int32_t* delta_row_host, const int32_t* delta_col_host,
                                const float* delta_val_host, int32_t n_delta, const float* g_flips,
                                const float* gw_full, const float* grho_local, int64_t n_global, int64_t row_begin,
                                int64_t row_end, float op_scale, float* out, egnn_stream_t stream) {
    EGNN_REQUIRE(n_global >= 0 && n_global < (int64_t(1) << 31) && row_begin >= 0 && row_end >= row_begin &&
                 row_end <= n_global, "bad row range");
    DeltaList d;
    int rc = fill_delta(d, delta_row_host, delta_col_host, delta_val_host, n_delta, n_global);
    if (rc) return rc;
    if (d.n == 0) return EGNN_OK;
    EGNN_REQUIRE(g_flips && gw_full && grho_local && out, "null pointer");
    shard_grad_flip_values_kernel<<<1, EGNN_MAX_DELTA, 0, (cudaStream_t)stream>>>(
        d, g_flips, gw_full, grho_local, row_end - row_begin, row_begin, op_scale, out);
    EGNN_LAUNCH_CHECK("shard_grad_flip_values_kernel launch");
    return EGNN_OK;
}

int egnn_graph_prep_sharded(const int32_t* rowptr_local, const int32_t* colidx_local, const float* vals_or_null,
                            int64_t n_global, int64_t row_begin, int64_t n_rows, int32_t phase,
                            double* colsum_full, float* diag_full, float* rowsum_local, float* dinv_full,
                            uint8_t* iso_full, float* x0_local, int32_t* unsorted_flag_or_null,
                            float* w_full_or_null, egnn_stream_t stream) {
    EGNN_REQUIRE(colsum_full && diag_full && rowsum_local, "null pointer");
    EGNN_REQUIRE(n_global >= 0 && row_begin >= 0 && n_rows >= 0 && row_begin + n_rows <= n_global, "bad row range");
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if (phase == 0) {      // local rows: row sums, diagonal, partial in-degree (caller all-reduces colsum/diag)
        EGNN_REQUIRE(rowptr_local != nullptr, "null rowptr");
        rc = check_cuda(cudaMemsetAsync(colsum_full, 0, sizeof(double) * n_global, st), "memset colsum"); if (rc) return rc;
        rc = check_cuda(cudaMemsetAsync(diag_full, 0, sizeof(float) * n_global, st), "memset diag"); if (rc) return rc;
        if (unsorted_flag_or_null) {
            rc = check_cuda(cudaMemsetAsync(unsorted_flag_or_null, 0, sizeof(int32_t), st), "memset flag"); if (rc) return rc;
        }
        if (n_rows == 0) return EGNN_OK;
        return launch_degree(rowptr_local, colidx_local, vals_or_null, n_rows, rowsum_local, diag_full + row_begin,
                             colsum_full, unsorted_flag_or_null, row_begin, st);
    }
    EGNN_REQUIRE(phase == 1 && dinv_full && iso_full, "bad phase or null outputs");
    if (n_global > 0) {    // after the all-reduce: normaliser of every node, x0 of the local rows
        normaliser_kernel<<<(unsigned)ceil_div64(n_global, 256), 256, 0, st>>>(colsum_full, diag_full, nullptr, n_global,
                                                                            dinv_full, iso_full, nullptr, w_full_or_null);
        EGNN_LAUNCH_CHECK("normaliser_kernel launch");
    }
    if (x0_local && n_rows > 0) {
        logdeg_kernel<<<(unsigned)ceil_div64(n_rows, 256), 256, 0, st>>>(rowsum_local, n_rows, x0_local);
        EGNN_LAUNCH_CHECK("logdeg_kernel launch");
    }
    return EGNN_OK;
}

// ---- sparse structure-gradient surrogate (surrogate.cuh) -------------------------
static int gcn_check(const int32_t* rowptr, int64_t n, int32_t h) {
    EGNN_REQUIRE(rowptr != nullptr, "null rowptr");
    EGNN_REQUIRE(n >= 1 && n < (int64_t(1) << 31), "n out of range");
    EGNN_REQUIRE(h >= 4 && h <= kGcnMaxHidden && h % 4 == 0, "hidden width must be a multiple of 4 in [4, 128]");
    return EGNN_OK;
}

int egnn_gcn_propagate(const int32_t* rowptr, const int32_t* colidx, const float* vals_or_null, const float* m,
                       const float* bias_or_null, float* y, float* deg_out_or_null, int64_t n, int32_t h,
                       const int32_t* delta_row_host, const int32_t* delta_col_host, const float* delta_val_host,
                       int32_t n_delta, egnn_stream_t stream) {
    int rc = gcn_check(rowptr, n, h);
    if (rc) return rc;
    EGNN_REQUIRE(m && y, "null pointer");
    EGNN_REQUIRE(vec_aligned(m, h) && vec_aligned(bias_or_null, h) && vec_aligned(y, h),
                 "m, bias and y must be 16-byte aligned");
    DeltaList d;
    rc = fill_delta(d, delta_row_host, delta_col_host, delta_val_host, n_delta, n);
    if (rc) return rc;
    const unsigned grid = (unsigned)ceil_div64(n * 32, 256);
    if (vals_or_null)
        gcn_propagate_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(rowptr, colidx, vals_or_null, m, bias_or_null, y,
                                                                           deg_out_or_null, n, h, d);
    else
        gcn_propagate_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(rowptr, colidx, nullptr, m, bias_or_null, y,
                                                                            deg_out_or_null, n, h, d);
    EGNN_LAUNCH_CHECK("gcn_propagate_kernel launch");
    return EGNN_OK;
}

int egnn_gcn_target_logits(const int32_t* rowptr, const int32_t* colidx, const float* vals_or_null, const float* z1,
                           const float* w2, const float* b2, int32_t target, int64_t n, int32_t h, int32_t n_classes,
                           float* logits_out, float* ctx, const int32_t* delta_row_host, const int32_t* delta_col_host,
                           const float* delta_val_host, int32_t n_delta, egnn_stream_t stream) {
    int rc = gcn_check(rowptr, n, h);
    if (rc) return rc;
    EGNN_REQUIRE(z1 && w2 && b2 && logits_out && ctx, "null pointer");
    EGNN_REQUIRE(vec_aligned(z1, h), "z1 must be 16-byte aligned");
    EGNN_REQUIRE(target >= 0 && target < n && n_classes >= 1, "bad target / classes");
    DeltaList d;
    rc = fill_delta(d, delta_row_host, delta_col_host, delta_val_host, n_delta, n);
    if (rc) return rc;
    if (vals_or_null)
        gcn_target_logits_kernel<true><<<1, 256, 0, (cudaStream_t)stream>>>(rowptr, colidx, vals_or_null, z1, w2, b2, target, h,
                                                                            n_classes, logits_out, ctx, d);
    else
        gcn_target_logits_kernel<false><<<1, 256, 0, (cudaStream_t)stream>>>(rowptr, colidx, nullptr, z1, w2, b2, target, h,
                                                                             n_classes, logits_out, ctx, d);
    EGNN_LAUNCH_CHECK("gcn_target_logits_kernel launch");
    return EGNN_OK;
}

int egnn_gcn_structure_grad(const int32_t* rowptr, const int32_t* colidx, const float* vals_or_null,
                            const float* upstream, const float* w2, const float* z1, const float* xw, const float* b1,
                            const float* deg, const float* ctx, int32_t target, int64_t n, int32_t h, int32_t n_classes,
                            float* grad_row, float* grad_col, const int32_t* delta_row_host,
                            const int32_t* delta_col_host, const float* delta_val_host, int32_t n_delta,
                            egnn_stream_t stream) {
    int rc = gcn_check(rowptr, n, h);
    if (rc) return rc;
    EGNN_REQUIRE(upstream && w2 && z1 && xw && b1 && deg && ctx && grad_row && grad_col, "null pointer");
    EGNN_REQUIRE(vec_aligned(z1, h) && vec_aligned(xw, h), "z1 and xw must be 16-byte aligned");
    EGNN_REQUIRE(target >= 0 && target < n && n_classes >= 1, "bad target / classes");
    DeltaList d;
    rc = fill_delta(d, delta_row_host, delta_col_host, delta_val_host, n_delta, n);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    rc = check_cuda(cudaMemsetAsync(grad_col, 0, sizeof(float) * n, st), "memset grad_col");
    if (rc) return rc;
    gcn_grad_row_kernel<<<grid_for(n * 8, 256), 256, 0, st>>>(upstream, w2, z1, xw, b1, ctx, target, n, h, n_classes, grad_row);
    EGNN_LAUNCH_CHECK("gcn_grad_row_kernel launch");
    if (vals_or_null)
        gcn_grad_col_kernel<true><<<1, 256, 0, st>>>(rowptr, colidx, vals_or_null, upstream, w2, z1, xw, b1, deg, ctx, grad_row,
                                                     target, h, n_classes, grad_col, d);
    else
        gcn_grad_col_kernel<false><<<1, 256, 0, st>>>(rowptr, colidx, nullptr, upstream, w2, z1, xw, b1, deg, ctx, grad_row,
                                                      target, h, n_classes, grad_col, d);
    EGNN_LAUNCH_CHECK("gcn_grad_col_kernel launch");
    return EGNN_OK;
}

int egnn_prescale(const float* x, const float* dinv_full, float* y, int64_t n_rows, int32_t f, int64_t row0,
                  egnn_stream_t stream) {
    EGNN_REQUIRE(x && dinv_full && y, "null pointer");
    EGNN_REQUIRE(n_rows >= 0 && f >= 1 && row0 >= 0, "bad shape");
    if (n_rows == 0) return EGNN_OK;
    prescale_kernel<<<grid_for(n_rows * f, 256), 256, 0, (cudaStream_t)stream>>>(x, dinv_full, y, n_rows, f, row0);
    EGNN_LAUNCH_CHECK("prescale_kernel launch");
    return EGNN_OK;
}

}  // extern "C"

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

static int fill_delta(DeltaList& d, const int32_t* r, const int32_t* c, const float* v, int32_t n) {
    EGNN_REQUIRE(n >= 0 && n <= EGNN_MAX_DELTA, "n_delta out of range");
    EGNN_REQUIRE(n == 0 || (r && c && v), "delta arrays missing");
    d.n = n;
    for (int i = 0; i < n; ++i) { d.row[i] = r[i]; d.col[i] = c[i]; d.val[i] = v[i]; }
    return EGNN_OK;
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

// PEER instantiation: operand in the exchange window, written by the other GPUs (world > 1).
// The adjoint (ADJ) runs on one GPU only.
template <int NZ_LOG2, bool ADJ>
static int launch_wide_n(const WideParams& p, dim3 grid, cudaStream_t st) {
    if constexpr (ADJ) return launch_wide_np<NZ_LOG2, false, true>(p, grid, st);
    else return p.peer.world > 1 ? launch_wide_np<NZ_LOG2, true, false>(p, grid, st)
                                 : launch_wide_np<NZ_LOG2, false, false>(p, grid, st);
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
    sp.cta_info = pl->cta_info; sp.rv_ptr = pl->rv_ptr; sp.vpart = pl->vpart; sp.sched = pl->sched;
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

int egnn_abi_version(void) { return 7; }

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
    cudaStream_t st = (cudaStream_t)stream;
    const int g = grid_for(rows * 32, 256);
    // rowptr values are absolute positions in colidx, so a row range is the same kernel on shifted row arrays
    if (vals_or_null)
        degree_kernel<true><<<g, 256, 0, st>>>(rowptr + row_begin, colidx, vals_or_null, rows, rowsum + row_begin,
                                               diag + row_begin, colsum, unsorted_flag_or_null, row_begin);
    else
        degree_kernel<false><<<g, 256, 0, st>>>(rowptr + row_begin, colidx, nullptr, rows, rowsum + row_begin,
                                                diag + row_begin, colsum, unsorted_flag_or_null, row_begin);
    EGNN_LAUNCH_CHECK("degree_kernel launch");
    return EGNN_OK;
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
    int rc = fill_delta(d, delta_row_host, delta_col_host, delta_val_host, n_delta);
    if (rc) return rc;
    for (int i = 0; i < n_delta; ++i)
        EGNN_REQUIRE(d.row[i] >= 0 && d.row[i] < n && d.col[i] >= 0 && d.col[i] < n, "delta index out of range");
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
    int rc = fill_delta(d, delta_row_host, delta_col_host, delta_val_host, n_delta);
    if (rc) return rc;
    for (int i = 0; i < n_delta; ++i)
        EGNN_REQUIRE(d.row[i] >= 0 && d.row[i] < n && d.col[i] >= 0 && d.col[i] < n, "delta index out of range");
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
    const size_t need = egnn_row_order_ws_bytes(n);
    if (!workspace || workspace_bytes < need) {
        set_error("row-order workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
        return EGNN_ERR_WORKSPACE;
    }
    const size_t arr = align_up(4 * (size_t)n, 256);
    char* ws = (char*)align_up((size_t)workspace, 256);
    uint32_t* keys = (uint32_t*)ws;
    uint32_t* keys_sorted = (uint32_t*)(ws + arr);
    int32_t* ids = (int32_t*)(ws + 2 * arr);
    void* cub_temp = ws + 3 * arr;
    size_t cub_bytes = row_order_cub_bytes(n);
    row_order_keys_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, st>>>(rowptr, (int)n, keys, ids);
    EGNN_LAUNCH_CHECK("row_order_keys_kernel launch");
    int rc = check_cuda(cub::DeviceRadixSort::SortPairs(cub_temp, cub_bytes, keys, keys_sorted, ids, order_out, (int)n, 0,
                                                        32, st), "sort rows by degree");
    if (rc) return rc;
    row_order_hubs_kernel<<<1, 32, 0, st>>>(keys_sorted, (int)n, order_out + n);
    EGNN_LAUNCH_CHECK("row_order_hubs_kernel launch");
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

static size_t blocked_ws_bytes(int64_t n) {
    int C = 1, CB = 32;
    narrow_geometry(n > 0 ? n : 1, &C, &CB);
    return align_up(4 * (size_t)(C + 1) * (size_t)n, 256) + align_up(4 * (size_t)C * (size_t)n, 256) +
           align_up(4 * (size_t)EGNN_MAX_ORDER * (size_t)C, 256);
}

size_t egnn_cheb_workspace_bytes(int64_t n, int32_t f) {
    // two T ping-pong slabs + two pre-scaled gather slabs (narrow F only)
    // f <= 4: two T slabs + two pre-scaled slabs; 4 < f < 8: two T slabs; f >= 8: two pre-scaled slabs
    const size_t width = f >= kWideMinF ? (size_t)((f + 3) / 4 * 4) : (size_t)f;     // wide slabs have 16-byte rows
    const size_t slab = align_up(sizeof(float) * (size_t)n * width, 256);
    // wide path: + one row counter per (order, feature tile) for the dynamic row schedule
    const size_t counters = f >= kWideMinF ? align_up(sizeof(unsigned) * (size_t)EGNN_MAX_ORDER * (size_t)((width + 127) / 128), 256) : 0;
    // f == 1: + segment table, partial sums and counters of the plan-free blocked kernel
    return slab * (f <= 4 ? 4 : 2) + counters + (f == 1 ? blocked_ws_bytes(n) : 0) + 256;
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
    cudaStream_t st = (cudaStream_t)stream;

    OrderParams p{};
    int rc = fill_delta(p.delta, delta_row_host, delta_col_host, delta_val_host, n_delta);
    if (rc) return rc;
    for (int i = 0; i < n_delta; ++i)
        EGNN_REQUIRE(p.delta.row[i] >= 0 && p.delta.row[i] < n && p.delta.col[i] >= 0 && p.delta.col[i] < n,
                     "delta index out of range");

    const size_t slab_elems = (size_t)n * (size_t)f;
    if (k == 0) {
        for (int s = 0; s < n_scales; ++s) p.c_prev[s] = coeffs_host[s];
        order0_kernel<<<grid_for((int64_t)slab_elems * n_scales, 256), 256, 0, st>>>(x0, out, n, f, n_scales, p);
        EGNN_LAUNCH_CHECK("order0_kernel launch");
        if (t_all_or_null) {
            rc = check_cuda(cudaMemcpyAsync(t_all_or_null, x0, sizeof(float) * slab_elems, cudaMemcpyDeviceToDevice, st), "copy T0");
            if (rc) return rc;
        }
        if (normalize_l1) {
            l1_normalize_kernel<<<grid_for(n * n_scales * 32, 256), 256, 0, st>>>(out, n * n_scales, f);
            EGNN_LAUNCH_CHECK("l1_normalize_kernel launch");
        }
        return EGNN_OK;
    }

    const OrderConfig cfg = choose_config(n, nnz, f);
    const size_t need = egnn_cheb_workspace_bytes(n, f);
    if (workspace == nullptr || workspace_bytes < need) {
        set_error("workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
        return EGNN_ERR_WORKSPACE;
    }
    const size_t slab = align_up(sizeof(float) * slab_elems, 256);
    char* ws = (char*)align_up((size_t)workspace, 256);
    float* tbuf[2] = {(float*)ws, (float*)(ws + slab)};
    float* ybuf[2] = {(float*)(ws + 2 * slab), (float*)(ws + 3 * slab)};

    if (t_all_or_null) {
        rc = check_cuda(cudaMemcpyAsync(t_all_or_null, x0, sizeof(float) * slab_elems, cudaMemcpyDeviceToDevice, st), "copy T0");
        if (rc) return rc;
    }
    if (cfg.prescaled && !sell_plan) {
        prescale_kernel<<<grid_for((int64_t)slab_elems, 256), 256, 0, st>>>(x0, dinv, ybuf[0], n, f, 0);
        EGNN_LAUNCH_CHECK("prescale_kernel launch");
    }

    if (sell_plan) {
        EGNN_REQUIRE(f == 1 && vals_or_null == nullptr, "the SELL plan serves F = 1 on a binary adjacency");
        EGNN_REQUIRE(sell_plan->n == n && sell_plan->n_cols == n && sell_plan->row0 == 0 && sell_plan->vpart && sell_plan->slice_off && sell_plan->blk_slice_ptr &&
                     sell_plan->rv_ptr && sell_plan->vslot && sell_plan->cta_info && sell_plan->sched, "SELL plan does not match the graph or is not filled");
        // all K orders in one persistent launch (sell_step.cuh); the first operand dinv (.) T_0 is
        // computed inside it
        SellStepParams sp{};
        step_fill_plan(sp, sell_plan);
        sp.delta = p.delta;
        sp.w_base = w_base_or_null; sp.rowsum_base = rowsum_base_or_null; sp.patch_x0 = default_signal ? 1 : 0;
        sp.dinv = dinv; sp.iso = iso; sp.x0 = x0;
        sp.operand_first = y0_or_null;       // dinv (.) T_0 kept by the caller (fixed per graph for the default signal)
        sp.operand[0] = ybuf[0]; sp.operand[1] = ybuf[1];
        sp.ydst[0][0] = ybuf[0]; sp.ydst[1][0] = ybuf[1]; sp.n_dst = 1;
        sp.tbuf[0] = tbuf[0]; sp.tbuf[1] = tbuf[1]; sp.t_all = t_all_or_null; sp.out = out;
        sp.normalize = normalize_l1; sp.a = op_scale; sp.b = op_shift;
        sp.world = 1; sp.rank = 0; sp.rows_per = n;
        if (order_events_host) {
            rc = check_cuda(cudaEventRecord((cudaEvent_t)order_events_host[0], st), "event record");
            if (rc) return rc;
        }
        rc = run_sell_step(sp, k, n_scales, coeffs_host, false, st);
        if (rc) return rc;
        if (order_events_host) {                      // one launch: events 0 and 1 bracket the whole step, the rest follow it
            for (int e = 1; e < 2 * k; ++e) {
                rc = check_cuda(cudaEventRecord((cudaEvent_t)order_events_host[e], st), "event record");
                if (rc) return rc;
            }
        }
        return EGNN_OK;
    }

    if (f == 1 && rows_sorted && (nnz >= kBlockedMinNnz || rows_sorted == 2) && nnz > 0) {
        // first use of a large graph (no SELL plan yet): plan-free column-blocked kernel (blocked.cuh)
        int C = 1, CB = 32;
        narrow_geometry(n, &C, &CB);
        char* extra = ws + 4 * slab;
        int32_t* seg = (int32_t*)extra;
        float* part = (float*)(extra + align_up(4 * (size_t)(C + 1) * (size_t)n, 256));
        unsigned* counters = (unsigned*)((char*)part + align_up(4 * (size_t)C * (size_t)n, 256));
        rc = check_cuda(cudaMemsetAsync(counters, 0, sizeof(unsigned) * (size_t)k * (size_t)C, st), "memset batch counters");
        if (rc) return rc;
        blocked_bounds_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, st>>>(rowptr, colidx, (int)n, C, CB, seg);
        EGNN_LAUNCH_CHECK("blocked_bounds_kernel launch");
        const size_t smem = sizeof(float) * (size_t)CB;
        const void* fn = vals_or_null ? (const void*)blocked_spmv_kernel<true> : (const void*)blocked_spmv_kernel<false>;
        rc = check_cuda(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                        "cudaFuncSetAttribute(blocked_spmv_kernel)");
        if (rc) return rc;
        BlockedParams bp{};
        bp.colidx = colidx; bp.vals = vals_or_null; bp.seg = seg; bp.part = part;
        bp.n = (int32_t)n; bp.C = C; bp.CB = CB; bp.n_cta = device_sm_count();
        if (bp.n_cta < C) bp.n_cta = C;
        BlockedEpilogueParams ep{};
        ep.delta = p.delta;
        ep.part = part; ep.dinv = dinv; ep.iso = iso; ep.out = out; ep.n = (int32_t)n; ep.C = C; ep.S = n_scales;
        ep.a = op_scale; ep.b = op_shift;
        const float* t_prev = x0;
        const float* t_prev2 = nullptr;
        for (int order = 1; order <= k; ++order) {
            const bool last = order == k;
            float* t_out;
            if (t_all_or_null) t_out = t_all_or_null + (size_t)order * slab_elems;
            else if (last) t_out = nullptr;
            else if (order == 1) t_out = tbuf[0];
            else if (order == 2) t_out = tbuf[1];
            else t_out = const_cast<float*>(t_prev2);
            if (order_events_host) {
                rc = check_cuda(cudaEventRecord((cudaEvent_t)order_events_host[2 * (order - 1)], st), "event record");
                if (rc) return rc;
            }
            bp.y = ybuf[(order - 1) & 1];
            bp.counter = counters + (size_t)(order - 1) * C;
            if (vals_or_null) blocked_spmv_kernel<true><<<bp.n_cta, kBlockedThreads, smem, st>>>(bp);
            else blocked_spmv_kernel<false><<<bp.n_cta, kBlockedThreads, smem, st>>>(bp);
            EGNN_LAUNCH_CHECK("blocked_spmv_kernel launch");
            ep.y_prev = bp.y; ep.tprev = t_prev; ep.tprev2 = t_prev2; ep.tk = t_out;
            ep.y_out = last ? nullptr : ybuf[order & 1];
            ep.first = order == 1; ep.normalize = last && normalize_l1;
            for (int s = 0; s < n_scales; ++s) {
                ep.c_prev[s] = coeffs_host[s * (k + 1) + order - 1];
                ep.c_k[s] = coeffs_host[s * (k + 1) + order];
            }
            blocked_epilogue_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, st>>>(ep);
            EGNN_LAUNCH_CHECK("blocked_epilogue_kernel launch");
            if (order_events_host) {
                rc = check_cuda(cudaEventRecord((cudaEvent_t)order_events_host[2 * (order - 1) + 1], st), "event record");
                if (rc) return rc;
            }
            t_prev2 = t_prev;
            t_prev = t_out;
        }
        return EGNN_OK;
    }

    if (f >= kWideMinF) {
        const int ldy = (f + 3) / 4 * 4;
        const RingConfig rcfg = ring_config(ldy);
        const size_t yslab = align_up(sizeof(float) * (size_t)n * (size_t)ldy, 256);
        float* yb[2] = {(float*)ws, (float*)(ws + yslab)};       // the two slabs hold dinv (.) T_k, rows padded to 16 bytes
        WideParams wp{};
        wp.delta = p.delta;
        wp.rowptr = rowptr; wp.colidx = colidx; wp.vals = vals_or_null;
        wp.perm = row_order_or_null; wp.n_hub = row_order_or_null ? row_order_or_null + n : nullptr;
        wp.dinv = dinv; wp.iso = iso; wp.out = out; wp.n_rows = n; wp.row0 = 0; wp.F = f; wp.ldy = ldy; wp.S = n_scales;
        wp.a = op_scale; wp.b = op_shift;
        prescale_pad_kernel<<<grid_for((int64_t)n * ldy, 256), 256, 0, st>>>(x0, dinv, yb[0], n, f, ldy, 0);
        EGNN_LAUNCH_CHECK("prescale_pad_kernel launch");
        unsigned* counters = (unsigned*)(ws + 2 * yslab);          // [k][grid_y], zeroed once per call
        rc = check_cuda(cudaMemsetAsync(counters, 0, sizeof(unsigned) * (size_t)k * (size_t)rcfg.grid_y, st), "memset row counters");
        if (rc) return rc;
        const bool fuse_norm_w = normalize_l1 && rcfg.grid_y == 1;
        const int sms = device_sm_count();
        for (int order = 1; order <= k; ++order) {
            const bool last = order == k;
            wp.first = order == 1;
            wp.normalize = last && fuse_norm_w;
            // dynamic rows pay off where rows are short and one feature tile covers the signal (arxiv
            // shape F = 128: 0.283 -> 0.23 ms per order); measured slower on long rows (Reddit shape
            // F = 64: 2.13 -> 2.48) and on many feature tiles (Physics F = 8415: 2.77 -> 3.3)
            const bool dynamic_rows = rcfg.grid_y == 1 && nnz < (int64_t)kWideDynamicMaxDegree * n;
            wp.row_counter = dynamic_rows ? counters + (size_t)(order - 1) * (size_t)rcfg.grid_y : nullptr;
            wp.ysrc = yb[(order - 1) & 1];
            wp.x0_own = order == 1 ? x0 : nullptr;
            wp.y2_own = order == 1 ? nullptr : yb[order & 1];
            wp.y_out = last ? nullptr : yb[order & 1];      // in place over dinv (.) T_{k-2} (own row only)
            wp.tk_out = t_all_or_null ? t_all_or_null + (size_t)order * slab_elems : nullptr;
            for (int s = 0; s < n_scales; ++s) {
                wp.c_prev[s] = coeffs_host[s * (k + 1) + order - 1];
                wp.c_k[s] = coeffs_host[s * (k + 1) + order];
            }
            if (order_events_host) {
                rc = check_cuda(cudaEventRecord((cudaEvent_t)order_events_host[2 * (order - 1)], st), "event record");
                if (rc) return rc;
            }
            rc = launch_wide(wp, rcfg, sms, st);
            if (rc) return rc;
            if (order_events_host) {
                rc = check_cuda(cudaEventRecord((cudaEvent_t)order_events_host[2 * (order - 1) + 1], st), "event record");
                if (rc) return rc;
            }
        }
        if (normalize_l1 && !fuse_norm_w) {
            l1_normalize_kernel<<<grid_for(n * n_scales * 32, 256), 256, 0, st>>>(out, n * n_scales, f);
            EGNN_LAUNCH_CHECK("l1_normalize_kernel launch");
        }
        return EGNN_OK;
    }

    p.rowptr = rowptr; p.colidx = colidx; p.vals = vals_or_null; p.dinv = dinv; p.iso = iso;
    p.out = out; p.acc_ws = nullptr; p.n_rows = n; p.row0 = 0; p.F = f; p.S = n_scales;
    p.a = op_scale; p.b = op_shift; p.mode = 0; p.fl_log2 = cfg.fl_log2; p.nz_log2 = cfg.nz_log2;

    const bool fuse_norm = normalize_l1 && cfg.grid_y == 1;
    const float* t_prev = x0;         // T_{k-1}
    const float* t_prev2 = nullptr;   // T_{k-2}
    for (int order = 1; order <= k; ++order) {
        const bool last = order == k;
        float* t_out;
        if (t_all_or_null) t_out = t_all_or_null + (size_t)order * slab_elems;
        else if (last) t_out = nullptr;                       // T_K itself is never read again
        else if (order == 1) t_out = tbuf[0];
        else if (order == 2) t_out = tbuf[1];
        else t_out = const_cast<float*>(t_prev2);             // overwrite T_{k-2} in place
        p.first = order == 1;
        p.normalize = last && fuse_norm;
        p.tprev_own = t_prev;
        p.tprev2_own = t_prev2;
        p.tk_own = t_out;
        p.gsrc = cfg.prescaled ? ybuf[(order - 1) & 1] : t_prev;
        p.y_own = (cfg.prescaled && !last) ? ybuf[order & 1] : nullptr;
        for (int s = 0; s < n_scales; ++s) {
            p.c_prev[s] = coeffs_host[s * (k + 1) + order - 1];
            p.c_k[s] = coeffs_host[s * (k + 1) + order];
        }
        if (order_events_host) {
            rc = check_cuda(cudaEventRecord((cudaEvent_t)order_events_host[2 * (order - 1)], st), "event record");
            if (rc) return rc;
        }
        rc = launch_order(p, cfg, st);
        if (rc) return rc;
        if (order_events_host) {
            rc = check_cuda(cudaEventRecord((cudaEvent_t)order_events_host[2 * (order - 1) + 1], st), "event record");
            if (rc) return rc;
        }
        t_prev2 = t_prev;
        t_prev = t_out;
    }
    if (normalize_l1 && !fuse_norm) {
        l1_normalize_kernel<<<grid_for(n * n_scales * 32, 256), 256, 0, st>>>(out, n * n_scales, f);
        EGNN_LAUNCH_CHECK("l1_normalize_kernel launch");
    }
    return EGNN_OK;
}

// ---- backward of the wavelet pass (csrc/adjoint.cuh) ------------------------------------------------
int egnn_cheb_adjoint(const int32_t* rowptr_t, const int32_t* colidx_t, const float* vals_t_or_null,
                      const float* dinv, const uint8_t* iso, int64_t n, int64_t nnz, int32_t f, int32_t k,
                      int32_t n_scales, const float* coeffs_host, float op_scale, float op_shift,
                      const float* cbar, const float* tbar_or_null, float* xbar,
                      const int32_t* delta_row_host, const int32_t* delta_col_host,
                      const float* delta_val_host, int32_t n_delta, void* workspace,
                      size_t workspace_bytes, egnn_stream_t stream, void* const* app_events_host,
                      const int32_t* row_order_or_null) {
    EGNN_REQUIRE(rowptr_t && dinv && iso && cbar && xbar && coeffs_host, "null pointer");
    EGNN_REQUIRE(nnz == 0 || colidx_t, "null colidx");
    EGNN_REQUIRE(n >= 0 && n < (int64_t(1) << 31) && nnz >= 0 && nnz < (int64_t(1) << 31), "n/nnz out of int32 range");
    EGNN_REQUIRE(f >= 1, "f must be >= 1");
    EGNN_REQUIRE(k >= 0 && k <= EGNN_MAX_ORDER, "k out of range");
    EGNN_REQUIRE(n_scales >= 1 && n_scales <= EGNN_MAX_SCALES, "n_scales out of range");
    EGNN_REQUIRE(vec_aligned(cbar, f) && vec_aligned(tbar_or_null, f) && vec_aligned(xbar, f),
                 "cbar, tbar and xbar must be 16-byte aligned when f % 4 == 0");
    if (n == 0) return EGNN_OK;
    cudaStream_t st = (cudaStream_t)stream;
    OrderParams p{};
    int rc = fill_delta(p.delta, delta_row_host, delta_col_host, delta_val_host, n_delta);
    if (rc) return rc;
    for (int i = 0; i < n_delta; ++i)
        EGNN_REQUIRE(p.delta.row[i] >= 0 && p.delta.row[i] < n && p.delta.col[i] >= 0 && p.delta.col[i] < n,
                     "delta index out of range");
    const size_t slab_elems = (size_t)n * (size_t)f;
    auto coef_row = [&](int m) {
        CoefRow c{};
        for (int s = 0; s < n_scales; ++s) c.c[s] = coeffs_host[s * (k + 1) + m];
        return c;
    };
    auto tbar_at = [&](int m) { return tbar_or_null ? tbar_or_null + (size_t)m * slab_elems : nullptr; };
    if (k == 0) {
        adjoint_prologue_kernel<<<grid_for((int64_t)slab_elems, 256), 256, 0, st>>>(
            cbar, tbar_at(0), dinv, xbar, nullptr, n, f, n_scales, f, coef_row(0));
        EGNN_LAUNCH_CHECK("adjoint_prologue_kernel launch");
        return EGNN_OK;
    }
    const size_t need = egnn_cheb_workspace_bytes(n, f);
    if (workspace == nullptr || workspace_bytes < need) {
        set_error("workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
        return EGNN_ERR_WORKSPACE;
    }
    char* ws = (char*)align_up((size_t)workspace, 256);
    // application j = 1..K produces b_m, m = K - j (b_0 = the signal's gradient)
    if (f >= kWideMinF) {
        const int ldy = (f + 3) / 4 * 4;
        const RingConfig rcfg = ring_config(ldy);
        const size_t yslab = align_up(sizeof(float) * (size_t)n * (size_t)ldy, 256);
        float* yb[2] = {(float*)ws, (float*)(ws + yslab)};        // dinv (.) b, rows padded to 16 bytes
        unsigned* counters = (unsigned*)(ws + 2 * yslab);
        rc = check_cuda(cudaMemsetAsync(counters, 0, sizeof(unsigned) * (size_t)k * (size_t)rcfg.grid_y, st), "memset row counters");
        if (rc) return rc;
        adjoint_prologue_kernel<<<grid_for((int64_t)n * ldy, 256), 256, 0, st>>>(
            cbar, tbar_at(k), dinv, nullptr, yb[0], n, f, n_scales, ldy, coef_row(k));
        EGNN_LAUNCH_CHECK("adjoint_prologue_kernel launch");
        WideParams wp{};
        wp.delta = p.delta;
        wp.rowptr = rowptr_t; wp.colidx = colidx_t; wp.vals = vals_t_or_null;
        wp.perm = row_order_or_null; wp.n_hub = row_order_or_null ? row_order_or_null + n : nullptr;
        wp.dinv = dinv; wp.iso = iso; wp.out = nullptr; wp.n_rows = n; wp.row0 = 0; wp.F = f; wp.ldy = ldy;
        wp.S = n_scales; wp.a = op_scale; wp.b = op_shift; wp.first = 0; wp.normalize = 0;
        wp.cbar = cbar; wp.x0_own = nullptr;
        const bool dynamic_rows = rcfg.grid_y == 1 && nnz < (int64_t)kWideDynamicMaxDegree * n;   // as the forward
        const int sms = device_sm_count();
        for (int j = 1; j <= k; ++j) {
            const int m = k - j;
            wp.row_counter = dynamic_rows ? counters + (size_t)(j - 1) * (size_t)rcfg.grid_y : nullptr;
            wp.ysrc = yb[(j - 1) & 1];
            wp.y2_own = j == 1 ? nullptr : yb[j & 1];
            wp.y_out = m == 0 ? nullptr : yb[j & 1];             // in place over dinv (.) b_{m+2} (own row only)
            wp.tk_out = m == 0 ? xbar : nullptr;
            wp.tbar = tbar_at(m);
            wp.c_adj = m == 0 ? 1.f : 2.f;
            for (int s = 0; s < n_scales; ++s) wp.c_k[s] = coeffs_host[s * (k + 1) + m];
            if (app_events_host) {
                rc = check_cuda(cudaEventRecord((cudaEvent_t)app_events_host[2 * (j - 1)], st), "event record");
                if (rc) return rc;
            }
            rc = launch_wide<true>(wp, rcfg, sms, st);
            if (rc) return rc;
            if (app_events_host) {
                rc = check_cuda(cudaEventRecord((cudaEvent_t)app_events_host[2 * (j - 1) + 1], st), "event record");
                if (rc) return rc;
            }
        }
        return EGNN_OK;
    }
    const OrderConfig cfg = choose_config(n, nnz, f);
    const size_t slab = align_up(sizeof(float) * slab_elems, 256);
    float* tbuf[2] = {(float*)ws, (float*)(ws + slab)};
    float* ybuf[2] = {(float*)(ws + 2 * slab), (float*)(ws + 3 * slab)};
    adjoint_prologue_kernel<<<grid_for((int64_t)slab_elems, 256), 256, 0, st>>>(
        cbar, tbar_at(k), dinv, tbuf[0], cfg.prescaled ? ybuf[0] : nullptr, n, f, n_scales, f, coef_row(k));
    EGNN_LAUNCH_CHECK("adjoint_prologue_kernel launch");
    p.rowptr = rowptr_t; p.colidx = colidx_t; p.vals = vals_t_or_null; p.dinv = dinv; p.iso = iso;
    p.out = nullptr; p.acc_ws = nullptr; p.n_rows = n; p.row0 = 0; p.F = f; p.S = n_scales;
    p.a = op_scale; p.b = op_shift; p.mode = 0; p.fl_log2 = cfg.fl_log2; p.nz_log2 = cfg.nz_log2;
    p.first = 0; p.normalize = 0; p.cbar = cbar;
    for (int j = 1; j <= k; ++j) {
        const int m = k - j;
        p.tprev_own = tbuf[(j - 1) & 1];
        p.tprev2_own = j == 1 ? nullptr : tbuf[j & 1];
        p.tk_own = m == 0 ? xbar : tbuf[j & 1];                  // in place over b_{m+2}
        p.gsrc = cfg.prescaled ? ybuf[(j - 1) & 1] : tbuf[(j - 1) & 1];
        p.y_own = (cfg.prescaled && m > 0) ? ybuf[j & 1] : nullptr;
        p.tbar = tbar_at(m);
        p.c_adj = m == 0 ? 1.f : 2.f;
        for (int s = 0; s < n_scales; ++s) p.c_k[s] = coeffs_host[s * (k + 1) + m];
        if (app_events_host) {
            rc = check_cuda(cudaEventRecord((cudaEvent_t)app_events_host[2 * (j - 1)], st), "event record");
            if (rc) return rc;
        }
        rc = launch_order<true>(p, cfg, st);
        if (rc) return rc;
        if (app_events_host) {
            rc = check_cuda(cudaEventRecord((cudaEvent_t)app_events_host[2 * (j - 1) + 1], st), "event record");
            if (rc) return rc;
        }
    }
    return EGNN_OK;
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
    const size_t need = egnn_cheb_coeff_grad_ws_bytes(k, n_scales);
    if (workspace == nullptr || workspace_bytes < need) {
        set_error("coefficient-gradient workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
        return EGNN_ERR_WORKSPACE;
    }
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
    const size_t need = egnn_csr_transpose_ws_bytes(n, nnz);
    if (workspace == nullptr || workspace_bytes < need) {
        set_error("transpose workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
        return EGNN_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const size_t arr = align_up(4 * (size_t)(nnz > 0 ? nnz : 1), 256);
    char* ws = (char*)align_up((size_t)workspace, 256);
    uint32_t* keys_sorted = (uint32_t*)ws;
    int32_t* ids = (int32_t*)(ws + arr);
    int32_t* ids_sorted = (int32_t*)(ws + 2 * arr);
    int32_t* counts = (int32_t*)(ws + 3 * arr);
    void* cub_temp = ws + 3 * arr + align_up(4 * (size_t)(n + 1), 256);
    size_t cub_bytes = transpose_cub_bytes(n, nnz);
    int rc = check_cuda(cudaMemsetAsync(counts, 0, sizeof(int32_t) * (size_t)(n + 1), st), "memset column counts");
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
    EGNN_REQUIRE(dinv_full && iso_full && out_local && coeffs_host && t_prev_local, "null pointer");
    EGNN_REQUIRE(row_begin >= 0 && row_end >= row_begin && row_end <= n, "bad row range");
    EGNN_REQUIRE(order >= 1 && order <= k_max && k_max <= EGNN_MAX_ORDER, "bad order");
    EGNN_REQUIRE(n_scales >= 1 && n_scales <= EGNN_MAX_SCALES, "n_scales out of range");
    EGNN_REQUIRE(phase >= 0 && phase <= 2, "bad phase");
    EGNN_REQUIRE(order == 1 || t_prev2_local, "T_{k-2} missing");
    const int64_t rows = row_end - row_begin;
    if (rows == 0) return EGNN_OK;
    cudaStream_t st = (cudaStream_t)stream;

    OrderParams p{};
    p.delta.n = 0;
    if (phase != 0) {                 // edge flips ride with the launch that gathers from the exchanged operand
        int drc = fill_delta(p.delta, delta_row_host, delta_col_host, delta_val_host, n_delta);
        if (drc) return drc;
        for (int i = 0; i < n_delta; ++i)
            EGNN_REQUIRE(p.delta.row[i] >= 0 && p.delta.row[i] < n && p.delta.col[i] >= 0 && p.delta.col[i] < n,
                         "delta index out of range");
    }
    p.vals = nullptr; p.dinv = dinv_full; p.iso = iso_full;
    p.tprev_own = t_prev_local; p.tprev2_own = t_prev2_local; p.tk_own = t_out_local; p.y_own = nullptr;
    p.out = out_local; p.acc_ws = acc_ws; p.n_rows = rows; p.row0 = row_begin; p.F = f; p.S = n_scales;
    p.a = op_scale; p.b = op_shift; p.first = order == 1;
    for (int s = 0; s < n_scales; ++s) {
        p.c_prev[s] = coeffs_host[s * (k_max + 1) + order - 1];
        p.c_k[s] = coeffs_host[s * (k_max + 1) + order];
    }
    OrderConfig cfg = choose_config(rows, nnz_hint, f);
    cfg.prescaled = false;            // sharded slabs carry plain T_k (what the exchange moves)
    p.fl_log2 = cfg.fl_log2; p.nz_log2 = cfg.nz_log2;
    const bool last = order == k_max;
    const bool fuse_norm = normalize_l1 && cfg.grid_y == 1;
    int rc;
    if (phase == 0) {                 // local columns: gathers hit the rank's own slab
        EGNN_REQUIRE(rowptr_local && acc_ws, "local half missing");
        p.rowptr = rowptr_local; p.colidx = colidx_local;
        p.gsrc = t_prev_local - row_begin * (int64_t)f;      // indexed by global column, only own rows touched
        p.mode = 1; p.normalize = 0;
        return launch_order(p, cfg, st);
    }
    EGNN_REQUIRE(t_prev_full != nullptr, "gathered T_{k-1} missing");
    p.gsrc = t_prev_full;
    p.normalize = last && fuse_norm;
    if (phase == 1) {                 // remote columns + epilogue
        EGNN_REQUIRE(rowptr_remote && acc_ws, "remote half missing");
        p.rowptr = rowptr_remote; p.colidx = colidx_remote; p.mode = 2;
    } else {                          // one launch over the unsplit rows
        EGNN_REQUIRE(rowptr_local != nullptr, "csr missing");
        p.rowptr = rowptr_local; p.colidx = colidx_local; p.mode = 0;
    }
    rc = launch_order(p, cfg, st);
    if (rc) return rc;
    if (last && normalize_l1 && !fuse_norm) {
        l1_normalize_kernel<<<grid_for(rows * n_scales * 32, 256), 256, 0, st>>>(out_local, rows * n_scales, f);
        EGNN_LAUNCH_CHECK("l1_normalize_kernel launch");
    }
    return EGNN_OK;
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
    if (!workspace || workspace_bytes < w.total_bytes) {
        set_error("sell workspace too small: need %zu bytes, got %zu", w.total_bytes, workspace_bytes);
        return EGNN_ERR_WORKSPACE;
    }
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
    int64_t tot[8];
    rc = check_cuda(cudaMemcpyAsync(tot, w.totals, 64, cudaMemcpyDeviceToHost, st), "copy totals"); if (rc) return rc;
    rc = check_cuda(cudaStreamSynchronize(st), "sync"); if (rc) return rc;
    plan->n = (int32_t)n;
    plan->n_cta = device_sm_count();               // persistent grid of the hot kernel: one CTA per SM
    plan->n_vrows = tot[kTotV];
    plan->n_slices = tot[kTotSlices];
    plan->n_entries = tot[kTotEntries];
    plan->n_rowv = tot[kTotRowV];
    return EGNN_OK;
}

int egnn_sell_fill(const int32_t* rowptr, const int32_t* colidx, int64_t n, int64_t nnz,
                   const egnn_sell_plan* plan, void* workspace, size_t workspace_bytes, egnn_stream_t stream) {
    int rc = sell_check_geometry(n, nnz, plan);
    if (rc) return rc;
    (void)rowptr;
    EGNN_REQUIRE(plan->slice_off && plan->blk_slice_ptr && plan->rv_ptr && plan->cta_info && plan->sched, "plan buffers not allocated");
    EGNN_REQUIRE(plan->n_cta >= 1 && plan->n_cta <= 4096, "n_cta out of range");
    EGNN_REQUIRE(plan->n_entries == 0 || plan->idx, "plan idx not allocated");
    EGNN_REQUIRE(plan->n_vrows == 0 || plan->vslot, "plan vslot not allocated");
    const int C = plan->n_blocks, CB = plan->col_block, lmax = plan->lmax;
    SellWs w = sell_ws_layout(workspace, n, nnz, C, lmax);
    if (!workspace || workspace_bytes < w.total_bytes) {
        set_error("sell workspace too small: need %zu bytes, got %zu", w.total_bytes, workspace_bytes);
        return EGNN_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    rc = check_cuda(cudaMemcpyAsync(plan->slice_off, w.slice_off, 4 * (plan->n_slices + 1), cudaMemcpyDeviceToDevice, st), "copy slice_off"); if (rc) return rc;
    rc = check_cuda(cudaMemcpyAsync(plan->blk_slice_ptr, w.bsp, 4 * (C + 1), cudaMemcpyDeviceToDevice, st), "copy blk_slice_ptr"); if (rc) return rc;
    rc = check_cuda(cudaMemcpyAsync(plan->rv_ptr, w.rv_ptr, 4 * (n + 1), cudaMemcpyDeviceToDevice, st), "copy rv_ptr"); if (rc) return rc;
    sell_cta_blocks_kernel<<<1, 32, 0, st>>>(w.slice_off, w.bsp, C, plan->n_cta, plan->cta_info, plan->sched);
    EGNN_LAUNCH_CHECK("sell_cta_blocks_kernel launch");
    // epilogue row ranges balanced by cost (nvrow / nv of the workspace are free again: reused for the costs and their prefix)
    sell_row_cost_kernel<<<(unsigned)ceil_div64(n + 1, 256), 256, 0, st>>>(w.rv_ptr, (int)n, w.nvrow);
    EGNN_LAUNCH_CHECK("sell_row_cost_kernel launch");
    size_t tb = w.cub_bytes;
    rc = check_cuda(cub::DeviceScan::ExclusiveSum(w.cub_temp, tb, w.nvrow, w.nv, (int)(n + 1), st), "scan row costs"); if (rc) return rc;
    sell_cta_rows_kernel<<<(unsigned)ceil_div64(plan->n_cta + 1, 128), 128, 0, st>>>(w.nv, (int)n, plan->n_cta,
                                                                                 plan->cta_info + 2 * plan->n_cta + kSellMaxBlocks);
    EGNN_LAUNCH_CHECK("sell_cta_rows_kernel launch");
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
    EGNN_REQUIRE(plan->vpart && plan->slice_off && plan->blk_slice_ptr && plan->rv_ptr && plan->vslot && plan->cta_info && plan->sched,
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
    int rc = fill_delta(sp.delta, delta_row_host, delta_col_host, delta_val_host, n_delta);
    if (rc) return rc;
    for (int i = 0; i < n_delta; ++i)
        EGNN_REQUIRE(sp.delta.row[i] >= 0 && sp.delta.row[i] < plan->n_cols && sp.delta.col[i] >= 0 && sp.delta.col[i] < plan->n_cols,
                     "delta index out of range");
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
    const size_t need = egnn_calibration_metrics_ws_bytes(n_classes, n_bins);
    if (!workspace || workspace_bytes < need) {
        set_error("metrics workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
        return EGNN_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    char* base = (char*)align_up((size_t)workspace, 256);
    const size_t arr = align_up(8 * (size_t)n_classes * n_bins, 256);
    EceWs ws;
    ws.sum_p = (double*)base;
    ws.count = (unsigned long long*)(base + arr);
    ws.hits = (unsigned long long*)(base + 2 * arr);
    ws.scalars = (double*)(base + 3 * arr);
    int rc = check_cuda(cudaMemsetAsync(base, 0, 3 * arr + 64, st), "memset metrics workspace");
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
    EGNN_REQUIRE(win->f == (f >= kWideMinF ? (f + 3) / 4 * 4 : f) && row0 + n_rows <= (int64_t)win->world * win->rows_per,
                 "window does not fit the signal");
    PeerPush pp{};
    fill_peer_push(pp, win, 0, true, true);
    int64_t blocks = ceil_div64(n_rows > 0 ? n_rows * win->f : 1, 1024);      // at most one CTA per SM: one system fence each
    const int sms = device_sm_count();
    if (blocks > sms) blocks = sms;
    peer_prescale_push_kernel<<<(unsigned)blocks, 1024, 0, (cudaStream_t)stream>>>(x_local, dinv_full, n_rows, row0, f, win->f, pp);
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
    const int ldy = (f + 3) / 4 * 4;
    EGNN_REQUIRE(win->f == ldy && (int64_t)win->world * win->rows_per >= n_global, "window does not fit the signal");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t rows = row_end - row_begin;
    const RingConfig rcfg = ring_config(ldy);
    WideParams wp{};
    rc = fill_delta(wp.delta, delta_row_host, delta_col_host, delta_val_host, n_delta);
    if (rc) return rc;
    for (int i = 0; i < n_delta; ++i)
        EGNN_REQUIRE(wp.delta.row[i] >= 0 && wp.delta.row[i] < n_global && wp.delta.col[i] >= 0 && wp.delta.col[i] < n_global,
                     "delta index out of range");
    wp.rowptr = rowptr_local; wp.colidx = colidx_local; wp.vals = vals_or_null;
    wp.perm = row_order_or_null; wp.n_hub = row_order_or_null ? row_order_or_null + rows : nullptr;
    wp.dinv = dinv_full; wp.iso = iso_full; wp.out = out_local; wp.n_rows = rows; wp.row0 = row_begin;
    wp.F = f; wp.ldy = ldy; wp.S = n_scales; wp.a = op_scale; wp.b = op_shift;
    const bool last = order == k_max;
    const bool fuse_norm = normalize_l1 && rcfg.grid_y == 1;
    wp.first = order == 1;
    wp.normalize = last && fuse_norm;
    wp.ysrc = peer_operand(win, win->rank, (order - 1) & 1);                  // full operand, global rows
    wp.x0_own = order == 1 ? x0_local : nullptr;
    float* own_next = peer_operand(win, win->rank, order & 1) + row_begin * (int64_t)ldy;
    wp.y2_own = order == 1 ? nullptr : own_next;                              // dinv (.) T_{k-2} of the own rows
    wp.y_out = (!last && win->world == 1) ? own_next : nullptr;               // single rank: plain store
    wp.tk_out = t_out_local_or_null;
    for (int s = 0; s < n_scales; ++s) {
        wp.c_prev[s] = coeffs_host[s * (k_max + 1) + order - 1];
        wp.c_k[s] = coeffs_host[s * (k_max + 1) + order];
    }
    fill_peer_push(wp.peer, win, order & 1, !last, false);
    rc = launch_wide(wp, rcfg, device_sm_count(), st);
    if (rc) return rc;
    if (last && normalize_l1 && !fuse_norm && rows > 0) {
        l1_normalize_kernel<<<grid_for(rows * n_scales * 32, 256), 256, 0, st>>>(out_local, rows * n_scales, f);
        EGNN_LAUNCH_CHECK("l1_normalize_kernel launch");
    }
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
        const int g = grid_for(n_rows * 32, 256);
        if (vals_or_null)
            degree_kernel<true><<<g, 256, 0, st>>>(rowptr_local, colidx_local, vals_or_null, n_rows, rowsum_local,
                                                   diag_full + row_begin, colsum_full, unsorted_flag_or_null, row_begin);
        else
            degree_kernel<false><<<g, 256, 0, st>>>(rowptr_local, colidx_local, nullptr, n_rows, rowsum_local,
                                                    diag_full + row_begin, colsum_full, unsorted_flag_or_null, row_begin);
        EGNN_LAUNCH_CHECK("degree_kernel launch");
        return EGNN_OK;
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
    DeltaList d;
    rc = fill_delta(d, delta_row_host, delta_col_host, delta_val_host, n_delta);
    if (rc) return rc;
    for (int i = 0; i < n_delta; ++i)
        EGNN_REQUIRE(d.row[i] >= 0 && d.row[i] < n && d.col[i] >= 0 && d.col[i] < n, "delta index out of range");
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
    EGNN_REQUIRE(target >= 0 && target < n && n_classes >= 1, "bad target / classes");
    DeltaList d;
    rc = fill_delta(d, delta_row_host, delta_col_host, delta_val_host, n_delta);
    if (rc) return rc;
    for (int i = 0; i < n_delta; ++i)
        EGNN_REQUIRE(d.row[i] >= 0 && d.row[i] < n && d.col[i] >= 0 && d.col[i] < n, "delta index out of range");
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
    EGNN_REQUIRE(target >= 0 && target < n && n_classes >= 1, "bad target / classes");
    DeltaList d;
    rc = fill_delta(d, delta_row_host, delta_col_host, delta_val_host, n_delta);
    if (rc) return rc;
    for (int i = 0; i < n_delta; ++i)
        EGNN_REQUIRE(d.row[i] >= 0 && d.row[i] < n && d.col[i] >= 0 && d.col[i] < n, "delta index out of range");
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

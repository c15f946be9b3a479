/*
 * egnn_b200.h - C ABI of libegnn_b200.so: the B200 (sm_100a) implementation of
 * the Chebyshev graph-wavelet feature path of the WATS calibrator.
 *
 * The reference (CaptainCuong/Efficient-GNN) has no FFI; its boundary for this
 * path is three Python functions and one nn.Module in calibration/WATS.py.
 * Each entry point below names the reference lines it replaces.  The host side
 * that mirrors the reference's Python signatures lives in
 * efficient-gnn_b200/wats.py and binds these symbols with ctypes
 * (INTEGRATION.md shows the stub a reference maintainer would add).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host;
 *   - the caller owns all buffers (torch tensors in practice) and passes the
 *     CUDA stream to launch on; the library keeps no state between calls
 *     except a thread-local last-error string;
 *   - every function returns 0 on success or a negative egnn_status; nothing
 *     throws across the ABI;
 *   - indices are int32 (nnz < 2^31), features float32, row-major.
 */
#ifndef EGNN_B200_H
#define EGNN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* egnn_stream_t; /* cudaStream_t */

enum egnn_status {
    EGNN_OK = 0,
    EGNN_ERR_INVALID_ARG = -1,
    EGNN_ERR_CUDA = -2,
    EGNN_ERR_UNSUPPORTED_ARCH = -3,
    EGNN_ERR_WORKSPACE = -4
};

#define EGNN_MAX_SCALES 8
#define EGNN_MAX_ORDER 64
#define EGNN_MAX_DELTA 64
#define EGNN_MAX_RANKS 16
#define EGNN_IPC_HANDLE_BYTES 64

/* ABI version of this header (bumped on any signature change). */
int egnn_abi_version(void);

/* Message of the last failure on the calling thread ("" if none). */
const char* egnn_last_error(void);

/* SM count / compute capability of the current device; fails with
 * EGNN_ERR_UNSUPPORTED_ARCH when the device is not sm_100. */
int egnn_device_info(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor);

/* ---- dense adjacency -> CSR ------------------------------------------------
 * Replaces `csr_matrix(adj.cpu().numpy())` (calibration/WATS.py:99): the
 * device->host copy of the dense [N,N] float32 adjacency and scipy's dense
 * scan.  Pass 1 counts stored (non-zero) entries per row and writes the
 * exclusive scan to rowptr[0..n]; *nonbinary (device int32) is set to 1 when
 * any stored value differs from 1.0f.  The caller reads rowptr[n], allocates
 * colidx (and vals when non-binary) and runs pass 2.  ld = row stride.      */
int egnn_dense_to_csr_count(const float* adj, int64_t n, int64_t ld,
                            int32_t* rowptr, int32_t* nonbinary,
                            egnn_stream_t stream);
int egnn_dense_to_csr_fill(const float* adj, int64_t n, int64_t ld,
                           const int32_t* rowptr, int32_t* colidx,
                           float* vals_or_null, egnn_stream_t stream);

/* ---- graph preparation -----------------------------------------------------
 * Replaces scipy `csgraph.laplacian(adj, normed=True)` as called by
 * compute_normalized_laplacian (calibration/WATS.py:24-27) and the degree
 * signal of calibration/WATS.py:58-59, without materialising L:
 *   w_j     = colsum_j(A) - A_jj            (in-degree, self loops excluded)
 *   iso_j   = (w_j == 0)
 *   dinv_j  = iso_j ? 1 : 1/sqrt(w_j)
 *   x0_i    = log1p(rowsum_i(A))            (self loops and weights included)
 * vals_or_null == NULL means a binary adjacency (all stored values 1).
 * Outputs dinv/iso/x0_logdeg (x0 may be NULL), w_out_or_null (the float32 w
 * before the sqrt) and rowsum_out, the base vectors egnn_patch_degrees needs.
 * diag_ws: [n] float32 scratch; colsum_ws: [n] float64 scratch.
 * unsorted_flag_or_null: device int32 set to 1 when some row's column indices
 * are not strictly increasing (the SELL plan needs sorted, duplicate-free rows). */
int egnn_graph_prep(const int32_t* rowptr, const int32_t* colidx,
                    const float* vals_or_null, int64_t n,
                    float* dinv, uint8_t* iso, float* x0_logdeg,
                    float* w_out_or_null, float* rowsum_out,
                    float* diag_ws, double* colsum_ws, int32_t* unsorted_flag_or_null,
                    egnn_stream_t stream);

/* The same pass in pieces, for ingestion pipelined with the host->device copy
 * of the CSR: the caller zero-fills colsum (and the flag) once, runs
 * egnn_degree_rows on each row range as its entries arrive (it accumulates
 * into colsum and writes rowsum/diag of the range), then egnn_graph_prep_finish. */
int egnn_degree_rows(const int32_t* rowptr, const int32_t* colidx, const float* vals_or_null,
                     int64_t n, int64_t row_begin, int64_t row_end,
                     float* rowsum, float* diag, double* colsum,
                     int32_t* unsorted_flag_or_null, egnn_stream_t stream);
int egnn_graph_prep_finish(const double* colsum, const float* diag, const float* rowsum,
                           int64_t n, float* dinv, uint8_t* iso, float* x0_logdeg,
                           float* w_out_or_null, egnn_stream_t stream);

/* UGCA recompute (the point where calib_attack/calib_fga.py:868,908,952 call
 * the calibrated surrogate on a perturbed adjacency): copies dinv/iso/x0 of
 * the base graph into the *_out vectors and re-derives the entries of every
 * node an edge flip touches.  Flip e adds delta_val[e] to
 * A[delta_row[e], delta_col[e]] (host arrays, n_delta <= EGNN_MAX_DELTA).
 * w/dinv/iso are full-length [n]; rowsum_base/x0_base/x0_out hold the rows
 * [row_begin, row_begin + n_rows) - the whole graph (0, n) on one GPU, the
 * rank's rows on a row shard (flips are global ids; every rank patches its
 * replicated dinv/iso and its own rows of x0).                               */
int egnn_patch_degrees(const float* w_base, const float* rowsum_base,
                       const float* dinv_base, const uint8_t* iso_base,
                       const float* x0_base, int64_t n,
                       const int32_t* delta_row_host, const int32_t* delta_col_host,
                       const float* delta_val_host, int32_t n_delta,
                       float* dinv_out, uint8_t* iso_out, float* x0_out,
                       int64_t row_begin, int64_t n_rows, egnn_stream_t stream);

/* The same patch without the three vector copies, for the recompute loop: the *_io vectors are
 * scratch copies of the base graph's dinv / iso / x0 / y0 = dinv (.) x0 (made once by the caller);
 * restore = 0 writes the patched values of every node a flip touches, restore = 1 puts the base
 * values back (queue it after the wavelet pass that used the patched vectors).               */
int egnn_patch_nodes(const float* w_base, const float* rowsum_base, const float* dinv_base,
                     const uint8_t* iso_base, const float* x0_base, const float* y0_base, int64_t n,
                     const int32_t* delta_row_host, const int32_t* delta_col_host,
                     const float* delta_val_host, int32_t n_delta,
                     float* dinv_io, uint8_t* iso_io, float* x0_io, float* y0_io,
                     int32_t restore, egnn_stream_t stream);

/* ---- SELL plan: one-time re-layout of a binary, column-sorted CSR -----------
 * New in this build (no reference counterpart: scipy streams plain CSR).  For
 * F = 1 - the reference's default signal, calibration/WATS.py:58-59 - the
 * orders run on a column-blocked sliced-ELL copy of the adjacency with 16-bit
 * block-local indices, whose operand block is staged in shared memory
 * (DESIGN.md "narrow path").  Building is two calls around the caller's
 * allocation:
 *   egnn_sell_geometry   picks n_blocks / col_block / lmax for n nodes;
 *   egnn_sell_prepare    counts (all passes but the last) in `workspace`,
 *                        SYNCHRONISES the stream and fills the size fields;
 *   (caller allocates slice_off[n_slices+1], blk_slice_ptr[n_blocks+1],
 *    idx[n_entries] (uint16, 256-byte aligned), rv_ptr[n+1], vslot[n_vrows], cta_info[3*n_cta+65],
 *    hub[n_cta+1+n_hub], sched[2112] uint32, vpart[n_rowv] float32 scratch: row i's partial sums are
 *    vpart[rv_ptr[i] .. rv_ptr[i+1]), virtual row v writes vpart[vslot[v]])
 *   egnn_sell_fill       writes the index stream; `workspace` must be the
 *                        one prepare used, untouched in between.
 * A plan is read-only afterwards except vpart and sched (one wavelet call at a
 * time per plan).                                                             */
typedef struct egnn_sell_plan {
    int32_t n, n_blocks, col_block, lmax; /* n: rows laid out (a row shard or the whole graph) */
    int32_t n_cols, row0;                 /* columns = global nodes; global id of row 0        */
    int32_t n_cta, reserved;              /* CTAs of the step kernel (set by prepare: SM count, one per SM) */
    int64_t n_slices, n_vrows, n_entries, n_rowv;
    int32_t* slice_off;
    int32_t* blk_slice_ptr;
    uint16_t* idx;
    int32_t* rv_ptr;
    int32_t* vslot;
    int32_t* cta_info;                    /* [3 * n_cta + 65]: column block and rank inside it of every CTA, start value
                                             of every block's slice counter, first row of every CTA's epilogue range
                                             (ranges of equal cost, not equal length) (egnn_sell_fill)                */
    float* vpart;
    uint32_t* sched;                      /* [2112] slice counters (one 128-byte line per column block) + grid-barrier
                                             counter of the step kernel (egnn_sell_fill
                                             initialises them; the kernel leaves them ready for the next launch)      */
    uint64_t* stamps;                     /* optional [4 + 2 * orders per launch]: globaltimer of CTA 0 at kernel start,
                                             after every grid barrier and at the end (phase breakdown for bench.py)   */
    int64_t n_hub;                        /* rows with more than 24 partial sums, summed by a whole warp (prepare)   */
    int32_t* hub;                         /* [n_cta + 1 + n_hub]: CTA g's hub rows are hub[n_cta + 1 + hub[g] ..
                                             n_cta + 1 + hub[g + 1]), ascending (egnn_sell_fill)                      */
} egnn_sell_plan;

int egnn_sell_geometry(int64_t n_cols, int64_t nnz, int32_t* n_blocks, int32_t* col_block, int32_t* lmax);
size_t egnn_sell_ws_bytes(int64_t n, int64_t nnz, int32_t n_blocks, int32_t lmax);
int egnn_sell_prepare(const int32_t* rowptr, const int32_t* colidx, int64_t n, int64_t nnz,
                      egnn_sell_plan* plan, void* workspace, size_t workspace_bytes,
                      egnn_stream_t stream);
int egnn_sell_fill(const int32_t* rowptr, const int32_t* colidx, int64_t n, int64_t nnz,
                   const egnn_sell_plan* plan, void* workspace, size_t workspace_bytes,
                   egnn_stream_t stream);

/* ---- fused Chebyshev-wavelet pass -----------------------------------------
 * Replaces the rescale (calibration/WATS.py:55), chebyshev_polynomials
 * (:29-37), the heat-coefficient combination (:65-68) and the row L1
 * normalisation (:71-72).  For k = 1..K one kernel computes
 *   T_k = m_k * L~ T_{k-1} - T_{k-2},   m_1 = 1, m_k = 2,
 *   L~ = op_scale * L_sym + op_shift * I   (reference: 2/lambda_max = 1 and -1),
 *   (L~ x)_i = theta_i x_i - op_scale dinv_i sum_{j != i} a_ij dinv_j x_j,
 *   theta_i = op_scale (1 - iso_i) + op_shift,
 * and accumulates out[i, s, :] += coeffs_host[s*(K+1)+k] * T_k[i, :] for all
 * n_scales scales in the same pass; the last order applies the L1
 * normalisation per (row, scale) when normalize_l1 != 0.
 *   x0            [n, f]        input signal T_0
 *   out           [n, n_scales, f]
 *   t_all_or_null [K+1, n, f]   when non-NULL every order is also stored
 *   delta_*       optional edge flips applied on top of the CSR (UGCA
 *                 recompute): entry e adds delta_val[e] to
 *                 A[delta_row[e], delta_col[e]]; dinv/iso/x0 passed in must
 *                 already describe the perturbed graph (egnn_patch_degrees).
 *                 Host pointers, n_delta <= EGNN_MAX_DELTA.
 * workspace: egnn_cheb_workspace_bytes(n, f) bytes, 256-byte aligned.
 * When f % 4 == 0 the kernels access x0, out and t_all_or_null with 16-byte
 * vector loads and stores: those must then be 16-byte aligned, else
 * EGNN_ERR_INVALID_ARG (nothing is launched).
 * order_events_host: NULL, or 2*K cudaEvent_t handles; events 2(k-1) and
 * 2(k-1)+1 are recorded on `stream` around order k's kernel (per-kernel
 * timing for the roofline report; no effect on results).  With a SELL plan the
 * whole step is one launch: events 0 and 1 bracket it, the rest follow it.
 * sell_plan_or_null: when given (f == 1, binary adjacency) the orders run on
 * the SELL plan; rowptr/colidx are then only used for the argument checks.
 * row_order_or_null: the processing order from egnn_row_order (used for
 * f >= 8: longest rows first, hub rows summed by a whole CTA); NULL = CSR order.
 * y0_or_null (SELL plan only): dinv (.) x0 [n] when the caller already holds it
 * (fixed per graph for the default signal log1p(degree)): the step kernel then
 * skips computing it.  Must match dinv and x0 (so not with edge flips).
 * rows_sorted: non-zero when every CSR row is sorted by column (the unsorted
 * flag of egnn_graph_prep): f == 1 without a plan on a large graph (nnz >= 4 M)
 * then runs the plan-free column-blocked kernel (csrc/blocked.cuh: operand
 * staged in shared memory, no re-layout) instead of the generic CSR kernel
 * (2: also on small graphs - tests).
 * w_base_or_null / rowsum_base_or_null (SELL plan + edge flips): the base
 * graph's in-degrees without self loops and row sums [n] (the `w` and `rowsum`
 * of egnn_graph_prep).  When given, dinv / iso / x0 / y0_or_null are the BASE
 * graph's vectors and the step kernel re-derives the entries of the nodes the
 * flips touch itself (the arithmetic of egnn_patch_nodes): a perturbed pass is
 * one launch, nothing to patch or restore.  default_signal != 0 says that x0
 * is log1p(row sum) and changes with the flips; 0 keeps the caller's x0.     */
size_t egnn_cheb_workspace_bytes(int64_t n, int32_t f);
int egnn_cheb_wavelet(const int32_t* rowptr, const int32_t* colidx,
                      const float* vals_or_null, const float* dinv,
                      const uint8_t* iso, const float* x0, int64_t n, int64_t nnz,
                      int32_t f, int32_t k, int32_t n_scales,
                      const float* coeffs_host, float op_scale, float op_shift,
                      float* out, float* t_all_or_null, int32_t normalize_l1,
                      const int32_t* delta_row_host, const int32_t* delta_col_host,
                      const float* delta_val_host, int32_t n_delta,
                      void* workspace, size_t workspace_bytes,
                      egnn_stream_t stream, void* const* order_events_host,
                      const egnn_sell_plan* sell_plan_or_null, const int32_t* row_order_or_null,
                      const float* y0_or_null, int32_t rows_sorted,
                      const float* w_base_or_null, const float* rowsum_base_or_null,
                      int32_t default_signal);

/* Processing order of the wide-signal kernel (new in this build): rows by
 * descending stored-entry count.  order_out: int32[n + 1] - the permutation,
 * then the number of leading rows long enough to be summed by a whole CTA.   */
size_t egnn_row_order_ws_bytes(int64_t n);
int egnn_row_order(const int32_t* rowptr, int64_t n, int32_t* order_out,
                   void* workspace, size_t workspace_bytes, egnn_stream_t stream);

/* ---- backward of the wavelet pass ------------------------------------------
 * With M = op_scale * L_sym + op_shift * I and C_s = sum_k alpha[s,k] T_k(M) X
 * (egnn_cheb_wavelet), the gradient of a loss w.r.t. X given upstream
 * gradients cbar = dLoss/dC [n, n_scales, f] and tbar_or_null = dLoss/dT_k
 * [K+1, n, f] is the Clenshaw sum
 *   v_k = sum_s alpha[s,k] cbar[:, s, :] + tbar_k,
 *   b_K = v_K,  b_k = v_k + 2 M^T b_{k+1} - b_{k+2} (k = K-1..1),
 *   xbar = v_0 + M^T b_1 - b_2,
 * K applications of M^T, each one launch of the adjoint instantiation of the
 * forward's order kernel (f >= 8: the wide kernel; every f < 8 the generic CSR
 * kernel, there is no SELL path).  coeffs_host is the forward's [S, K+1].
 * rowptr_t/colidx_t/vals_t: the TRANSPOSED adjacency (egnn_csr_transpose; the
 * graph's own CSR when it is symmetric) with the FORWARD's dinv / iso (scipy
 * normalises by column sums on both sides).  delta_*: the forward's flips with
 * rows and columns swapped (dinv / iso already patched, as for the forward).
 * cbar, tbar_or_null and xbar must be 16-byte aligned when f % 4 == 0 (as
 * x0 / out / t_all of egnn_cheb_wavelet), else EGNN_ERR_INVALID_ARG.
 * workspace: egnn_cheb_workspace_bytes(n, f).  app_events_host: NULL or 2*K
 * events recorded around application j = 1..K (events 2(j-1), 2(j-1)+1).
 * row_order_or_null: egnn_row_order of the transposed CSR (f >= 8).          */
int egnn_cheb_adjoint(const int32_t* rowptr_t, const int32_t* colidx_t,
                      const float* vals_t_or_null, const float* dinv, const uint8_t* iso,
                      int64_t n, int64_t nnz, int32_t f, int32_t k, int32_t n_scales,
                      const float* coeffs_host, float op_scale, float op_shift,
                      const float* cbar, const float* tbar_or_null, float* xbar,
                      const int32_t* delta_row_host, const int32_t* delta_col_host,
                      const float* delta_val_host, int32_t n_delta,
                      void* workspace, size_t workspace_bytes, egnn_stream_t stream,
                      void* const* app_events_host, const int32_t* row_order_or_null);

/* egnn_cheb_adjoint that also keeps every Clenshaw vector (new in ABI 8):
 * b_all [K+1, n, f] receives xbar in slab 0 and b_m in slab m = 1..K (the
 * lambda_k of the adjacency gradient below).  Same kernels as
 * egnn_cheb_adjoint; b_all must be 16-byte aligned when f % 4 == 0.          */
int egnn_cheb_adjoint_all(const int32_t* rowptr_t, const int32_t* colidx_t,
                          const float* vals_t_or_null, const float* dinv, const uint8_t* iso,
                          int64_t n, int64_t nnz, int32_t f, int32_t k, int32_t n_scales,
                          const float* coeffs_host, float op_scale, float op_shift,
                          const float* cbar, const float* tbar_or_null, float* xbar,
                          const int32_t* delta_row_host, const int32_t* delta_col_host,
                          const float* delta_val_host, int32_t n_delta,
                          void* workspace, size_t workspace_bytes, egnn_stream_t stream,
                          void* const* app_events_host, const int32_t* row_order_or_null,
                          float* b_all);

/* ---- gradient w.r.t. the adjacency (ABI 8) ---------------------------------
 * a = op_scale, d = dinv, lam = [K, n, f] stack b_1..b_K (slabs 1..K of
 * egnn_cheb_adjoint_all's b_all), t = [K, n, f] stack T_0..T_{K-1} (the
 * forward's t_all); m_1 = 1, m_k = 2 for k >= 2:
 *   g_ij   = sum_k m_k <d_i lam_k[i,:], d_j T_{k-1}[j,:]>
 *   R_i    = sum_{j != i} A_ij g_ij,   Q_i = sum_{j != i} A_ji g_ji
 *   gw_i   = (a/2) d_i^2 (R_i + Q_i), 0 for an isolated node
 *   grho_i = xbar_i / (1 + rowsum_i) (default signal x0 = log1p(rowsum)), else 0
 *   dLoss/dA_ij = [i != j] (-a g_ij + gw_j) + grho_i.
 * An isolated node's d is held at 1 (w^-1/2 has no derivative at w = 0).
 * All sums run in a fixed order (float32 chunks, float64 carry, no atomics):
 * bitwise deterministic.
 *
 * egnn_adj_grad_degree: gw and grho [n] from the CSR and its transpose
 * (egnn_csr_transpose, or the CSR itself when symmetric); xbar_or_null /
 * rowsum_or_null: the signal's gradient [n] and the row sums, f = 1 default
 * signal only (NULL: grho = 0).  workspace: egnn_adj_grad_degree_ws_bytes(n).
 * egnn_adj_grad_pairs: out[p] = dLoss/dA at (rows[p], cols[p]), any pattern
 * (entries need not be stored in the CSR; indices in [0, n)).
 * egnn_adj_grad_dense: the whole [n, n] gradient into out with row stride ld. */
size_t egnn_adj_grad_degree_ws_bytes(int64_t n);
int egnn_adj_grad_degree(const int32_t* rowptr, const int32_t* colidx, const float* vals_or_null,
                         const int32_t* rowptr_t, const int32_t* colidx_t, const float* vals_t_or_null,
                         const float* dinv, const uint8_t* iso, int64_t n, int64_t nnz, int32_t f,
                         int32_t k, float op_scale, const float* lam, const float* t,
                         const float* xbar_or_null, const float* rowsum_or_null, float* gw, float* grho,
                         void* workspace, size_t workspace_bytes, egnn_stream_t stream);

/* egnn_adj_grad_degree of a perturbed graph A' = A + sum_p v_p e_r e_c^T (new
 * in ABI 12; egnn_adj_grad_degree is this call without flips).  The CSR (and
 * its transpose) hold A; the flips (host arrays, n_delta <= EGNN_MAX_DELTA,
 * indices in [0, n), repeats allowed) add their terms to R and Q:
 *   R_r += v_p g_rc,  Q_c += v_p g_rc   for every flip p = (r, c, v) with r != c
 * (a diagonal flip enters only the row sums), folded in flip-list order.  dinv,
 * iso and rowsum_or_null must be those of A' (egnn_patch_nodes, plus the
 * flips' row sums), as in the perturbed forward.  dLoss/dA'_rc of the flips
 * themselves: egnn_adj_grad_pairs on the flip list with these gw and grho.
 * A refused flip list launches nothing.                                      */
int egnn_adj_grad_degree_flips(const int32_t* rowptr, const int32_t* colidx, const float* vals_or_null,
                               const int32_t* rowptr_t, const int32_t* colidx_t, const float* vals_t_or_null,
                               const float* dinv, const uint8_t* iso, int64_t n, int64_t nnz, int32_t f,
                               int32_t k, float op_scale, const float* lam, const float* t,
                               const float* xbar_or_null, const float* rowsum_or_null,
                               const int32_t* delta_row_host, const int32_t* delta_col_host,
                               const float* delta_val_host, int32_t n_delta, float* gw, float* grho,
                               void* workspace, size_t workspace_bytes, egnn_stream_t stream);
int egnn_adj_grad_pairs(const int32_t* rows, const int32_t* cols, int64_t n_pairs, const float* dinv,
                        const float* lam, const float* t, const float* gw, const float* grho,
                        int64_t n, int32_t f, int32_t k, float op_scale, float* out, egnn_stream_t stream);
int egnn_adj_grad_dense(const float* dinv, const float* lam, const float* t, const float* gw,
                        const float* grho, int64_t n, int32_t f, int32_t k, float op_scale,
                        float* out, int64_t ld, egnn_stream_t stream);

/* Row L1 normalisation out of place, h = c / (sum_f |c| + 1e-8) per row of f
 * values (n_vec rows), and its backward: cbar_out = cbar_in + (hbar -
 * sign(c) <hbar, h>) / r with r recomputed from c and sign(0) = 0.
 * cbar_in_or_null may alias cbar_out; NULL adds to zero.                     */
int egnn_l1_normalize(const float* c, float* h, int64_t n_vec, int32_t f, egnn_stream_t stream);
int egnn_l1_normalize_backward(const float* c, const float* hbar, const float* cbar_in_or_null,
                               float* cbar_out, int64_t n_vec, int32_t f, egnn_stream_t stream);

/* Gradient w.r.t. the heat coefficients: grad_out[s*(K+1)+k] = <cbar[:, s, :],
 * T_k> (device float64 [S, K+1]) from cbar [n, S, f] and the forward's orders
 * t_all [K+1, n, f].  Summed in float64 in a fixed order: deterministic.      */
size_t egnn_cheb_coeff_grad_ws_bytes(int32_t k, int32_t n_scales);
int egnn_cheb_coeff_grad(const float* cbar, const float* t_all, int64_t n, int32_t f, int32_t k,
                         int32_t n_scales, double* grad_out, void* workspace,
                         size_t workspace_bytes, egnn_stream_t stream);

/* CSR transpose: rowptr_t [n+1], colidx_t / vals_t [nnz] (vals_t NULL iff
 * vals NULL).  A stable radix sort by column: every row of the transpose comes
 * out sorted, and the result does not depend on the launch (deterministic).  */
size_t egnn_csr_transpose_ws_bytes(int64_t n, int64_t nnz);
int egnn_csr_transpose(const int32_t* rowptr, const int32_t* colidx, const float* vals_or_null,
                       int64_t n, int64_t nnz, int32_t* rowptr_t, int32_t* colidx_t,
                       float* vals_t_or_null, void* workspace, size_t workspace_bytes,
                       egnn_stream_t stream);

/* ---- fused temperature head (SURVEY 8f.2) ----------------------------------
 * Inference form of WATS.forward, calibration/WATS.py:122-130:
 *   t_i = w2 . relu(W1 feats_i + b1) + b2;  T_i = log(exp(t_i) + 1.1);
 *   out_i = log_softmax(logits_i / T_i).
 * feats [n, f], w1 [hidden, f] (torch Linear layout), b1 [hidden], w2 [hidden],
 * b2 [1], logits/out [n, n_classes]; temps_out_or_null [n] receives T_i.
 * f, hidden <= 64.  Training keeps torch autograd (the host code only calls
 * this under torch.no_grad()).                                               */
int egnn_temperature_head(const float* feats, const float* w1, const float* b1,
                          const float* w2, const float* b2, const float* logits,
                          float* out, float* temps_out_or_null, int64_t n, int32_t f,
                          int32_t hidden, int32_t n_classes, egnn_stream_t stream);

/* ---- sparse structure-gradient surrogate (SURVEY 8f.3) -----------------------
 * What the UGCA attack needs from the calibrated surrogate, without the dense
 * [N,N] forward / backward of calib_attack/calib_fga.py:864-890: the logits of
 * ONE target node of the reference's two-layer row-normalised GCN
 * (src/gnn/model.py:43-52: A_n = D^-1 A with deg 0 -> 1; Z1 = A_n X W1^T + b1;
 * logits = (A_n relu(Z1)) W2^T + b2) on a CSR adjacency (+ edge flips), and row
 * and column `target` of dLoss/dA - the only parts calib_fga.py:881 reads.
 *   egnn_gcn_propagate      y = A_n m + bias (m = X W1^T [n,h], y = Z1), deg_out = raw row sums
 *   egnn_gcn_target_logits  logits_out [n_classes] of node `target`; ctx (EGNN_GCN_CTX_FLOATS
 *                           floats) carries (A_n relu(Z1))[target,:], deg and the diagonal entry
 *   egnn_gcn_structure_grad grad_row[m] = dLoss/dA[target,m], grad_col[i] = dLoss/dA[i,target]
 *                           for upstream = dLoss/dlogits[target,:] [n_classes] (device)
 * h: hidden width, a multiple of 4 up to 128.  Rows of m, bias, y, z1 and xw are
 * accessed with 16-byte vector loads and stores, so those pointers must be 16-byte
 * aligned; a misaligned one is refused with EGNN_ERR_INVALID_ARG before any launch.
 * delta_*: flips as in egnn_cheb_wavelet (the same list must be passed to all
 * three calls of one evaluation).                                               */
#define EGNN_GCN_CTX_FLOATS 136
int egnn_gcn_propagate(const int32_t* rowptr, const int32_t* colidx, const float* vals_or_null,
                       const float* m, const float* bias_or_null, float* y, float* deg_out_or_null,
                       int64_t n, int32_t h,
                       const int32_t* delta_row_host, const int32_t* delta_col_host,
                       const float* delta_val_host, int32_t n_delta, egnn_stream_t stream);
int egnn_gcn_target_logits(const int32_t* rowptr, const int32_t* colidx, const float* vals_or_null,
                           const float* z1, const float* w2, const float* b2, int32_t target,
                           int64_t n, int32_t h, int32_t n_classes, float* logits_out, float* ctx,
                           const int32_t* delta_row_host, const int32_t* delta_col_host,
                           const float* delta_val_host, int32_t n_delta, egnn_stream_t stream);
int egnn_gcn_structure_grad(const int32_t* rowptr, const int32_t* colidx, const float* vals_or_null,
                            const float* upstream, const float* w2, const float* z1, const float* xw,
                            const float* b1, const float* deg, const float* ctx, int32_t target,
                            int64_t n, int32_t h, int32_t n_classes, float* grad_row, float* grad_col,
                            const int32_t* delta_row_host, const int32_t* delta_col_host,
                            const float* delta_val_host, int32_t n_delta, egnn_stream_t stream);

/* ---- calibration metrics on the device (SURVEY 8f.4) --------------------------
 * The evaluation triple of benchmark_calibration_methods.py:100-127 on the
 * samples selected by mask_or_null (uint8 [n]; NULL = all): out3[0] accuracy,
 * out3[1] mean maximum probability, out3[2] class-wise ECE of utils/ece.py:8-89
 * (n_bins right-closed bins per class, bins with < 4 samples skipped, mean over
 * classes).  x: [n, n_classes] probabilities, or log-probabilities when is_log;
 * labels int64 [n]; out3: device double[3].                                     */
size_t egnn_calibration_metrics_ws_bytes(int32_t n_classes, int32_t n_bins);
int egnn_calibration_metrics(const float* x, int32_t is_log, const int64_t* labels,
                             const uint8_t* mask_or_null, int64_t n, int32_t n_classes,
                             int32_t n_bins, double* out3, void* workspace,
                             size_t workspace_bytes, egnn_stream_t stream);

/* ---- row-sharded variant (1-D partition, SURVEY 8e) -------------------------
 * One order on the rows [row_begin, row_end) this rank owns; new in this
 * build (the reference is single-device).  t_prev_full is the exchanged
 * [n, f] T_{k-1}; t_prev_local / t_prev2_local / t_out_local / out_local are
 * the rank's own [rows, f] / [rows, n_scales, f] slabs.  `phase` selects the
 * half of the column-split CSR:
 *   0 = local columns only: partial sums -> acc_ws (runs while the exchange
 *       of T_{k-1} is in flight; gathers touch t_prev_local only),
 *   1 = remote columns + acc_ws, then the fused epilogue,
 *   2 = the unsplit rows in one launch (rowptr_local/colidx_local = full CSR
 *       of the rank's rows).
 * nnz_hint sizes the lane layout (mean row length of the launched half).
 * delta_*: edge flips with GLOBAL ids (UGCA recompute on a sharded graph),
 * applied by the launch that sees the exchanged operand (phase 1 or 2).      */
int egnn_cheb_order_sharded(const int32_t* rowptr_local, const int32_t* colidx_local,
                            const int32_t* rowptr_remote, const int32_t* colidx_remote,
                            const float* dinv_full, const uint8_t* iso_full,
                            const float* t_prev_full, const float* t_prev_local,
                            const float* t_prev2_local, float* t_out_local,
                            float* out_local, float* acc_ws,
                            int64_t n, int64_t nnz_hint, int64_t row_begin, int64_t row_end,
                            int32_t f, int32_t order, int32_t k_max, int32_t n_scales,
                            const float* coeffs_host, float op_scale, float op_shift,
                            int32_t normalize_l1, int32_t phase,
                            const int32_t* delta_row_host, const int32_t* delta_col_host,
                            const float* delta_val_host, int32_t n_delta,
                            egnn_stream_t stream);

/* ---- exchange window over peer memory (NVLink / NVSwitch) -------------------
 * New in this build.  Each rank allocates one window with egnn_peer_alloc
 * (cudaMalloc, zero-filled, exported as a CUDA IPC handle), the host code
 * exchanges the 64-byte handles (torch.distributed) and every rank maps the
 * others' windows with egnn_peer_open.  The sharded order kernels then store
 * the next order's operand straight into every rank's window and signal with
 * flags inside it, so an order needs no collective launch (csrc/peer.cuh).
 * base[r] is rank r's window as mapped in this process (base[rank]: own).   */
typedef struct egnn_peer_window {
    int32_t rank, world;
    int64_t rows_per;            /* rows per rank; the exchanged operand has world * rows_per rows */
    int32_t f;                   /* its columns */
    int32_t reserved;
    void* base[EGNN_MAX_RANKS];
} egnn_peer_window;

size_t egnn_peer_window_bytes(int64_t rows_per, int32_t world, int32_t f);
int egnn_peer_alloc(size_t bytes, void** dev_ptr, void* ipc_handle_out /* EGNN_IPC_HANDLE_BYTES */);
int egnn_peer_open(const void* ipc_handle, void** dev_ptr);
int egnn_peer_close(void* dev_ptr);
int egnn_peer_free(void* dev_ptr);
/* Device address of operand buffer `which` (0/1) inside the caller's own window. */
void* egnn_peer_operand(const egnn_peer_window* win, int32_t which);
/* Copies the window's error word to *error_out (synchronises `stream`); non-zero
 * means a flag wait timed out (a peer never arrived).                         */
int egnn_peer_error(const egnn_peer_window* win, int32_t* error_out, egnn_stream_t stream);

/* Diagnostic: total nanoseconds the first CTA of the consuming kernels spent
 * waiting for peer flags, and the number of waits (synchronises `stream`).   */
int egnn_peer_wait_stats(const egnn_peer_window* win, uint64_t* total_ns, uint64_t* waits,
                         int32_t reset, egnn_stream_t stream);

/* The narrow (F = 1) path on a row shard: orders order_begin..order_end of
 * the step in ONE persistent cooperative launch over the rank's plan (plan->n
 * rows starting at plan->row0, plan->n_cols columns; csrc/sell_step.cuh).
 * Per order: SELL SpMV against the full operand dinv (.) T_{k-1} [n_cols],
 * grid barrier, epilogue on the local rows (T_k, scale accumulation into
 * out_local [rows, n_scales], next operand dinv (.) T_k), grid barrier.
 *   x0_local        [rows] T_0 of the own rows
 *   tbuf0/tbuf1     [rows] each: T_k (k >= 1) lives in tbuf[(k-1)&1]; the same
 *                   two buffers must be passed to every call of a step
 *   t_all_or_null   [k_max+1, rows]: every order stored (then tbuf* unused);
 *                   the caller fills row block 0 with T_0
 *   delta_*         edge flips (GLOBAL row/col ids, host arrays) applied on
 *                   top of the plan; dinv/iso/x0 must describe the perturbed graph -
 *                   or, with w_base_or_null / rowsum_base_or_null [n_cols] given
 *                   (see egnn_cheb_wavelet), the base graph: the kernel then
 *                   re-derives the touched nodes itself, on every rank alike
 * With win_or_null (world > 1) the exchange is fused and the whole step is one
 * call (order_begin = 1, order_end = k_max): before staging a column block the
 * kernel waits for the flags of the ranks that own those columns, the epilogue
 * stores dinv (.) T_k into buffer k&1 of EVERY rank's window, and after the
 * closing grid barrier one CTA raises this rank's flag everywhere.
 * y_first_full, when given, is the operand of order_begin held by every rank
 * (e.g. the default signal): it is read from there and nothing is waited for;
 * when NULL and order_begin == 1 the kernel computes dinv (.) T_0 itself.
 * Without a window a shard runs ONE order per call on the gathered operand
 * y_first_full and leaves dinv (.) T_k of its rows in y_slab{k&1} [rows] for the
 * caller's exchange; a plan that covers all columns' rows (one rank) runs the
 * whole step with y_slab0/1 [n_cols] as its operand buffers.                 */
int egnn_sell_step_sharded(const egnn_sell_plan* plan, const float* dinv_full,
                           const uint8_t* iso_full, const float* x0_local,
                           const float* y_first_full, float* y_slab0, float* y_slab1,
                           float* tbuf0, float* tbuf1, float* t_all_or_null, float* out_local,
                           int32_t order_begin, int32_t order_end, int32_t k_max,
                           int32_t n_scales, const float* coeffs_host, float op_scale,
                           float op_shift, int32_t normalize_l1,
                           const int32_t* delta_row_host, const int32_t* delta_col_host,
                           const float* delta_val_host, int32_t n_delta,
                           const float* w_base_or_null, const float* rowsum_base_or_null,
                           int32_t default_signal,
                           const egnn_peer_window* win_or_null, egnn_stream_t stream);

/* y[r, :] = dinv_full[row0 + r] * x[r, :]: the gather operand of order 1 on
 * the narrow path (later orders get it from the epilogue).                   */
int egnn_prescale(const float* x, const float* dinv_full, float* y, int64_t n_rows,
                  int32_t f, int64_t row0, egnn_stream_t stream);

/* The same product stored into operand buffer 0 of every rank's window: first
 * kernel of a fused-exchange step.  x_local is [n_rows, f]; the window rows are
 * win->f wide (f for the narrow path, f rounded up to a multiple of 4 for
 * f >= 8; padding columns are zeroed).  It first waits until every peer has
 * finished the previous step, then stores and signals.                       */
int egnn_peer_prescale_push(const float* x_local, const float* dinv_full, int64_t n_rows,
                            int64_t row0, int32_t f, const egnn_peer_window* win,
                            egnn_stream_t stream);

/* One order of the wide (f >= 8) path on a row shard with the exchange fused
 * (new in this build): the wide kernel runs on the rank's CSR rows
 * [row_begin, row_end) (global column ids) against operand buffer (order-1)&1
 * of its window - after waiting for the peers' flags - and its epilogue stores
 * dinv (.) T_k of the own rows into buffer order&1 of EVERY rank's window, then
 * signals.  win->f must be f rounded up to a multiple of 4.  x0_local: exact
 * T_0 rows (order 1 only).  t_out_local_or_null: T_k rows [rows, f] when the
 * caller wants every order.  row_order_or_null: egnn_row_order of the shard.
 * delta_*: edge flips with GLOBAL ids applied on top of the shard's CSR.      */
int egnn_wide_order_sharded(const int32_t* rowptr_local, const int32_t* colidx_local,
                            const float* vals_or_null, const int32_t* row_order_or_null,
                            const float* dinv_full, const uint8_t* iso_full,
                            const float* x0_local, float* t_out_local_or_null, float* out_local,
                            int64_t n_global, int64_t row_begin, int64_t row_end,
                            int32_t f, int32_t order, int32_t k_max, int32_t n_scales,
                            const float* coeffs_host, float op_scale, float op_shift,
                            int32_t normalize_l1,
                            const int32_t* delta_row_host, const int32_t* delta_col_host,
                            const float* delta_val_host, int32_t n_delta,
                            const egnn_peer_window* win, egnn_stream_t stream);

/* ---- backward of the row-sharded pass (new in ABI 9) ------------------------
 * The Clenshaw sum of egnn_cheb_adjoint on the rows [row_begin, row_end) a
 * rank owns, one call per application: app = 0 is the prologue b_K = v_K, app
 * = 1..K produces b_m with m = K - app (m = 0: the signal's gradient xbar).
 * The CSR is the rank's rows of the TRANSPOSED adjacency (global column ids,
 * rows sorted), or the rank's own shard when every shard equals its
 * transpose; dinv_full / iso_full are the forward's (patched when it had
 * flips).  cbar_local [rows, n_scales, f] and tbar_local_or_null [K+1, rows, f]
 * are the rank's rows of the upstream gradients.  delta_*: the forward's flips
 * with rows and columns swapped, GLOBAL ids.
 *
 * egnn_cheb_adjoint_sharded: the generic CSR kernel's adjoint instantiation
 * with the phases of egnn_cheb_order_sharded (0: local columns -> acc_ws while
 * the exchange of b_{m+1} is in flight, 1: remote columns + epilogue, 2: the
 * unsplit rows).  app 0 writes b_K to b_out_local and ignores the CSR and the
 * phase.  b_prev_full: the exchanged [n, f] b_{m+1}; b_prev_local /
 * b_prev2_local_or_null: the rank's b_{m+1} / b_{m+2} rows (NULL at app 1);
 * b_out_local receives b_m (may alias b_prev2_local).  Every array is
 * accessed with 16-byte vectors when f % 4 == 0 and must then be 16-byte
 * aligned, else EGNN_ERR_INVALID_ARG and nothing is launched.                */
int egnn_cheb_adjoint_sharded(const int32_t* rowptr_local, const int32_t* colidx_local,
                              const int32_t* rowptr_remote, const int32_t* colidx_remote,
                              const float* dinv_full, const uint8_t* iso_full, const float* b_prev_full,
                              const float* b_prev_local, const float* b_prev2_local_or_null,
                              float* b_out_local, const float* cbar_local,
                              const float* tbar_local_or_null, float* acc_ws,
                              int64_t n, int64_t nnz_hint, int64_t row_begin, int64_t row_end,
                              int32_t f, int32_t app, int32_t k_max, int32_t n_scales,
                              const float* coeffs_host, float op_scale, float op_shift, int32_t phase,
                              const int32_t* delta_row_host, const int32_t* delta_col_host,
                              const float* delta_val_host, int32_t n_delta, egnn_stream_t stream);

/* egnn_wide_adjoint_sharded: f >= 8, k_max >= 1, the exchange fused through
 * the forward's window (win->f = f rounded up to a multiple of 4) and its
 * flag protocol.  app 0 forms b_K and stores dinv (.) b_K into buffer 0 of
 * every rank's window after every peer has finished the kernels before it;
 * app j runs the wide kernel's adjoint instantiation against buffer (j-1)&1
 * after the peers' flags and stores dinv (.) b_m of the own rows into buffer
 * j&1 of every window; app K writes xbar_local [rows, f] instead.
 * row_order_or_null: egnn_row_order of the CSR passed.  cbar, tbar and xbar
 * must be 16-byte aligned when f % 4 == 0, else EGNN_ERR_INVALID_ARG.        */
int egnn_wide_adjoint_sharded(const int32_t* rowptr_local, const int32_t* colidx_local,
                              const int32_t* row_order_or_null, const float* dinv_full,
                              const uint8_t* iso_full, const float* cbar_local,
                              const float* tbar_local_or_null, float* xbar_local,
                              int64_t n_global, int64_t row_begin, int64_t row_end,
                              int32_t f, int32_t app, int32_t k_max, int32_t n_scales,
                              const float* coeffs_host, float op_scale, float op_shift,
                              const int32_t* delta_row_host, const int32_t* delta_col_host,
                              const float* delta_val_host, int32_t n_delta,
                              const egnn_peer_window* win, egnn_stream_t stream);

/* ---- weighted shards and the edge-weight gradient of a shard (new in ABI 11) --
 * egnn_cheb_order_sharded_vals / egnn_cheb_adjoint_sharded_vals: the entries
 * above with float32 values of the local and remote halves (in the halves'
 * entry order; both NULL = binary, exactly the entries above).  The adjoint's
 * values are those of the rank's rows of the TRANSPOSED adjacency.  The
 * adjoint keeps every Clenshaw vector when the caller passes a distinct
 * b_out_local per application instead of rotating over b_{m+2}.
 * egnn_wide_adjoint_sharded_all: egnn_wide_adjoint_sharded with the values of
 * the transposed shard and b_out_local_or_null [rows, f]: b_m of the own rows
 * for every app with m >= 1 (app 0: b_K), the sharded analogue of
 * egnn_cheb_adjoint_all.  b_out must be 16-byte aligned when f % 4 == 0.      */
int egnn_cheb_order_sharded_vals(const int32_t* rowptr_local, const int32_t* colidx_local,
                                 const float* vals_local_or_null,
                                 const int32_t* rowptr_remote, const int32_t* colidx_remote,
                                 const float* vals_remote_or_null,
                                 const float* dinv_full, const uint8_t* iso_full,
                                 const float* t_prev_full, const float* t_prev_local,
                                 const float* t_prev2_local, float* t_out_local,
                                 float* out_local, float* acc_ws,
                                 int64_t n, int64_t nnz_hint, int64_t row_begin, int64_t row_end,
                                 int32_t f, int32_t order, int32_t k_max, int32_t n_scales,
                                 const float* coeffs_host, float op_scale, float op_shift,
                                 int32_t normalize_l1, int32_t phase,
                                 const int32_t* delta_row_host, const int32_t* delta_col_host,
                                 const float* delta_val_host, int32_t n_delta,
                                 egnn_stream_t stream);
int egnn_cheb_adjoint_sharded_vals(const int32_t* rowptr_local, const int32_t* colidx_local,
                                   const float* vals_local_or_null,
                                   const int32_t* rowptr_remote, const int32_t* colidx_remote,
                                   const float* vals_remote_or_null,
                                   const float* dinv_full, const uint8_t* iso_full, const float* b_prev_full,
                                   const float* b_prev_local, const float* b_prev2_local_or_null,
                                   float* b_out_local, const float* cbar_local,
                                   const float* tbar_local_or_null, float* acc_ws,
                                   int64_t n, int64_t nnz_hint, int64_t row_begin, int64_t row_end,
                                   int32_t f, int32_t app, int32_t k_max, int32_t n_scales,
                                   const float* coeffs_host, float op_scale, float op_shift, int32_t phase,
                                   const int32_t* delta_row_host, const int32_t* delta_col_host,
                                   const float* delta_val_host, int32_t n_delta, egnn_stream_t stream);
int egnn_wide_adjoint_sharded_all(const int32_t* rowptr_local, const int32_t* colidx_local,
                                  const float* vals_or_null, const int32_t* row_order_or_null,
                                  const float* dinv_full, const uint8_t* iso_full, const float* cbar_local,
                                  const float* tbar_local_or_null, float* xbar_local,
                                  float* b_out_local_or_null,
                                  int64_t n_global, int64_t row_begin, int64_t row_end,
                                  int32_t f, int32_t app, int32_t k_max, int32_t n_scales,
                                  const float* coeffs_host, float op_scale, float op_shift,
                                  const int32_t* delta_row_host, const int32_t* delta_col_host,
                                  const float* delta_val_host, int32_t n_delta,
                                  const egnn_peer_window* win, egnn_stream_t stream);

/* Edge-weight gradient of a row shard (section 11's terms on the rows
 * [row_begin, row_end); DESIGN.md section 13).  Pre-scaled, node-major
 * stacks [rows, K*F] per rank, all-gathered by the caller into [N', K*F]
 * (N' >= n_global, rank r's rows at row_begin_r):
 *   pl[i] = (m_1 d_i lam_1[i], ..., m_K d_i lam_K[i]),  pt[i] = (d_i T_0[i], ..., d_i T_{K-1}[i])
 * egnn_adj_grad_stacks_sharded: pl_local / pt_local [rows, K*F] from lam_all
 *   [K+1, lam_slab_rows, f] (slab k = b_k; slab 0 unused) and t_all [K+1,
 *   t_slab_rows, f] (the forward's orders of the own rows).
 * egnn_adj_grad_degree_sharded: g_out[q] = g_ij at every stored entry q of
 *   the shard (0 on the diagonal), R over the shard, Q over the rank's rows
 *   of the transposed adjacency, then gw_local / grho_local [rows] (section
 *   11; xbar/rowsum: default signal only).  row_order*_or_null: egnn_row_order
 *   of the two CSRs (longest rows first).  pl_full / pt_full must be 16-byte
 *   aligned when K*F % 4 == 0.  workspace: egnn_adj_grad_degree_sharded_ws_bytes.
 * egnn_adj_grad_entries_sharded: out[q] = dLoss/dA at stored entry q = (i, j)
 *   = [i != j] (-a g_q + gw_full[j]) + grho_local[i - row_begin], from the
 *   all-gathered gw_full [N'] (g may be NULL when k == 0).
 * Fixed summation order, no atomics: bitwise reproducible.                    */
int egnn_adj_grad_stacks_sharded(const float* lam_all, int64_t lam_slab_rows, const float* t_all,
                                 int64_t t_slab_rows, const float* dinv_full, int64_t n_global,
                                 int64_t row_begin, int64_t row_end, int32_t f, int32_t k,
                                 float* pl_local, float* pt_local, egnn_stream_t stream);
size_t egnn_adj_grad_degree_sharded_ws_bytes(int64_t rows);
int egnn_adj_grad_degree_sharded(const int32_t* rowptr, const int32_t* colidx, const float* vals_or_null,
                                 const int32_t* row_order_or_null, const int32_t* rowptr_t,
                                 const int32_t* colidx_t, const float* vals_t_or_null,
                                 const int32_t* row_order_t_or_null, const float* dinv_full,
                                 const uint8_t* iso_full, int64_t n_global, int64_t row_begin,
                                 int64_t row_end, int32_t f, int32_t k, float op_scale,
                                 const float* pl_full, const float* pt_full,
                                 const float* xbar_local_or_null, const float* rowsum_local_or_null,
                                 float* g_out, float* gw_local, float* grho_local,
                                 void* workspace, size_t workspace_bytes, egnn_stream_t stream);
int egnn_adj_grad_entries_sharded(const int32_t* rowptr, const int32_t* colidx, int64_t n_global,
                                  int64_t row_begin, int64_t row_end, int32_t k, const float* g,
                                  const float* gw_full, const float* grho_local, float op_scale,
                                  float* out, egnn_stream_t stream);

/* ---- gradients through the edge flips of a row shard (new in ABI 13) --------
 * The pass ran on A' = A + sum_p v_p e_{r_p} e_{c_p}^T (every rank passes the
 * same global flip list: host arrays, n_delta <= EGNN_MAX_DELTA, indices below
 * n_global, checked before anything launches); DESIGN.md section 15.
 * egnn_adj_grad_degree_sharded_flips: egnn_adj_grad_degree_sharded (which is
 *   this call without flips) with dinv_full / iso_full / pl_full / pt_full of
 *   A', plus g_flips_out[p] = g_{r_p c_p} = <pl[r_p], pt[c_p]> of every flip
 *   (device, [n_delta]; the same bits on every rank) and the flips' part of
 *   the degree terms: R[r_p] += v_p g_p on the rank owning row r_p, Q[c_p] +=
 *   v_p g_p on the rank owning row c_p, for every off-diagonal flip, folded in
 *   flip-list order.  rowsum_local: the row sums of A' (default signal only).
 * egnn_adj_grad_flips_sharded: out[p] = dLoss/dv_p = grho_local[r_p - row_begin]
 *   + [r_p != c_p] (-a g_flips[p] + gw_full[c_p]) for the flips whose row this
 *   rank owns, 0 for the others (device, [n_delta]); the caller adds the
 *   ranks' rows in rank order, which hands every rank the owner's bits.       */
int egnn_adj_grad_degree_sharded_flips(const int32_t* rowptr, const int32_t* colidx,
                                       const float* vals_or_null, const int32_t* row_order_or_null,
                                       const int32_t* rowptr_t, const int32_t* colidx_t,
                                       const float* vals_t_or_null, const int32_t* row_order_t_or_null,
                                       const float* dinv_full, const uint8_t* iso_full, int64_t n_global,
                                       int64_t row_begin, int64_t row_end, int32_t f, int32_t k,
                                       float op_scale, const float* pl_full, const float* pt_full,
                                       const float* xbar_local_or_null, const float* rowsum_local_or_null,
                                       const int32_t* delta_row_host, const int32_t* delta_col_host,
                                       const float* delta_val_host, int32_t n_delta, float* g_flips_out,
                                       float* g_out, float* gw_local, float* grho_local,
                                       void* workspace, size_t workspace_bytes, egnn_stream_t stream);
int egnn_adj_grad_flips_sharded(const int32_t* delta_row_host, const int32_t* delta_col_host,
                                const float* delta_val_host, int32_t n_delta, const float* g_flips,
                                const float* gw_full, const float* grho_local, int64_t n_global,
                                int64_t row_begin, int64_t row_end, float op_scale, float* out,
                                egnn_stream_t stream);

/* Degree pass of a row shard (scipy semantics as egnn_graph_prep).  phase 0:
 * row sums of the local rows, their diagonal entries into diag_full[row_begin..]
 * and the shard's contribution to the in-degree in colsum_full (both zeroed
 * first); the caller then sums colsum_full and diag_full over the ranks
 * (all-reduce).  phase 1: dinv/iso of every node (and the in-degree weight w
 * into w_full_or_null, kept for egnn_patch_degrees) and x0 = log1p(rowsum) of
 * the local rows.                                                             */
int egnn_graph_prep_sharded(const int32_t* rowptr_local, const int32_t* colidx_local,
                            const float* vals_or_null, int64_t n_global, int64_t row_begin,
                            int64_t n_rows, int32_t phase, double* colsum_full, float* diag_full,
                            float* rowsum_local, float* dinv_full, uint8_t* iso_full,
                            float* x0_local, int32_t* unsorted_flag_or_null,
                            float* w_full_or_null, egnn_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* EGNN_B200_H */

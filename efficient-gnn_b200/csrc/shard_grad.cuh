// Gradient of the row-sharded wavelet pass w.r.t. the edge weights of a shard (DESIGN.md section 13).
//
// Section 11's terms with the rows restricted to the rank's [row0, row0 + rows).  The operands are
// exchanged once, pre-scaled and node-major: row j of the [N, K*F] stacks is
//   PL[j] = (m_1 d_j lambda_1[j], ..., m_K d_j lambda_K[j])      (m_1 = 1, m_k = 2)
//   PT[j] = (d_j T_0[j], ..., d_j T_{K-1}[j])
// so g_ij = sum_k m_k <d_i lambda_k[i], d_j T_{k-1}[j]> = <PL[i], PT[j]> is one contiguous dot product
// of length K*F (no per-product index arithmetic), read with 16-byte loads when K*F % 4 == 0.
//   R_i = sum_{j != i} A_ij <PL[i], PT[j]>      over the rank's rows of A (g_ij kept per entry)
//   Q_i = sum_{j != i} A^T_ij <PT[i], PL[j]>    over the rank's rows of A^T
// With edge flips (section 15) the stacks are built on the flipped graph's d, and the flips add their
// part of R / Q and get their own gradient (shard_grad_flip_terms_kernel, shard_grad_flip_values_kernel).
// Every sum runs in a fixed order (float32 chunks, float64 carry, no atomics): bitwise reproducible.
#pragma once

#include "common.cuh"
#include "prep.cuh"

namespace egnn {

constexpr int kShardGradChunk = 32;      // float32 partial sums cover this many products, then spill into fp64
constexpr int kShardGradOwnRegs = 4;     // vectors of the own row a lane keeps in registers across its entries

// pl / pt [rows, K*F] of the own rows from lam_all [K+1, lam_slab_rows, F] (slabs 1..K: lambda_k) and
// t_all [K+1, t_slab_rows, F] (slabs 0..K-1: T_k); d = dinv of the own rows.
__global__ void __launch_bounds__(256)
shard_grad_stacks_kernel(const float* __restrict__ lam_all, int64_t lam_slab, const float* __restrict__ t_all,
                         int64_t t_slab, const float* __restrict__ d, int64_t rows, int32_t F, int32_t K,
                         float* __restrict__ pl, float* __restrict__ pt) {
    const int64_t KF = (int64_t)K * F;
    const int64_t total = rows * KF;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = idx / KF;
        const int64_t e = idx - i * KF;
        const int k = (int)(e / F);
        const int64_t off = i * F + (e - (int64_t)k * F);
        const float di = __ldg(d + i);
        pl[idx] = (k ? 2.f : 1.f) * di * __ldg(lam_all + (int64_t)(k + 1) * lam_slab + off);
        pt[idx] = di * __ldg(t_all + (int64_t)k * t_slab + off);
    }
}

template <int VEC> struct ShardVec;
template <> struct ShardVec<1> {
    using T = float;
    __device__ static T zero() { return 0.f; }
    __device__ static T load(const float* p) { return __ldg(p); }
    __device__ static float dot(T a, T b, float acc) { return fmaf(a, b, acc); }
};
template <> struct ShardVec<4> {
    using T = float4;
    __device__ static T zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
    __device__ static T load(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
    __device__ static float dot(T a, T b, float acc) {
        acc = fmaf(a.x, b.x, acc);
        acc = fmaf(a.y, b.y, acc);
        acc = fmaf(a.z, b.z, acc);
        return fmaf(a.w, b.w, acc);
    }
};

// out[r] = sum_{q in row r, col_q != row0 + r} A_q <own[row0 + r], gath[col_q]> over the rank's rows, and
// g_out[q] = <own[row0 + r], gath[col_q]> (0 on the diagonal) when g_out is given.  One warp per row,
// rows in perm order when given (longest first); 32 >> fl_log2 entries side by side, 1 << fl_log2 lanes
// across the K*F / VEC vectors of an entry.  The lane's share of the own row stays in registers for
// the whole row (up to kShardGradOwnRegs vectors; a longer row re-reads the rest through L1).
template <int VEC>
__global__ void __launch_bounds__(256)
shard_grad_dot_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                      const float* __restrict__ vals, const int32_t* __restrict__ perm,
                      const float* __restrict__ own, const float* __restrict__ gath, int64_t rows, int64_t row0,
                      int32_t KF, int32_t fl_log2, double* __restrict__ out, float* __restrict__ g_out) {
    using V = ShardVec<VEC>;
    const int lane = threadIdx.x & 31;
    const int FL = 1 << fl_log2;
    const int lf = lane & (FL - 1);
    const int grp = lane >> fl_log2;
    const int NZ = 32 >> fl_log2;
    const int nvec = KF / VEC;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t w = warp; w < rows; w += nwarps) {
        const int64_t r = perm ? (int64_t)perm[w] : w;
        const int64_t node = row0 + r;
        const float* orow = own + node * (int64_t)KF;
        typename V::T o[kShardGradOwnRegs];
#pragma unroll
        for (int u = 0; u < kShardGradOwnRegs; ++u) {
            const int c = lf + u * FL;
            o[u] = c < nvec ? V::load(orow + (int64_t)c * VEC) : V::zero();
        }
        double s = 0.0;
        const int q1 = rowptr[r + 1];
        for (int q0 = rowptr[r]; q0 < q1; q0 += NZ) {
            const int q = q0 + grp;
            const bool live = q < q1;
            const int j = live ? ld_stream_i32(colidx + q) : (int)node;
            double hi = 0.0;
            if (j != node) {
                const float* grow = gath + (int64_t)j * KF;
                float acc = 0.f;
                int cnt = 0;
#pragma unroll
                for (int u = 0; u < kShardGradOwnRegs; ++u) {
                    const int c = lf + u * FL;
                    if (c < nvec) {
                        acc = V::dot(o[u], V::load(grow + (int64_t)c * VEC), acc);
                        cnt += VEC;
                        if (cnt >= kShardGradChunk) { hi += (double)acc; acc = 0.f; cnt = 0; }
                    }
                }
                for (int c = lf + kShardGradOwnRegs * FL; c < nvec; c += FL) {
                    acc = V::dot(V::load(orow + (int64_t)c * VEC), V::load(grow + (int64_t)c * VEC), acc);
                    cnt += VEC;
                    if (cnt >= kShardGradChunk) { hi += (double)acc; acc = 0.f; cnt = 0; }
                }
                hi += (double)acc;
            }
            // every lane of the group takes part in the shuffles; lane lf == 0 holds the fixed-order total
            for (int m = FL >> 1; m > 0; m >>= 1) hi += __shfl_xor_sync(0xffffffffu, hi, m);
            if (live && j != node) s = fma((double)(vals ? ld_stream_f32(vals + q) : 1.f), hi, s);
            if (g_out && live && lf == 0) g_out[q] = (float)hi;
        }
        for (int m = FL; m < 32; m <<= 1) s += __shfl_xor_sync(0xffffffffu, s, m);
        if (lane == 0) out[r] = s;
    }
}

// dLoss/dA at the rank's stored entries: out[q] = grho_r + [j != i] ((float)(-a g_q) + gw_full[j]) for
// entry q = (i, j) of local row r, i = row0 + r (g NULL: K = 0, g = 0).  One warp per row, lanes across
// its entries.
__global__ void __launch_bounds__(256)
shard_grad_entries_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                          const float* __restrict__ g, const float* __restrict__ gw_full,
                          const float* __restrict__ grho, int64_t rows, int64_t row0, float a,
                          float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < rows; r += nwarps) {
        const int64_t node = row0 + r;
        const float gr = grho ? __ldg(grho + r) : 0.f;
        const int q1 = rowptr[r + 1];
        for (int q = rowptr[r] + lane; q < q1; q += 32) {
            const int j = ld_stream_i32(colidx + q);
            float v = gr;
            if (j != node) v += (g ? (float)(-(double)a * (double)ld_stream_f32(g + q)) : 0.f) + __ldg(gw_full + j);
            __stcs(out + q, v);
        }
    }
}

// Edge flips A' = A + sum_p v_p e_{r_p} e_{c_p}^T on a row shard (DESIGN.md section 15).  g_p =
// <PL[r_p], PT[c_p]> of every flip from the all-gathered stacks, with the lane layout and summation of
// shard_grad_dot_kernel (so a flip on a stored entry gets that entry's g bit for bit, and every rank the
// same g_p), written to g_out [n_delta]; then R[r_p] += v_p g_p on the rank that owns row r_p and
// Q[c_p] += v_p g_p on the rank that owns row c_p, for every off-diagonal flip, on top of the two
// shard_grad_dot_kernel launches.  One CTA of kShardFlipWarps warps, one warp per flip; one thread folds
// the products in flip-list order (no atomics: several flips on one node are bitwise reproducible).
constexpr int kShardFlipWarps = 32;

template <int VEC>
__global__ void __launch_bounds__(32 * kShardFlipWarps)
shard_grad_flip_terms_kernel(DeltaList d, const float* __restrict__ pl, const float* __restrict__ pt, int64_t rows,
                             int64_t row0, int32_t KF, int32_t fl_log2, float* __restrict__ g_out,
                             double* __restrict__ r_out, double* __restrict__ q_out) {
    using V = ShardVec<VEC>;
    __shared__ double g[EGNN_MAX_DELTA];
    const int lane = threadIdx.x & 31;
    const int FL = 1 << fl_log2;
    const int nvec = KF / VEC;
    for (int p = threadIdx.x >> 5; p < d.n; p += kShardFlipWarps) {
        const float* orow = pl + (int64_t)d.row[p] * KF;
        const float* grow = pt + (int64_t)d.col[p] * KF;
        double hi = 0.0;
        if (lane < FL) {
            float acc = 0.f;
            int cnt = 0;
            for (int c = lane; c < nvec; c += FL) {
                acc = V::dot(V::load(orow + (int64_t)c * VEC), V::load(grow + (int64_t)c * VEC), acc);
                cnt += VEC;
                if (cnt >= kShardGradChunk) { hi += (double)acc; acc = 0.f; cnt = 0; }
            }
            hi += (double)acc;
        }
        for (int m = FL >> 1; m > 0; m >>= 1) hi += __shfl_xor_sync(0xffffffffu, hi, m);
        if (lane == 0) {
            g[p] = hi;
            g_out[p] = (float)hi;
        }
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    for (int p = 0; p < d.n; ++p) {
        const int64_t r = d.row[p] - row0, c = d.col[p] - row0;
        if (r == c) continue;                                // a diagonal flip enters only rho
        const double vg = (double)d.val[p] * g[p];
        if (r >= 0 && r < rows) r_out[r] += vg;
        if (c >= 0 && c < rows) q_out[c] += vg;
    }
}

// dLoss/dv_p of the flips whose row this rank owns, out[p] = grho_{r_p} + [r_p != c_p] ((float)(-a g_p) +
// gw_full[c_p]) (the arithmetic of shard_grad_entries_kernel), and 0 for every other flip: the caller
// adds the ranks' rows, so the owner's value reaches every rank unchanged.  One thread per flip.
__global__ void __launch_bounds__(EGNN_MAX_DELTA)
shard_grad_flip_values_kernel(DeltaList d, const float* __restrict__ g, const float* __restrict__ gw_full,
                              const float* __restrict__ grho, int64_t rows, int64_t row0, float a,
                              float* __restrict__ out) {
    const int p = threadIdx.x;
    if (p >= d.n) return;
    const int64_t r = d.row[p] - row0;
    const int c = d.col[p];
    float v = 0.f;
    if (r >= 0 && r < rows) {
        v = grho[r];
        if (r + row0 != c) v += (float)(-(double)a * (double)g[p]) + gw_full[c];
    }
    out[p] = v;
}

}  // namespace egnn

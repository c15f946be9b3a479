// Gradient of the wavelet pass w.r.t. the adjacency (DESIGN.md section 11).
//
// With M = a L + b I, L = I' - D^-1/2 A D^-1/2 (I' = the non-isolated diagonal, d = dinv), the
// adjoint vectors lambda_k = b_k of the Clenshaw pass (egnn_cheb_adjoint_all) and the forward's
// orders T_k:
//   g_ij   = sum_{k=1..K} m_k < d_i lambda_k[i,:], d_j T_{k-1}[j,:] >     (m_1 = 1, m_k = 2)
//   R_i    = sum_{j != i} A_ij g_ij,   Q_i = sum_{j != i} A_ji g_ji
//   gw_i   = (a/2) d_i^2 (R_i + Q_i)   (0 for an isolated node: d held at 1)
//   grho_i = Xbar_i / (1 + rho_i)      (default signal x0 = log1p(rho) only)
//   dA_ij  = [i != j] (-a g_ij + gw_j) + grho_i
// Operands come as stacks of K slabs [K, n, F]: lambda = b_1..b_K, T = T_0..T_{K-1}; element
// e = k * F + f of row i is own[k][i, f].  Every sum runs in a fixed order (float32 chunks, float64
// carry, no atomics): the results are bitwise reproducible.
#pragma once

#include "common.cuh"

namespace egnn {

constexpr int kStackChunk = 32;          // float32 partial sums cover this many products, then spill into fp64

// sum over e = lf, lf + FL, ... < K*F of m_k own[k][own_off + f] * gath[k][gath_off + f]
__device__ __forceinline__ double stack_dot(const float* __restrict__ own, const float* __restrict__ gath,
                                            int64_t own_off, int64_t gath_off, int64_t slab, int F, int K,
                                            int lf, int FL) {
    double hi = 0.0;
    float acc = 0.f;
    int cnt = 0;
    if (F >= FL) {
        for (int k = 0; k < K; ++k) {
            const float mk = k ? 2.f : 1.f;
            const float* o = own + (int64_t)k * slab + own_off;
            const float* g = gath + (int64_t)k * slab + gath_off;
            for (int f = lf; f < F; f += FL) {
                acc = fmaf(mk * __ldg(o + f), __ldg(g + f), acc);
                if (++cnt == kStackChunk) { hi += (double)acc; acc = 0.f; cnt = 0; }
            }
        }
    } else {                                             // narrow signals: lanes run across the orders
        const int KF = K * F;
        for (int e = lf; e < KF; e += FL) {
            const int k = e / F;
            const int f = e - k * F;
            const int64_t off = (int64_t)k * slab + f;
            acc = fmaf((k ? 2.f : 1.f) * __ldg(own + off + own_off), __ldg(gath + off + gath_off), acc);
            if (++cnt == kStackChunk) { hi += (double)acc; acc = 0.f; cnt = 0; }
        }
    }
    return hi + (double)acc;
}

// out[i] = d_i sum_{j != i, stored} A_ij d_j sum_k m_k <own_k[i], gath_k[j]>: R over the CSR with
// (lambda, T), Q over the transposed CSR with (T, lambda).  One warp per row, 32 >> fl_log2 entries
// side by side, 1 << fl_log2 lanes across the K*F products of an entry.
__global__ void __launch_bounds__(256)
adj_grad_degree_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                       const float* __restrict__ vals, const float* __restrict__ dinv, const float* __restrict__ own,
                       const float* __restrict__ gath, int64_t n, int32_t F, int32_t K, int32_t fl_log2,
                       double* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int FL = 1 << fl_log2;
    const int lf = lane & (FL - 1);
    const int grp = lane >> fl_log2;
    const int NZ = 32 >> fl_log2;
    const int64_t slab = n * (int64_t)F;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t row = warp; row < n; row += nwarps) {
        double s = 0.0;
        const int q1 = rowptr[row + 1];
        for (int q = rowptr[row] + grp; q < q1; q += NZ) {
            const int j = ld_stream_i32(colidx + q);
            if (j == row) continue;                          // stored self loops are not part of L
            const float w = (vals ? ld_stream_f32(vals + q) : 1.f) * __ldg(dinv + j);
            s = fma((double)w, stack_dot(own, gath, row * F, (int64_t)j * F, slab, F, K, lf, FL), s);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) out[row] = (double)dinv[row] * s;
    }
}

// gw = (a/2) d^2 (R + Q) (0 where isolated), grho = xbar / (1 + rowsum) (0 without xbar)
__global__ void __launch_bounds__(256)
adj_grad_finish_kernel(const double* __restrict__ r, const double* __restrict__ q, const float* __restrict__ dinv,
                       const uint8_t* __restrict__ iso, const float* __restrict__ xbar, const float* __restrict__ rowsum,
                       int64_t n, float a, float* __restrict__ gw, float* __restrict__ grho) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double d = (double)dinv[i];
        gw[i] = iso[i] ? 0.f : (float)(0.5 * (double)a * d * d * (r[i] + q[i]));
        grho[i] = xbar ? (float)((double)xbar[i] / (1.0 + (double)rowsum[i])) : 0.f;
    }
}

// out[p] = [r != c] (-a g_rc + gw_c) + grho_r for pairs (r, c) = (rows[p], cols[p]); 32 >> fl_log2
// pairs per warp, each reduced over its 1 << fl_log2 lanes in a fixed order.
__global__ void __launch_bounds__(256)
adj_grad_pairs_kernel(const int32_t* __restrict__ rows, const int32_t* __restrict__ cols, int64_t n_pairs,
                      const float* __restrict__ dinv, const float* __restrict__ lam, const float* __restrict__ t,
                      const float* __restrict__ gw, const float* __restrict__ grho, int64_t n, int32_t F, int32_t K,
                      int32_t fl_log2, float a, float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int FL = 1 << fl_log2;
    const int lf = lane & (FL - 1);
    const int grp = lane >> fl_log2;
    const int NZ = 32 >> fl_log2;
    const int64_t slab = n * (int64_t)F;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t base = warp * NZ; base < n_pairs; base += nwarps * NZ) {
        const int64_t p = base + grp;
        int r = 0, c = 0;
        double g = 0.0;
        if (p < n_pairs) {
            r = rows[p];
            c = cols[p];
            g = stack_dot(lam, t, (int64_t)r * F, (int64_t)c * F, slab, F, K, lf, FL);
        }
        for (int o = FL >> 1; o > 0; o >>= 1) g += __shfl_xor_sync(0xffffffffu, g, o);
        if (p < n_pairs && lf == 0) {
            float v = grho[r];
            if (r != c) v += (float)(-(double)a * (double)dinv[r] * (double)dinv[c] * g) + gw[c];
            out[p] = v;
        }
    }
}

// ---- dense [n, n] gradient: a tiled float32 outer product over the K*F products --------------------
// CTA tile 64 x 64, 256 threads of 4 x 4 outputs (rows 4 ty.., columns 4 tx..: one float4 store per
// row); the K*F dimension in chunks of 32 staged in shared memory, chunk totals carried in float64.
constexpr int kDenseTile = 64;
constexpr int kDenseChunk = 32;
constexpr int kDenseThreads = 256;

__global__ void __launch_bounds__(kDenseThreads)
adj_grad_dense_kernel(const float* __restrict__ lam, const float* __restrict__ t, const float* __restrict__ dinv,
                      const float* __restrict__ gw, const float* __restrict__ grho, int64_t n, int32_t F, int32_t K,
                      float a, float* __restrict__ out, int64_t ld, int32_t vec_ok) {
    __shared__ __align__(16) float As[kDenseChunk][kDenseTile];
    __shared__ __align__(16) float Bs[kDenseChunk][kDenseTile];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int64_t row0 = (int64_t)blockIdx.y * kDenseTile, col0 = (int64_t)blockIdx.x * kDenseTile;
    const int64_t slab = n * (int64_t)F;
    const int KF = K * F;
    float acc[4][4];
    double hi[4][4];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) { acc[r][c] = 0.f; hi[r][c] = 0.0; }
    for (int e0 = 0; e0 < KF; e0 += kDenseChunk) {
        const int ne = min(kDenseChunk, KF - e0);
        __syncthreads();
        for (int idx = threadIdx.x; idx < kDenseChunk * kDenseTile; idx += kDenseThreads) {
            const int r = idx & (kDenseTile - 1), el = idx >> 6;
            const int e = e0 + el;
            float va = 0.f, vb = 0.f;
            if (el < ne) {
                const int k = e / F;
                const int64_t off = (int64_t)k * slab + (e - k * F);
                const int64_t i = row0 + r, j = col0 + r;
                if (i < n) va = (k ? 2.f : 1.f) * dinv[i] * __ldg(lam + off + i * F);
                if (j < n) vb = dinv[j] * __ldg(t + off + j * F);
            }
            As[el][r] = va;
            Bs[el][r] = vb;
        }
        __syncthreads();
        for (int ee = 0; ee < ne; ++ee) {
            const float4 av = *reinterpret_cast<const float4*>(&As[ee][ty * 4]);
            const float4 bv = *reinterpret_cast<const float4*>(&Bs[ee][tx * 4]);
            const float ar[4] = {av.x, av.y, av.z, av.w}, bc[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[r][c] = fmaf(ar[r], bc[c], acc[r][c]);
        }
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int c = 0; c < 4; ++c) { hi[r][c] += (double)acc[r][c]; acc[r][c] = 0.f; }
    }
    const int64_t j0 = col0 + tx * 4;
    float gwc[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) gwc[c] = j0 + c < n ? gw[j0 + c] : 0.f;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int64_t i = row0 + ty * 4 + r;
        if (i >= n) break;
        const float gr = grho[i];
        float v[4];
#pragma unroll
        for (int c = 0; c < 4; ++c)
            v[c] = (j0 + c == i ? 0.f : (float)(-(double)a * hi[r][c]) + gwc[c]) + gr;
        float* dst = out + i * ld + j0;
        if (vec_ok && j0 + 3 < n) {
            __stcs(reinterpret_cast<float4*>(dst), make_float4(v[0], v[1], v[2], v[3]));
        } else {
#pragma unroll
            for (int c = 0; c < 4; ++c)
                if (j0 + c < n) __stcs(dst + c, v[c]);
        }
    }
}

}  // namespace egnn

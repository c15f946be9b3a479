// Backward of the wavelet pass (the adjoint order kernels themselves are the ADJ
// instantiations of cheb.cuh / wide.cuh): the Clenshaw prologue, the out-of-place
// row L1 normalisation and its backward, the heat-coefficient gradient and the
// CSR transpose the adjoint gathers over.
//
// Adjoint pass, M = a L + b I, C_s = sum_k alpha[s,k] T_k(M) X:
//   v_k = sum_s alpha[s,k] Cbar_s + Tbar_k,
//   b_K = v_K,  b_k = v_k + 2 M^T b_{k+1} - b_{k+2} (k = K-1..1),  Xbar = v_0 + M^T b_1 - b_2:
// K operator applications whatever S is.
#pragma once

#include "common.cuh"
#include "peer.cuh"

namespace egnn {

struct CoefRow {
    float c[EGNN_MAX_SCALES];
};

// b_K = v_K = tbar + sum_s c[s] * cbar[:, s, :] into b_out [n, F] (K = 0: that is the signal's gradient)
// and dinv (.) b_K into y_out [n, ldy] (columns F..ldy-1 zeroed), either may be NULL.
// The sum runs in the order of the adjoint epilogues.
__global__ void __launch_bounds__(256)
adjoint_prologue_kernel(const float* __restrict__ cbar, const float* __restrict__ tbar, const float* __restrict__ dinv,
                        float* __restrict__ b_out, float* __restrict__ y_out, int64_t n, int32_t F, int32_t S,
                        int32_t ldy, const __grid_constant__ CoefRow c) {
    const int64_t total = n * ldy;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / ldy;
        const int col = (int)(i - r * ldy);
        float v = 0.f;
        if (col < F) {
            if (tbar) v = tbar[r * F + col];
            for (int s = 0; s < S; ++s) v = fmaf(c.c[s], cbar[(r * S + s) * F + col], v);
            if (b_out) b_out[r * F + col] = v;
        }
        if (y_out) y_out[i] = dinv[r] * v;
    }
}

// Row-sharded twin of adjoint_prologue_kernel + peer_prescale_push_kernel: v_K of the local rows
// (same sum order), dinv (.) v_K stored into operand buffer 0 of every rank's window (rows ldy wide,
// padding zeroed) once every peer has finished the kernels before it, then signalled.
__global__ void __launch_bounds__(1024)
adjoint_prologue_push_kernel(const float* __restrict__ cbar, const float* __restrict__ tbar,
                             const float* __restrict__ dinv_full, int64_t n_rows, int64_t row0, int32_t F, int32_t S,
                             int32_t ldy, const __grid_constant__ CoefRow c, const __grid_constant__ PeerPush pp) {
    peer_producer_wait_first(pp);
    const int64_t total = n_rows * ldy;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / ldy;
        const int col = (int)(i - r * ldy);
        float v = 0.f;
        if (col < F) {
            if (tbar) v = tbar[r * F + col];
            for (int s = 0; s < S; ++s) v = fmaf(c.c[s], cbar[(r * S + s) * F + col], v);
        }
        const float y = dinv_full[row0 + r] * v;
        for (int p = 0; p < pp.world; ++p) pp.dst[p][(row0 + r) * ldy + col] = y;
    }
    peer_producer_signal(pp);
}

// h[r, :] = c[r, :] / (sum_f |c[r, f]| + 1e-8), one warp per row vector (as l1_normalize_kernel)
__global__ void __launch_bounds__(256)
l1_normalize_out_kernel(const float* __restrict__ c, float* __restrict__ h, int64_t n_vec, int32_t F) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < n_vec; r += nwarps) {
        const float* row = c + r * F;
        float s = 0.f;
        for (int f = lane; f < F; f += 32) s += fabsf(row[f]);
        s = warp_sum(s);
        const float inv = 1.f / (s + 1e-8f);
        for (int f = lane; f < F; f += 32) h[r * F + f] = row[f] * inv;
    }
}

// cbar_out = cbar_in + (hbar - sign(c) <hbar, h>) / r with h = c / r, r = sum_f |c| + 1e-8 recomputed
// from c (sign(0) = 0).  cbar_in may be NULL (zero) or alias cbar_out.
__global__ void __launch_bounds__(256)
l1_normalize_backward_kernel(const float* __restrict__ c, const float* __restrict__ hbar, const float* cbar_in,
                             float* cbar_out, int64_t n_vec, int32_t F) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < n_vec; r += nwarps) {
        const float* row = c + r * F;
        const float* g = hbar + r * F;
        float s = 0.f;
        for (int f = lane; f < F; f += 32) s += fabsf(row[f]);
        s = warp_sum(s);
        const float inv = 1.f / (s + 1e-8f);
        float d = 0.f;
        for (int f = lane; f < F; f += 32) d = fmaf(g[f], row[f] * inv, d);
        d = warp_sum(d);
        for (int f = lane; f < F; f += 32) {
            const float x = row[f];
            const float sg = x > 0.f ? 1.f : (x < 0.f ? -1.f : 0.f);
            const float base = cbar_in ? cbar_in[r * F + f] : 0.f;
            cbar_out[r * F + f] = base + (g[f] - sg * d) * inv;
        }
    }
}

// ---- heat-coefficient gradient: G[s, k] = <cbar[:, s, :], T_k> ------------------------------------
// A fixed number of CTAs, each summing a fixed row range in float64; CTA partials are added in CTA
// order by coeff_grad_finish_kernel, so the result does not depend on the device or the launch.
constexpr int kCoefGradBlocks = 296;
constexpr int kCoefGradThreads = 256;

__global__ void __launch_bounds__(kCoefGradThreads)
coeff_grad_partial_kernel(const float* __restrict__ cbar, const float* __restrict__ t_all, int64_t n, int32_t F,
                          int32_t K, int32_t S, double* __restrict__ partial) {
    __shared__ double red[kCoefGradThreads / 32][EGNN_MAX_SCALES];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int64_t chunk = ceil_div64(n, gridDim.x);
    const int64_t e0 = min(n, (int64_t)blockIdx.x * chunk) * F;
    const int64_t e1 = min(n, (int64_t)(blockIdx.x + 1) * chunk) * F;
    const int64_t slab = n * (int64_t)F;
    for (int k = 0; k <= K; ++k) {
        double acc[EGNN_MAX_SCALES];
#pragma unroll
        for (int s = 0; s < EGNN_MAX_SCALES; ++s) acc[s] = 0.0;
        for (int64_t e = e0 + threadIdx.x; e < e1; e += blockDim.x) {
            const int64_t r = e / F;
            const int64_t f = e - r * F;
            const double t = (double)t_all[(int64_t)k * slab + e];
#pragma unroll
            for (int s = 0; s < EGNN_MAX_SCALES; ++s)
                if (s < S) acc[s] = fma((double)cbar[(r * S + s) * F + f], t, acc[s]);
        }
#pragma unroll
        for (int s = 0; s < EGNN_MAX_SCALES; ++s) {
            if (s >= S) break;
            double v = acc[s];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0) red[wid][s] = v;
        }
        __syncthreads();
        if (threadIdx.x < S) {
            double v = 0.0;
            for (int w = 0; w < kCoefGradThreads / 32; ++w) v += red[w][threadIdx.x];
            partial[((int64_t)blockIdx.x * S + threadIdx.x) * (K + 1) + k] = v;
        }
        __syncthreads();
    }
}

__global__ void coeff_grad_finish_kernel(const double* __restrict__ partial, int n_blocks, int n_out,
                                         double* __restrict__ out) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n_out) return;
    double v = 0.0;
    for (int b = 0; b < n_blocks; ++b) v += partial[(int64_t)b * n_out + q];
    out[q] = v;
}

// ---- CSR transpose -------------------------------------------------------------------------------
// entry ids 0..nnz-1 (the sort's values) and the entry count of every column
__global__ void __launch_bounds__(256)
transpose_count_kernel(const int32_t* __restrict__ colidx, int64_t nnz, int32_t* __restrict__ ids,
                       int32_t* __restrict__ counts) {
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nnz; q += (int64_t)gridDim.x * blockDim.x) {
        ids[q] = (int32_t)q;
        atomicAdd(counts + colidx[q], 1);
    }
}

// entry p of the transpose is entry ids_sorted[p] of the CSR: its row (found by binary search in
// rowptr) becomes the column
__global__ void __launch_bounds__(256)
transpose_fill_kernel(const int32_t* __restrict__ rowptr, int64_t n, const float* __restrict__ vals,
                      const int32_t* __restrict__ ids_sorted, int64_t nnz, int32_t* __restrict__ colidx_t,
                      float* __restrict__ vals_t) {
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < nnz; p += (int64_t)gridDim.x * blockDim.x) {
        const int32_t q = ids_sorted[p];
        int64_t lo = 0, hi = n;                  // last row r with rowptr[r] <= q
        while (hi - lo > 1) {
            const int64_t mid = (lo + hi) >> 1;
            if (rowptr[mid] <= q) lo = mid; else hi = mid;
        }
        colidx_t[p] = (int32_t)lo;
        if (vals_t) vals_t[p] = vals[q];
    }
}

}  // namespace egnn

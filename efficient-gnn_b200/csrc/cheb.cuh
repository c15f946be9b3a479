// Fused Chebyshev-order kernel: CSR SpMM over the scaled normalised Laplacian
// with the degree scaling applied on the fly, the three-term recurrence in the
// epilogue and all wavelet scales accumulated in the same pass.
// Reference semantics: calibration/WATS.py:29-37 (recurrence), :55 (rescale),
// :65-68 (combination), :71-72 (row L1 normalisation).
//
// HBM/L2-bound gather kernel - CUDA cores only (not a dense contraction).
// Lane layout inside a warp (all powers of two, chosen on the host):
//     rows_per_warp x NZ (non-zeros in parallel) x FL (feature lanes)
// each feature lane owns U groups of VEC consecutive features (VEC=4 -> 128-bit
// gathers of T_{k-1} rows); partial sums of the NZ lanes meet through xor
// shuffles, then the NZ==0 lanes run the epilogue for their features.
#pragma once

#include "common.cuh"
#include "prep.cuh"

namespace egnn {

struct OrderParams {
    // CSR of the rows this launch owns (local row r <-> global node row0 + r)
    const int32_t* rowptr;
    const int32_t* colidx;
    const float* vals;       // NULL: binary adjacency
    const float* dinv;       // [n_global] 1/sqrt(w), 1 for isolated
    const uint8_t* iso;      // [n_global]
    const float* gsrc;       // gather source indexed by GLOBAL column: T_{k-1}, or dinv*T_{k-1} (PRESCALED)
    const float* tprev_own;  // [n_rows, F] T_{k-1} rows of this launch
    const float* tprev2_own; // [n_rows, F] T_{k-2}; may alias tk_own (read-then-write per element)
    float* tk_own;           // [n_rows, F] or NULL
    float* y_own;            // [n_rows, F] dinv*T_k for the next order's gathers, or NULL
    float* out;              // [n_rows, S, F]
    float* acc_ws;           // [n_rows, F] partial sums (split launches)
    int64_t n_rows;
    int64_t row0;
    int32_t F;
    int32_t S;
    float a;                 // operator = a * L_sym + b * I  (reference: a = 2/lambda_max = 1, b = -1)
    float b;
    int32_t first;           // order 1: T_1 = L~ T_0, out = c0*T_0 + c1*T_1
    int32_t normalize;       // last order, fuse the row L1 normalisation (needs gridDim.y == 1)
    int32_t mode;            // 0: whole order; 1: partial sums -> acc_ws; 2: add acc_ws, then epilogue
    int32_t fl_log2;
    int32_t nz_log2;
    float c_prev[EGNN_MAX_SCALES];
    float c_k[EGNN_MAX_SCALES];
    DeltaList delta;
    // adjoint instantiation (ADJ): b = c_adj * (M^T b_{k+1})_i - b_{k+2} + v_k with
    // v_k[i, :] = tbar[i, :] + sum_s c_k[s] * cbar[i, s, :]; tprev_own = b_{k+1}, tprev2_own = b_{k+2}
    // (NULL: zero), tk_own = b_k, y_own = dinv * b_k.  Appended so the forward layout is unchanged.
    const float* cbar;       // [n_rows, S, F]
    const float* tbar;       // [n_rows, F] or NULL
    float c_adj;             // 2, or 1 on the last application (it yields the signal's gradient)
};

template <int VEC> struct FeatVec;
template <> struct FeatVec<1> {
    float v[1];
    __device__ __forceinline__ void load(const float* p) { v[0] = __ldg(p); }
    __device__ __forceinline__ void load_plain(const float* p) { v[0] = *p; }
    __device__ __forceinline__ void store(float* p) const { *p = v[0]; }
};
template <> struct FeatVec<4> {
    float v[4];
    __device__ __forceinline__ void load(const float* p) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(p));
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    }
    __device__ __forceinline__ void load_plain(const float* p) {
        const float4 t = *reinterpret_cast<const float4*>(p);
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    }
    __device__ __forceinline__ void store(float* p) const {
        *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    }
};

constexpr int kOrderBlock = 256;
constexpr int kNzUnroll = 4;
constexpr int kChunkIters = 16;          // fp32 partial sums cover <= 64 entries, then spill into fp64
constexpr int kLongRowIters = 8;         // rows needing more loop trips than this go to the whole warp

// One lane's share of a row: entries q_first, q_first + stride, ... < q_end.
// Two-level summation: float32 FMAs over chunks of kChunkIters * kNzUnroll
// entries, chunk totals added in float64 (the reference (scipy) accumulates in float64;
// long rows of equal addends would otherwise round the same way every step).
template <int VEC, int U, bool HAS_VALS, bool PRESCALED>
__device__ __forceinline__ void accumulate_row(const OrderParams& p, int q_first, int q_end, int stride,
                                               int grow, const int (&fidx)[U], const bool (&fok)[U],
                                               float (&acc)[U][VEC]) {
    const int F = p.F;
    double hi[U][VEC];
#pragma unroll
    for (int u = 0; u < U; ++u)
#pragma unroll
        for (int v = 0; v < VEC; ++v) { hi[u][v] = 0.0; acc[u][v] = 0.f; }
    int q0 = q_first;
    while (q0 < q_end) {
        for (int it = 0; it < kChunkIters && q0 < q_end; ++it, q0 += stride * kNzUnroll) {
            int c[kNzUnroll];
            float w[kNzUnroll];
#pragma unroll
            for (int j = 0; j < kNzUnroll; ++j) {
                const int q = q0 + j * stride;
                const bool ok = q < q_end;
                c[j] = ok ? ld_stream_i32(p.colidx + q) : grow;
                float wv = 0.f;
                if (ok) wv = HAS_VALS ? ld_stream_f32(p.vals + q) : 1.f;
                w[j] = wv;
            }
#pragma unroll
            for (int j = 0; j < kNzUnroll; ++j) {
                if (c[j] == grow) w[j] = 0.f;                  // stored self loops are not part of L
                if (!PRESCALED) w[j] *= __ldg(p.dinv + c[j]);
            }
#pragma unroll
            for (int j = 0; j < kNzUnroll; ++j) {
                const float* src = p.gsrc + (int64_t)c[j] * F;
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    if (fok[u]) {
                        FeatVec<VEC> x;
                        x.load(src + fidx[u]);
#pragma unroll
                        for (int v = 0; v < VEC; ++v) acc[u][v] = fmaf(w[j], x.v[v], acc[u][v]);
                    }
                }
            }
        }
        if (q0 < q_end) {                                       // more chunks follow: spill
#pragma unroll
            for (int u = 0; u < U; ++u)
#pragma unroll
                for (int v = 0; v < VEC; ++v) { hi[u][v] += (double)acc[u][v]; acc[u][v] = 0.f; }
        }
    }
#pragma unroll
    for (int u = 0; u < U; ++u)
#pragma unroll
        for (int v = 0; v < VEC; ++v) acc[u][v] = (float)(hi[u][v] + (double)acc[u][v]);
}

template <int VEC, int U, bool HAS_VALS, bool PRESCALED, bool ADJ = false>
__global__ void __launch_bounds__(kOrderBlock)
cheb_order_kernel(const __grid_constant__ OrderParams p) {
    const int lane = threadIdx.x & 31;
    const int FL = 1 << p.fl_log2;
    const int NZ = 1 << p.nz_log2;
    const int glog = p.fl_log2 + p.nz_log2;
    const int group = 1 << glog;
    const int rows_per_warp = 32 >> glog;
    const int sub = lane >> glog;
    const int gl = lane & (group - 1);
    const int fl = gl & (FL - 1);
    const int nzl = gl >> p.fl_log2;
    const int F = p.F;

    const int64_t warp_global = (int64_t)blockIdx.x * (kOrderBlock / 32) + (threadIdx.x >> 5);
    const int64_t row = warp_global * rows_per_warp + sub;
    const bool row_ok = row < p.n_rows;
    const int grow = (int)(p.row0 + (row_ok ? row : 0));
    const int f_tile = blockIdx.y * (FL * VEC * U);

    int fidx[U];
    bool fok[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
        fidx[u] = f_tile + (u * FL + fl) * VEC;
        fok[u] = fidx[u] < F;
    }

    int start = 0, end = 0;
    if (row_ok) {
        start = __ldg(p.rowptr + row);
        end = __ldg(p.rowptr + row + 1);
    }

    // rows of ordinary length: the row's lane group walks it; hub rows are
    // deferred to the whole warp (warp-per-row), so one lane group never
    // serialises tens of thousands of entries.
    const bool is_long = (group < 32) && (end - start > NZ * kNzUnroll * kLongRowIters);
    float acc[U][VEC];
    accumulate_row<VEC, U, HAS_VALS, PRESCALED>(p, start + nzl, is_long ? start : end, NZ, grow, fidx, fok, acc);
    for (int o = FL; o < group; o <<= 1) {
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int v = 0; v < VEC; ++v) acc[u][v] += __shfl_xor_sync(0xffffffffu, acc[u][v], o);
    }
    unsigned long_mask = __ballot_sync(0xffffffffu, is_long && gl == 0);
    while (long_mask) {
        const int leader = __ffs(long_mask) - 1;
        long_mask &= long_mask - 1;
        const int l_start = __shfl_sync(0xffffffffu, start, leader);
        const int l_end = __shfl_sync(0xffffffffu, end, leader);
        const int l_grow = __shfl_sync(0xffffffffu, grow, leader);
        float part[U][VEC];
        accumulate_row<VEC, U, HAS_VALS, PRESCALED>(p, l_start + (lane >> p.fl_log2), l_end, 32 >> p.fl_log2,
                                                    l_grow, fidx, fok, part);
        for (int o = FL; o < 32; o <<= 1) {
#pragma unroll
            for (int u = 0; u < U; ++u)
#pragma unroll
                for (int v = 0; v < VEC; ++v) part[u][v] += __shfl_xor_sync(0xffffffffu, part[u][v], o);
        }
        if (sub == (leader >> glog)) {
#pragma unroll
            for (int u = 0; u < U; ++u)
#pragma unroll
                for (int v = 0; v < VEC; ++v) acc[u][v] = part[u][v];
        }
    }

    const bool writer = row_ok && (nzl == 0);

    // edge flips on top of the CSR (UGCA recompute); tiny host-provided list
    if (p.delta.n > 0 && writer) {
        for (int e = 0; e < p.delta.n; ++e) {
            if (p.delta.row[e] == grow && p.delta.col[e] != grow) {
                const int c = p.delta.col[e];
                float w = p.delta.val[e];
                if (!PRESCALED) w *= __ldg(p.dinv + c);
                const float* src = p.gsrc + (int64_t)c * F;
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    if (fok[u]) {
                        FeatVec<VEC> x;
                        x.load(src + fidx[u]);
#pragma unroll
                        for (int v = 0; v < VEC; ++v) acc[u][v] = fmaf(w, x.v[v], acc[u][v]);
                    }
                }
            }
        }
    }

    if (p.mode == 1) {           // first half of a split order: park the partial sums
        if (writer) {
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (fok[u]) {
                    FeatVec<VEC> t;
#pragma unroll
                    for (int v = 0; v < VEC; ++v) t.v[v] = acc[u][v];
                    t.store(p.acc_ws + row * F + fidx[u]);
                }
        }
        return;
    }
    if (p.mode == 2 && writer) {
#pragma unroll
        for (int u = 0; u < U; ++u)
            if (fok[u]) {
                FeatVec<VEC> t;
                t.load_plain(p.acc_ws + row * F + fidx[u]);
#pragma unroll
                for (int v = 0; v < VEC; ++v) acc[u][v] += t.v[v];
            }
    }

    if constexpr (ADJ) {         // adjoint epilogue (Clenshaw step): no scale accumulation
        if (!writer) return;
        const float di = __ldg(p.dinv + grow);
        const float theta = fmaf(p.a, 1.f - (float)__ldg(p.iso + grow), p.b);
        const float nscale = -p.a * di;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (!fok[u]) continue;
            const int64_t off = row * F + fidx[u];
            FeatVec<VEC> own, b2, v, t;
#pragma unroll
            for (int j = 0; j < VEC; ++j) { own.v[j] = 0.f; b2.v[j] = 0.f; v.v[j] = 0.f; }
            if (theta != 0.f) own.load_plain(p.tprev_own + off);
            if (p.tprev2_own) b2.load_plain(p.tprev2_own + off);
            if (p.tbar) v.load_plain(p.tbar + off);
            for (int s = 0; s < p.S; ++s) {
                t.load_plain(p.cbar + (row * p.S + s) * F + fidx[u]);
#pragma unroll
                for (int j = 0; j < VEC; ++j) v.v[j] = fmaf(p.c_k[s], t.v[j], v.v[j]);
            }
#pragma unroll
            for (int j = 0; j < VEC; ++j)
                t.v[j] = fmaf(p.c_adj, fmaf(theta, own.v[j], nscale * acc[u][j]), v.v[j] - b2.v[j]);
            if (p.tk_own) t.store(p.tk_own + off);       // may alias tprev2_own: read above
            if (p.y_own) {
#pragma unroll
                for (int j = 0; j < VEC; ++j) t.v[j] *= di;
                t.store(p.y_own + off);
            }
        }
        return;
    }

    // ---- epilogue: Laplacian scaling, recurrence, scale accumulation -------
    float di = 1.f, theta = 0.f;
    if (writer) {
        di = __ldg(p.dinv + grow);
        theta = fmaf(p.a, 1.f - (float)__ldg(p.iso + grow), p.b);
    }
    const float nscale = -p.a * di;
    float tk[U][VEC];
    float xprev[U][VEC];
#pragma unroll
    for (int u = 0; u < U; ++u) {
#pragma unroll
        for (int v = 0; v < VEC; ++v) { tk[u][v] = 0.f; xprev[u][v] = 0.f; }
        if (writer && fok[u]) {
            const int64_t off = row * F + fidx[u];
            if (theta != 0.f || p.first) {
                FeatVec<VEC> t;
                t.load_plain(p.tprev_own + off);
#pragma unroll
                for (int v = 0; v < VEC; ++v) xprev[u][v] = t.v[v];
            }
            FeatVec<VEC> t2;
#pragma unroll
            for (int v = 0; v < VEC; ++v) t2.v[v] = 0.f;
            if (!p.first) t2.load_plain(p.tprev2_own + off);
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                const float lap = fmaf(theta, xprev[u][v], nscale * acc[u][v]);
                tk[u][v] = p.first ? lap : fmaf(2.f, lap, -t2.v[v]);
            }
            FeatVec<VEC> o;
            if (p.tk_own) {
#pragma unroll
                for (int v = 0; v < VEC; ++v) o.v[v] = tk[u][v];
                o.store(p.tk_own + off);
            }
            if (p.y_own) {
#pragma unroll
                for (int v = 0; v < VEC; ++v) o.v[v] = di * tk[u][v];
                o.store(p.y_own + off);
            }
        }
    }

    for (int s = 0; s < p.S; ++s) {
        float o[U][VEC];
        float l1 = 0.f;
#pragma unroll
        for (int u = 0; u < U; ++u) {
#pragma unroll
            for (int v = 0; v < VEC; ++v) o[u][v] = 0.f;
            if (writer && fok[u]) {
                const int64_t off = (row * p.S + s) * F + fidx[u];
                if (p.first) {
#pragma unroll
                    for (int v = 0; v < VEC; ++v)
                        o[u][v] = fmaf(p.c_k[s], tk[u][v], p.c_prev[s] * xprev[u][v]);
                } else {
                    FeatVec<VEC> t;
                    t.load_plain(p.out + off);
#pragma unroll
                    for (int v = 0; v < VEC; ++v) o[u][v] = fmaf(p.c_k[s], tk[u][v], t.v[v]);
                }
#pragma unroll
                for (int v = 0; v < VEC; ++v) l1 += fabsf(o[u][v]);
            }
        }
        if (p.normalize) {       // uniform branch: every lane takes part in the shuffles
            for (int off = 1; off < FL; off <<= 1) l1 += __shfl_xor_sync(0xffffffffu, l1, off);
            const float inv = 1.f / (l1 + 1e-8f);
#pragma unroll
            for (int u = 0; u < U; ++u)
#pragma unroll
                for (int v = 0; v < VEC; ++v) o[u][v] *= inv;
        }
        if (writer) {
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (fok[u]) {
                    FeatVec<VEC> t;
#pragma unroll
                    for (int v = 0; v < VEC; ++v) t.v[v] = o[u][v];
                    t.store(p.out + (row * p.S + s) * F + fidx[u]);
                }
        }
    }
}

// out[i, s, :] /= (sum_f |out[i, s, f]| + 1e-8): used when one warp tile does
// not span the whole feature row (F > 128) and for K == 0.
__global__ void __launch_bounds__(256)
l1_normalize_kernel(float* __restrict__ out, int64_t n_vec, int32_t F) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < n_vec; r += nwarps) {
        float* row = out + r * F;
        float s = 0.f;
        for (int f = lane; f < F; f += 32) s += fabsf(row[f]);
        s = warp_sum(s);
        const float inv = 1.f / (s + 1e-8f);
        for (int f = lane; f < F; f += 32) row[f] *= inv;
    }
}

// K == 0: out[i, s, :] = c0[s] * x0[i, :]
__global__ void __launch_bounds__(256)
order0_kernel(const float* __restrict__ x0, float* __restrict__ out, int64_t n, int32_t F, int32_t S,
              const __grid_constant__ OrderParams p) {
    const int64_t total = n * S * F;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int f = (int)(i % F);
        const int s = (int)((i / F) % S);
        const int64_t r = i / ((int64_t)F * S);
        out[i] = p.c_prev[s] * x0[r * F + f];
    }
}

// y = dinv (.) x, row-wise (gather operand of the first order in PRESCALED mode)
__global__ void __launch_bounds__(256)
prescale_kernel(const float* __restrict__ x, const float* __restrict__ dinv, float* __restrict__ y,
                int64_t n, int32_t F, int64_t row0) {
    const int64_t total = n * F;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x)
        y[i] = dinv[row0 + i / F] * x[i];
}

}  // namespace egnn

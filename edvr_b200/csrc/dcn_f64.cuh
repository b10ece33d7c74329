// dcn_f64.cuh — double-precision DCNv2 / DCNv1 operator (forward and backward), NCHW fp64 in / out.
//
// The fp64 counterpart of dcn_fused.cuh + dcn_backward.cuh for callers that hand the operator `double` tensors (the
// reference dispatches its kernels on double as well).  Every quantity stays in fp64: sample coordinates, bilinear weights,
// masks, products and accumulators.  No tcgen05 (it has no f64 kind): the three GEMMs run on the fp64 tensor-core path,
// mma.sync m8n8k4 .f64 (DMMA), from one tiled kernel with per-operand gather functors.  Any kh x kw, per-axis stride / pad /
// dilation, any C, Cout and dg with C % dg == 0.
//   forward : out[n][co][p]  = bias[co] + sum_{c,k} W[co][c][k] * S(n, c, k, p)                 (S gathered in the loader)
//   gcol    : gcol[n][c*K+k][p] = sum_co W[co][c][k] * gO[n][co][p]                            (a chunk of images at a time)
//   coord   : grad_offset / grad_mask, one thread per (n, dg, tap, pixel), channels reduced in order; grad_x scatter
//             with fp64 atomics
//   wgrad   : part[s][co][c*K+k] = sum_{q in split s} gO[q][co] * S(q, c, k); grad_weight += scale * sum_s part[s] in
//             split order (bit-reproducible); grad_bias += fixed-order sum over pixels
// S = bilinear sample of x at the offset position times the mask (1 for DCNv1).  Borders as dcn_backward.cuh and the
// reference: a sample outside (-1, H) x (-1, W) is zero, partial corners are used where in bounds, and the coordinate
// gradient is zero at coordinate -1.
#pragma once
#include "common.cuh"

namespace eb {

struct F64Geom {
    int N, C, H, W, Cout, kh, kw, sh, sw, ph, pw, dh, dw, dg, Ho, Wo;
};

constexpr int F64_BM = 64, F64_BN = 64, F64_BK = 16, F64_THREADS = 256, F64_LD = F64_BM + 8;   // +8: conflict-free rows

__device__ __forceinline__ void dmma_m8n8k4(double (&d)[2], double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
                 : "+d"(d[0]), "+d"(d[1])
                 : "d"(a), "d"(b));
}

// Bilinear sample position of (image n, deformable group g, tap k, output pixel p); false when outside (-1, H) x (-1, W).
struct F64Pos {
    double h, w, mk;
};
__device__ __forceinline__ bool f64_position(const F64Geom& G, const double* __restrict__ offset,
                                             const double* __restrict__ mask, int n, int g, int k, int p, F64Pos* s) {
    const int K = G.kh * G.kw, HW = G.Ho * G.Wo;
    const int ho = p / G.Wo, wo = p - ho * G.Wo, ki = k / G.kw, kj = k - ki * G.kw;
    const size_t ob = (static_cast<size_t>(n) * G.dg + g) * 2 * K * HW + p;
    s->h = static_cast<double>(ho * G.sh - G.ph + ki * G.dh) + __ldg(offset + ob + static_cast<size_t>(2 * k) * HW);
    s->w = static_cast<double>(wo * G.sw - G.pw + kj * G.dw) + __ldg(offset + ob + static_cast<size_t>(2 * k + 1) * HW);
    s->mk = mask ? __ldg(mask + ((static_cast<size_t>(n) * G.dg + g) * K + k) * HW + p) : 1.0;
    return s->h > -1.0 && s->w > -1.0 && s->h < static_cast<double>(G.H) && s->w < static_cast<double>(G.W);
}

// The four corners of a sample (zero where out of bounds) and their bilinear weights.
struct F64Corners {
    int hl, wl;
    bool t, b, l, r;
    double lh, lw, hh, hw;
};
__device__ __forceinline__ F64Corners f64_corners(const F64Geom& G, double h, double w) {
    F64Corners q;
    const double hf = floor(h), wf = floor(w);
    q.hl = static_cast<int>(hf);
    q.wl = static_cast<int>(wf);
    q.lh = h - hf;
    q.lw = w - wf;
    q.hh = 1.0 - q.lh;
    q.hw = 1.0 - q.lw;
    q.t = q.hl >= 0;
    q.b = q.hl + 1 <= G.H - 1;
    q.l = q.wl >= 0;
    q.r = q.wl + 1 <= G.W - 1;
    return q;
}

// S(n, c, k, p): masked bilinear sample of channel c
__device__ __forceinline__ double f64_sample(const F64Geom& G, const double* __restrict__ x, const double* __restrict__ offset,
                                             const double* __restrict__ mask, int n, int c, int k, int p) {
    F64Pos s;
    if (!f64_position(G, offset, mask, n, c / (G.C / G.dg), k, p, &s)) return 0.0;
    const F64Corners q = f64_corners(G, s.h, s.w);
    const double* xc = x + (static_cast<size_t>(n) * G.C + c) * G.H * G.W;
    const size_t o = static_cast<size_t>(q.hl) * G.W + q.wl;
    const double v1 = (q.t && q.l) ? __ldg(xc + o) : 0.0;
    const double v2 = (q.t && q.r) ? __ldg(xc + o + 1) : 0.0;
    const double v3 = (q.b && q.l) ? __ldg(xc + o + G.W) : 0.0;
    const double v4 = (q.b && q.r) ? __ldg(xc + o + G.W + 1) : 0.0;
    return (q.hh * q.hw * v1 + q.hh * q.lw * v2 + q.lh * q.hw * v3 + q.lh * q.lw * v4) * s.mk;
}

// ---- C[m][n] = sum_k A(k, m) * B(k, n), one 64 x 64 tile per CTA, K in steps of 16 through shared memory.
// Op supplies the operands, the K range of blockIdx.z and the store:
//   M, N; k_range(z, &k0, &k1); a(z, k, m); b(z, k, n); store(z, m, n, v); A_K_FAST / B_K_FAST pick the loader's thread
//   order (true: consecutive threads walk k, the contiguous index of that operand in memory).
template <class Op>
__global__ void __launch_bounds__(F64_THREADS) f64_gemm_kernel(const Op op) {
    __shared__ double As[F64_BK][F64_LD];
    __shared__ double Bs[F64_BK][F64_LD];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = warp & 1, wn = warp >> 1;                 // 2 x 4 warps, 32 x 16 outputs each
    const int m0 = blockIdx.x * F64_BM, n0 = blockIdx.y * F64_BN, z = blockIdx.z;
    int k0, k1;
    op.k_range(z, &k0, &k1);

    double acc[4][2][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    // element e (0..3) of this thread's share of a 16 x 64 operand slab
    auto slot = [&](bool k_fast, int e, int* kk, int* mm) {
        if (k_fast) { *kk = tid & 15; *mm = (tid >> 4) + 16 * e; }
        else        { *kk = (tid >> 6) + 4 * e; *mm = tid & 63; }
    };
    double ra[4], rb[4];
    auto fetch = [&](int kb) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            int kk, mm;
            slot(Op::A_K_FAST, e, &kk, &mm);
            const int k = kb + kk, m = m0 + mm;
            ra[e] = (k < k1 && m < op.M) ? op.a(z, k, m) : 0.0;
            slot(Op::B_K_FAST, e, &kk, &mm);
            const int kn = kb + kk, n = n0 + mm;
            rb[e] = (kn < k1 && n < op.N) ? op.b(z, kn, n) : 0.0;
        }
    };
    auto stash = [&]() {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            int kk, mm;
            slot(Op::A_K_FAST, e, &kk, &mm);
            As[kk][mm] = ra[e];
            slot(Op::B_K_FAST, e, &kk, &mm);
            Bs[kk][mm] = rb[e];
        }
    };

    if (k0 < k1) fetch(k0);
    for (int kb = k0; kb < k1; kb += F64_BK) {
        stash();
        __syncthreads();
        if (kb + F64_BK < k1) fetch(kb + F64_BK);            // next slab's loads in flight during the MMAs
#pragma unroll
        for (int kq = 0; kq < F64_BK; kq += 4) {
            const int kr = kq + (lane & 3);
            double a[4], b[2];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = As[kr][wm * 32 + i * 8 + (lane >> 2)];
#pragma unroll
            for (int j = 0; j < 2; ++j) b[j] = Bs[kr][wn * 16 + j * 8 + (lane >> 2)];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 2; ++j) dmma_m8n8k4(acc[i][j], a[i], b[j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int m = m0 + wm * 32 + i * 8 + (lane >> 2), n = n0 + wn * 16 + j * 8 + 2 * (lane & 3) + e;
                if (m < op.M && n < op.N) op.store(z, m, n, acc[i][j][e]);
            }
}

// forward: z = image, m = output pixel, n = output channel, k = c*K + tap
struct F64FwdOp {
    static constexpr bool A_K_FAST = false, B_K_FAST = true;
    F64Geom G;
    const double *x, *offset, *mask, *weight, *bias;
    double* out;
    int n_first, M, N;
    __device__ void k_range(int, int* k0, int* k1) const { *k0 = 0; *k1 = G.C * G.kh * G.kw; }
    __device__ double a(int z, int k, int m) const {
        const int K = G.kh * G.kw, c = k / K;
        return f64_sample(G, x, offset, mask, n_first + z, c, k - c * K, m);
    }
    __device__ double b(int, int k, int n) const { return __ldg(weight + static_cast<size_t>(n) * G.C * G.kh * G.kw + k); }
    __device__ void store(int z, int m, int n, double v) const {
        out[(static_cast<size_t>(n_first + z) * G.Cout + n) * M + m] = v + (bias ? __ldg(bias + n) : 0.0);
    }
};

// gcol for images n0 .. n0 + gridDim.z - 1: z = image in the chunk, m = output pixel, n = c*K + tap, k = output channel
struct F64GcolOp {
    static constexpr bool A_K_FAST = false, B_K_FAST = false;
    F64Geom G;
    const double *weight, *grad_out;
    double* gcol;       // [chunk][C*K][Ho*Wo]
    int n_first, M, N;
    __device__ void k_range(int, int* k0, int* k1) const { *k0 = 0; *k1 = G.Cout; }
    __device__ double a(int z, int k, int m) const {
        return __ldg(grad_out + (static_cast<size_t>(n_first + z) * G.Cout + k) * M + m);
    }
    __device__ double b(int, int k, int n) const { return __ldg(weight + static_cast<size_t>(k) * N + n); }
    __device__ void store(int z, int m, int n, double v) const { gcol[(static_cast<size_t>(z) * N + n) * M + m] = v; }
};

// wgrad partials: z = split of the pixels q = n*Ho*Wo + p, m = output channel, n = c*K + tap
struct F64WgradOp {
    static constexpr bool A_K_FAST = true, B_K_FAST = true;
    F64Geom G;
    const double *x, *offset, *mask, *grad_out;
    double* part;       // [splits][Cout][C*K]
    int M, N, q_per_split, Q;
    __device__ void k_range(int z, int* k0, int* k1) const {
        *k0 = z * q_per_split;
        *k1 = min(Q, *k0 + q_per_split);
    }
    __device__ double a(int, int k, int m) const {
        const int HW = G.Ho * G.Wo, n = k / HW;
        return __ldg(grad_out + (static_cast<size_t>(n) * G.Cout + m) * HW + (k - n * HW));
    }
    __device__ double b(int, int k, int nn) const {
        const int HW = G.Ho * G.Wo, n = k / HW, K = G.kh * G.kw, c = nn / K;
        return f64_sample(G, x, offset, mask, n, c, nn - c * K, k - n * HW);
    }
    __device__ void store(int z, int m, int n, double v) const { part[(static_cast<size_t>(z) * M + m) * N + n] = v; }
};

// grad_offset, grad_mask and the grad_x scatter for images n_first .. n_first + n_count - 1.  grad_x must be zeroed.
__global__ void f64_coord_scatter_kernel(const F64Geom G, const double* __restrict__ x, const double* __restrict__ offset,
                                         const double* __restrict__ mask, const double* __restrict__ gcol, int n_first,
                                         int n_count, double* __restrict__ grad_x, double* __restrict__ grad_offset,
                                         double* __restrict__ grad_mask) {
    const int K = G.kh * G.kw, HW = G.Ho * G.Wo, cpg = G.C / G.dg;
    const long long total = static_cast<long long>(n_count) * G.dg * K * HW;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int p = static_cast<int>(i % HW);
        const int k = static_cast<int>((i / HW) % K);
        const int g = static_cast<int>((i / HW / K) % G.dg);
        const int nl = static_cast<int>(i / HW / K / G.dg), n = n_first + nl;
        F64Pos s;
        double goh = 0.0, gow = 0.0, gm = 0.0;
        if (f64_position(G, offset, mask, n, g, k, p, &s)) {
            const F64Corners q = f64_corners(G, s.h, s.w);
            const size_t o = static_cast<size_t>(q.hl) * G.W + q.wl, plane = static_cast<size_t>(G.H) * G.W;
            const double* gc = gcol + (static_cast<size_t>(nl) * G.C * K + static_cast<size_t>(g) * cpg * K + k) * HW + p;
            const size_t xb = (static_cast<size_t>(n) * G.C + static_cast<size_t>(g) * cpg) * plane;
            for (int c = 0; c < cpg; ++c) {
                const double gce = gc[static_cast<size_t>(c) * K * HW];
                const double* xc = x + xb + c * plane;
                double* gxc = grad_x + xb + c * plane;
                const double v1 = (q.t && q.l) ? __ldg(xc + o) : 0.0;
                const double v2 = (q.t && q.r) ? __ldg(xc + o + 1) : 0.0;
                const double v3 = (q.b && q.l) ? __ldg(xc + o + G.W) : 0.0;
                const double v4 = (q.b && q.r) ? __ldg(xc + o + G.W + 1) : 0.0;
                gm += gce * (q.hh * q.hw * v1 + q.hh * q.lw * v2 + q.lh * q.hw * v3 + q.lh * q.lw * v4);
                goh += gce * (q.hw * (v3 - v1) + q.lw * (v4 - v2));
                gow += gce * (q.hh * (v2 - v1) + q.lh * (v4 - v3));
                const double sg = gce * s.mk;
                if (q.t && q.l) atomicAdd(gxc + o, q.hh * q.hw * sg);
                if (q.t && q.r) atomicAdd(gxc + o + 1, q.hh * q.lw * sg);
                if (q.b && q.l) atomicAdd(gxc + o + G.W, q.lh * q.hw * sg);
                if (q.b && q.r) atomicAdd(gxc + o + G.W + 1, q.lh * q.lw * sg);
            }
            goh *= s.mk;
            gow *= s.mk;
        }
        const size_t ob = (static_cast<size_t>(n) * G.dg + g) * 2 * K * HW + p;
        grad_offset[ob + static_cast<size_t>(2 * k) * HW] = goh;
        grad_offset[ob + static_cast<size_t>(2 * k + 1) * HW] = gow;
        if (grad_mask) grad_mask[((static_cast<size_t>(n) * G.dg + g) * K + k) * HW + p] = gm;
    }
}

// grad_weight[i] += scale * (part[0][i] + part[1][i] + ...)
__global__ void f64_wgrad_reduce_kernel(const double* __restrict__ part, int splits, long long n, double scale,
                                        double* __restrict__ grad_weight) {
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        double s = 0.0;
        for (int z = 0; z < splits; ++z) s += part[z * n + i];
        grad_weight[i] += scale * s;
    }
}

// grad_bias[co] += sum_{n,p} gO[n][co][p]; one 256-thread block per channel, fixed partition and reduction tree
__global__ void f64_bias_kernel(const double* __restrict__ go, double* __restrict__ gb, int N, int Cout, int HW) {
    const int co = blockIdx.x;
    double s = 0.0;
    for (int n = 0; n < N; ++n) {
        const double* r = go + (static_cast<size_t>(n) * Cout + co) * HW;
        for (int p = threadIdx.x; p < HW; p += blockDim.x) s += r[p];
    }
    __shared__ double red[256];
    red[threadIdx.x] = s;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) gb[co] += red[0];
}

}  // namespace eb

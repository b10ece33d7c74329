// elementwise.cuh — the HBM-bound stages of the EDVR graph on NHWC fp16 tensors, plus the
// layout converters at the NCHW-fp32 boundary and the weight packer.  Each thread moves
// 16-byte vectors (8 halfs); fp32 math inside.
#pragma once
#include "common.cuh"
#include "epilogue.cuh"

namespace eb {

struct H8 { float v[8]; };
__device__ __forceinline__ H8 h8_load(const __half* p) {
    uint4 u = ldg_nc_v4(p);
    H8 r;
    float2 a = unpack_h2(u.x), b = unpack_h2(u.y), c = unpack_h2(u.z), d = unpack_h2(u.w);
    r.v[0] = a.x; r.v[1] = a.y; r.v[2] = b.x; r.v[3] = b.y; r.v[4] = c.x; r.v[5] = c.y; r.v[6] = d.x; r.v[7] = d.y;
    return r;
}
__device__ __forceinline__ void h8_store(__half* p, const H8& r) {
    *reinterpret_cast<uint4*>(p) = make_uint4(pack_h2(r.v[0], r.v[1]), pack_h2(r.v[2], r.v[3]),
                                              pack_h2(r.v[4], r.v[5]), pack_h2(r.v[6], r.v[7]));
}

// ------------------------------------------------------------------ NCHW fp32 <-> NHWC fp16
// grid: (ceil(HW/32), ceil(C/32), N), block (32, 8)
__global__ void nchw_f32_to_nhwc_f16_kernel(const float* __restrict__ src, __half* __restrict__ dst,
                                            int C, int HW, int dst_pix_stride, int dst_ch_off) {
    __shared__ float tile[32][33];
    const int n = blockIdx.z, p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    for (int i = threadIdx.y; i < 32; i += 8) {
        const int c = c0 + i, p = p0 + threadIdx.x;
        tile[i][threadIdx.x] = (c < C && p < HW) ? src[(static_cast<size_t>(n) * C + c) * HW + p] : 0.f;
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += 8) {
        const int p = p0 + i, c = c0 + threadIdx.x;
        if (p < HW && c < C)
            dst[(static_cast<size_t>(n) * HW + p) * dst_pix_stride + dst_ch_off + c] =
                __float2half_rn(tile[threadIdx.x][i]);
    }
}
// half-precision operator entry (eb_mdcn_forward_f16): the same transpose from an fp16 NCHW tensor, and flat converters
__global__ void nchw_f16_to_nhwc_f16_kernel(const __half* __restrict__ src, __half* __restrict__ dst, int C, int HW) {
    __shared__ __half tile[32][34];
    const int n = blockIdx.z, p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    for (int i = threadIdx.y; i < 32; i += 8) {
        const int c = c0 + i, p = p0 + threadIdx.x;
        tile[i][threadIdx.x] = (c < C && p < HW) ? src[(static_cast<size_t>(n) * C + c) * HW + p] : __float2half(0.f);
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += 8) {
        const int p = p0 + i, c = c0 + threadIdx.x;
        if (p < HW && c < C) dst[(static_cast<size_t>(n) * HW + p) * C + c] = tile[threadIdx.x][i];
    }
}
__global__ void half_to_float_kernel(const __half* __restrict__ src, float* __restrict__ dst, long long n) {
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * blockDim.x)
        dst[i] = __half2float(src[i]);
}
__global__ void float_to_half_kernel(const float* __restrict__ src, __half* __restrict__ dst, long long n) {
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * blockDim.x)
        dst[i] = __float2half_rn(src[i]);
}
__global__ void nhwc_f16_to_nchw_f32_kernel(const __half* __restrict__ src, float* __restrict__ dst,
                                            int C, int HW, int src_pix_stride, int src_ch_off) {
    __shared__ float tile[32][33];
    const int n = blockIdx.z, p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    for (int i = threadIdx.y; i < 32; i += 8) {
        const int p = p0 + i, c = c0 + threadIdx.x;
        tile[i][threadIdx.x] = (p < HW && c < C)
            ? __half2float(src[(static_cast<size_t>(n) * HW + p) * src_pix_stride + src_ch_off + c]) : 0.f;
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += 8) {
        const int c = c0 + i, p = p0 + threadIdx.x;
        if (c < C && p < HW) dst[(static_cast<size_t>(n) * C + c) * HW + p] = tile[threadIdx.x][i];
    }
}

// ------------------------------------------------------------------ weight packer
// out element group (16 B): [nt][chunk][tap][kc][n][0..7]; one thread per group.
__global__ void pack_weight_kernel(const float* __restrict__ w, int cout, int cin, int ktaps, int BN, int n_tiles_n,
                                   __half* __restrict__ out) {
    const int nchunks = cin / 64;
    const long long total = static_cast<long long>(n_tiles_n) * nchunks * ktaps * 8 * BN;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        long long r = i;
        const int n = r % BN; r /= BN;
        const int kc = r % 8; r /= 8;
        const int tap = r % ktaps; r /= ktaps;
        const int chunk = r % nchunks; r /= nchunks;
        const int nt = static_cast<int>(r);
        int srow = nt * BN + n;
        if (srow >= cout) srow = -1;
        H8 v;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int ci = chunk * 64 + kc * 8 + e;
            v.v[e] = srow >= 0 ? w[(static_cast<size_t>(srow) * cin + ci) * ktaps + tap] : 0.f;
        }
        h8_store(out + i * 8, v);
    }
}
// CTA-pair kernel (conv_pair.cuh): [nt][rank 2][chunk of 32 ch][tap][k16 step 2][plane 2][BN/2 rows][8] fp16 - each
// CTA of a pair keeps its half of the output channels resident, K steps in consumption order.
__device__ __forceinline__ void bf8_store(__half* p, const H8& r) {
    *reinterpret_cast<uint4*>(p) = make_uint4(pack_bf2(r.v[0], r.v[1]), pack_bf2(r.v[2], r.v[3]),
                                              pack_bf2(r.v[4], r.v[5]), pack_bf2(r.v[6], r.v[7]));
}
template <bool BF16>
__global__ void pack_weight_pair_kernel(const float* __restrict__ w, int cout, int cin, int ktaps, int BN, int n_tiles_n,
                                        __half* __restrict__ out) {
    const int nchunks = cin / 32, half = BN / 2;
    const long long total = static_cast<long long>(n_tiles_n) * 2 * nchunks * ktaps * 4 * half;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        long long r = i;
        const int row = r % half; r /= half;
        const int plane = r % 2; r /= 2;
        const int h = r % 2; r /= 2;
        const int tap = r % ktaps; r /= ktaps;
        const int chunk = r % nchunks; r /= nchunks;
        const int rank = r % 2; r /= 2;
        const int nt = static_cast<int>(r);
        int srow = nt * BN + rank * half + row;
        if (srow >= cout) srow = -1;
        H8 v;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int ci = chunk * 32 + h * 16 + plane * 8 + e;
            v.v[e] = srow >= 0 ? w[(static_cast<size_t>(srow) * cin + ci) * ktaps + tap] : 0.f;
        }
        if (BF16) bf8_store(out + i * 8, v); else h8_store(out + i * 8, v);
    }
}
// Fused DCN site (dcn_site.cuh): conv_offset weights [dg*27][cin][3][3] -> [chunk of 32 ch][tap][k16 2][plane 2][224 rows][8]
// fp16, rows in TMEM column order r = g*27 + 3*tap + e with e = 0: dh, 1: dw, 2: mask logit; source rows follow the
// reference: offsets g*18 + 2*tap + e, masks dg*18 + g*9 + tap (arch_util.py:244-247, deform_conv_cuda_kernel.cu:600-613).
__device__ __forceinline__ int dcn_site_src_row(int r, int dg) {
    if (r >= dg * 27) return -1;
    const int g = r / 27, rem = r % 27, t = rem / 3, e = rem % 3;
    return e < 2 ? g * 18 + 2 * t + e : dg * 18 + g * 9 + t;
}
__global__ void pack_offset_weight_kernel(const float* __restrict__ w, const float* __restrict__ b, int cin, int dg, int rows,
                                          __half* __restrict__ out, float* __restrict__ b_out) {
    const int nchunks = cin / 32;
    const long long total = static_cast<long long>(nchunks) * 9 * 4 * rows;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        long long r = i;
        const int row = r % rows; r /= rows;
        const int plane = r % 4; r /= 4;              // k16 * 2 + plane-in-k16
        const int tap = r % 9; r /= 9;
        const int chunk = static_cast<int>(r);
        const int srow = dcn_site_src_row(row, dg);
        H8 v;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int ci = chunk * 32 + plane * 8 + e;
            v.v[e] = srow >= 0 ? w[(static_cast<size_t>(srow) * cin + ci) * 9 + tap] : 0.f;
        }
        h8_store(out + i * 8, v);
        if (i < rows) b_out[i] = (b != nullptr && srow >= 0) ? b[srow] : 0.f;      // i == row for chunk 0, tap 0, plane 0
    }
}
// CTA-pair DCN site (dcn_pair.cuh): conv_offset weights -> [half 2][cta 2][chunk of 32 ch][tap][k16 2][plane 2][56 rows][8] fp16.
// Column j of offset half h (TMEM column 256 + 112 h + j) is deformable group h * dg/2 + j / 27, tap (j % 27) / 3, component
// j % 3 (dh, dw, mask logit); CTA k of the pair holds the rows j in [56 k, 56 k + 56) (B operand split along N); columns
// beyond (dg/2) * 27 are zero.  Source rows follow the reference: offsets g*18 + 2*tap + e, masks dg*18 + g*9 + tap
// (arch_util.py:244-247, deform_conv_cuda_kernel.cu:600-613).  b_out[112 h + j] = bias of that column.
__device__ __forceinline__ int dcn_pair_src_row(int h, int j, int dg) {
    const int gph = dg >> 1;
    if (j >= gph * 27) return -1;
    const int g = h * gph + j / 27, rem = j % 27, t = rem / 3, e = rem % 3;
    return e < 2 ? g * 18 + 2 * t + e : dg * 18 + g * 9 + t;
}
__global__ void pack_offset_weight_pair_kernel(const float* __restrict__ w, const float* __restrict__ b, int cin, int dg,
                                               __half* __restrict__ out, float* __restrict__ b_out) {
    const int nchunks = cin / 32;
    const long long total = 4ll * nchunks * 9 * 4 * 56;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        long long r = i;
        const int row = r % 56; r /= 56;
        const int plane = r % 4; r /= 4;              // k16 * 2 + plane-in-k16
        const int tap = r % 9; r /= 9;
        const int chunk = r % nchunks; r /= nchunks;
        const int rank = r % 2; r /= 2;
        const int h = static_cast<int>(r);
        const int srow = dcn_pair_src_row(h, rank * 56 + row, dg);
        H8 v;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int ci = chunk * 32 + plane * 8 + e;
            v.v[e] = srow >= 0 ? w[(static_cast<size_t>(srow) * cin + ci) * 9 + tap] : 0.f;
        }
        h8_store(out + i * 8, v);
        if (i < 224) {
            const int sb = dcn_pair_src_row(static_cast<int>(i) / 112, static_cast<int>(i) % 112, dg);
            b_out[i] = (b != nullptr && sb >= 0) ? b[sb] : 0.f;
        }
    }
}
// Training step, data gradient: dgrad of a stride-1 convolution with weights w[co][ci][tap] is the convolution of grad_out
// with W'[ci][co][taps-1-tap] (transposed, spatially flipped).  This packs W' straight from w in the CTA-pair layout
// ([nt][rank 2][chunk of 32 grad_out channels][tap][k16 2][plane 2][BN/2 rows = input channels][8]); grad_out channels beyond
// `cout` and rows beyond `cin` are zero.
template <bool BF16>
__global__ void pack_weight_pair_dgrad_kernel(const float* __restrict__ w, int cout, int cin, int ktaps, int k_channels,
                                              int BN, int n_tiles_n, __half* __restrict__ out) {
    const int nchunks = k_channels / 32, half = BN / 2;
    const long long total = static_cast<long long>(n_tiles_n) * 2 * nchunks * ktaps * 4 * half;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        long long r = i;
        const int row = r % half; r /= half;
        const int plane = r % 2; r /= 2;
        const int h = r % 2; r /= 2;
        const int tap = r % ktaps; r /= ktaps;
        const int chunk = r % nchunks; r /= nchunks;
        const int rank = r % 2; r /= 2;
        const int nt = static_cast<int>(r);
        const int ci = nt * BN + rank * half + row;                 // output row of the dgrad conv = input channel of w
        H8 v;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int co = chunk * 32 + h * 16 + plane * 8 + e;     // K index of the dgrad conv = output channel of w
            v.v[e] = (ci < cin && co < cout) ? w[(static_cast<size_t>(co) * cin + ci) * ktaps + (ktaps - 1 - tap)] : 0.f;
        }
        if (BF16) bf8_store(out + i * 8, v); else h8_store(out + i * 8, v);
    }
}
__global__ void pack_bias_kernel(const float* __restrict__ b, int cout, int n_packed, float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_packed) return;
    out[i] = (b != nullptr && i < cout) ? b[i] : 0.f;
}

// ------------------------------------------------------------------ conv_first (Cin = 3)
// thread = (4 consecutive pixels of a row, 8 output channels): each weight read from smem feeds 4 FMAs.
// weights staged as ws[k = c*9+dy*3+dx][Cout] so that the 8 channels of a thread are two LDS.128.
__global__ void conv_first_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                  const float* __restrict__ bias, __half* __restrict__ out, int N,
                                  int H, int W, int Cout, int out_pix_stride, int act) {
    extern __shared__ float ws[];   // [27][Cout] + [Cout]
    float* bs = ws + Cout * 27;
    for (int i = threadIdx.x; i < Cout * 27; i += blockDim.x) ws[(i % 27) * Cout + i / 27] = w[i];
    for (int i = threadIdx.x; i < Cout; i += blockDim.x) bs[i] = bias ? bias[i] : 0.f;
    __syncthreads();
    const int groups = Cout / 8, W4 = (W + 3) / 4;
    const long long total = static_cast<long long>(N) * H * W4 * groups;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int g = i % groups;
        const long long q = i / groups;
        const int x0 = (q % W4) * 4, yh = (q / W4) % H, n = q / (static_cast<long long>(W4) * H);
        float in[3][3][6];
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                for (int dx = 0; dx < 6; ++dx) {
                    const int yy = yh + dy - 1, xx = x0 + dx - 1;
                    in[c][dy][dx] = (yy >= 0 && yy < H && xx >= 0 && xx < W)
                        ? __ldg(x + ((static_cast<size_t>(n) * 3 + c) * H + yy) * W + xx) : 0.f;
                }
        float acc[4][8];
#pragma unroll
        for (int p = 0; p < 4; ++p)
#pragma unroll
            for (int e = 0; e < 8; ++e) acc[p][e] = bs[g * 8 + e];
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                for (int dx = 0; dx < 3; ++dx) {
                    const float4 wa = *reinterpret_cast<const float4*>(ws + (c * 9 + dy * 3 + dx) * Cout + g * 8);
                    const float4 wb = *reinterpret_cast<const float4*>(ws + (c * 9 + dy * 3 + dx) * Cout + g * 8 + 4);
                    const float wv[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
#pragma unroll
                    for (int p = 0; p < 4; ++p)
#pragma unroll
                        for (int e = 0; e < 8; ++e) acc[p][e] = fmaf(wv[e], in[c][dy][dx + p], acc[p][e]);
                }
#pragma unroll
        for (int p = 0; p < 4; ++p) {
            if (x0 + p >= W) break;
            H8 r;
#pragma unroll
            for (int e = 0; e < 8; ++e) r.v[e] = apply_act(acc[p][e], act);
            h8_store(out + ((static_cast<size_t>(n) * H + yh) * W + x0 + p) * out_pix_stride + g * 8, r);
        }
    }
}

// ------------------------------------------------------------------ conv_last (Cin -> 3) + base
__device__ __forceinline__ float bilinear_up_sample(const float* __restrict__ im, int h, int w,
                                                    int oy, int ox, int scale) {
    // PyTorch upsample_bilinear2d, align_corners=False (edvr_arch.py:417-418)
    const float rs = 1.0f / static_cast<float>(scale);
    float sy = rs * (oy + 0.5f) - 0.5f, sx = rs * (ox + 0.5f) - 0.5f;
    sy = sy < 0.f ? 0.f : sy;
    sx = sx < 0.f ? 0.f : sx;
    const int y0 = static_cast<int>(sy), x0 = static_cast<int>(sx);
    const int y1 = y0 + (y0 < h - 1 ? 1 : 0), x1 = x0 + (x0 < w - 1 ? 1 : 0);
    const float ly = sy - y0, lx = sx - x0, hy = 1.f - ly, hx = 1.f - lx;
    return hy * (hx * im[y0 * w + x0] + lx * im[y0 * w + x1]) +
           ly * (hx * im[y1 * w + x0] + lx * im[y1 * w + x1]);
}
// thread = 4 consecutive HR pixels of a row x 3 outputs; smem weights ws[dy][c8][dx][e][co] (72 floats per
// (dy, c8)), so each LDS.128 feeds 16 FMAs and each 16-byte input load 36.
__global__ void conv_last_kernel(const __half* __restrict__ x, int x_pix_stride,
                                 const float* __restrict__ w, const float* __restrict__ bias,
                                 const float* __restrict__ base, long long base_img_stride, int scale,
                                 float* __restrict__ out, int N, int H, int W, int Cin) {
    extern __shared__ float ws[];
    const int C8 = Cin / 8;
    for (int i = threadIdx.x; i < 27 * Cin; i += blockDim.x) {
        const int co = i / (Cin * 9), rem = i % (Cin * 9), c = rem / 9, tap = rem % 9;
        const int dy = tap / 3, dx = tap % 3;
        ws[(((dy * C8 + c / 8) * 3 + dx) * 8 + (c & 7)) * 3 + co] = w[i];
    }
    __syncthreads();
    const int W4 = (W + 3) / 4;
    const long long total = static_cast<long long>(N) * H * W4;
    for (long long q = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; q < total;
         q += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int x0 = (q % W4) * 4, yh = (q / W4) % H, n = q / (static_cast<long long>(W4) * H);
        float acc[4][3];
#pragma unroll
        for (int p = 0; p < 4; ++p) { acc[p][0] = bias ? bias[0] : 0.f; acc[p][1] = bias ? bias[1] : 0.f; acc[p][2] = bias ? bias[2] : 0.f; }
        for (int dy = 0; dy < 3; ++dy) {
            const int yy = yh + dy - 1;
            if (yy < 0 || yy >= H) continue;
            const __half* row = x + (static_cast<size_t>(n) * H + yy) * W * x_pix_stride;
            for (int c8 = 0; c8 < C8; ++c8) {
                H8 v[6];
#pragma unroll
                for (int j = 0; j < 6; ++j) {
                    const int xx = x0 + j - 1;
                    if (xx >= 0 && xx < W) v[j] = h8_load(row + static_cast<size_t>(xx) * x_pix_stride + c8 * 8);
                    else {
#pragma unroll
                        for (int e = 0; e < 8; ++e) v[j].v[e] = 0.f;
                    }
                }
                const float4* wq = reinterpret_cast<const float4*>(ws + (dy * C8 + c8) * 72);
                float wl[72];
#pragma unroll
                for (int t = 0; t < 18; ++t) { const float4 f = wq[t]; wl[4 * t] = f.x; wl[4 * t + 1] = f.y; wl[4 * t + 2] = f.z; wl[4 * t + 3] = f.w; }
#pragma unroll
                for (int dx = 0; dx < 3; ++dx)
#pragma unroll
                    for (int e = 0; e < 8; ++e)
#pragma unroll
                        for (int p = 0; p < 4; ++p) {
                            const float iv = v[p + dx].v[e];
                            acc[p][0] = fmaf(iv, wl[(dx * 8 + e) * 3 + 0], acc[p][0]);
                            acc[p][1] = fmaf(iv, wl[(dx * 8 + e) * 3 + 1], acc[p][1]);
                            acc[p][2] = fmaf(iv, wl[(dx * 8 + e) * 3 + 2], acc[p][2]);
                        }
            }
        }
        const size_t plane = static_cast<size_t>(H) * W;
        const int bh = H / scale, bw = W / scale;
        const float* b = base + static_cast<size_t>(n) * base_img_stride;
#pragma unroll
        for (int p = 0; p < 4; ++p) {
            const int xw = x0 + p;
            if (xw >= W) break;
            float* o = out + static_cast<size_t>(n) * 3 * plane + static_cast<size_t>(yh) * W + xw;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float* bc = b + static_cast<size_t>(c) * bh * bw;
                const float bv = scale == 1 ? bc[yh * bw + xw] : bilinear_up_sample(bc, bh, bw, yh, xw, scale);
                o[c * plane] = acc[p][c] + bv;
            }
        }
    }
}

// out[n, c, y, x] += bilinear x`scale` of base[n, c] (scale 4) or base itself (scale 1): the `+ base` of edvr_arch.py:414-419
// when conv_last runs on the tensor cores (its NCHW store leaves conv + bias in `out`)
__global__ void add_base_kernel(const float* __restrict__ base, long long base_img_stride, int scale,
                                float* __restrict__ out, int N, int C, int H, int W) {
    const long long total = static_cast<long long>(N) * C * H * W;
    const int bh = H / scale, bw = W / scale;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int x = i % W, y = (i / W) % H, c = (i / (static_cast<long long>(W) * H)) % C;
        const long long n = i / (static_cast<long long>(W) * H * C);
        const float* bc = base + n * base_img_stride + static_cast<size_t>(c) * bh * bw;
        out[i] += scale == 1 ? bc[y * bw + x] : bilinear_up_sample(bc, bh, bw, y, x, scale);
    }
}

// ------------------------------------------------------------------ frame staging either side of the network (SURVEY §8 f2)
// Decoded frames -> network input: what read_img_seq does after cv2.imread (basicsr/data/data_util.py:28-32, img2tensor
// basicsr/utils/img_util.py:22-27): uint8 [N][H][W][3] BGR -> fp32 [N][3][H][W] RGB (bgr2rgb) = u / 255, a correctly rounded
// fp32 division (the library is built with --use_fast_math: __fdiv_rn keeps the IEEE quotient).  Bit-exact.
__global__ void frames_u8_to_f32_kernel(const uint8_t* __restrict__ src, float* __restrict__ dst, int HW, long long total,
                                        int bgr2rgb) {
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long n = i / HW;
        const int p = static_cast<int>(i - n * HW);
        const uint8_t* s = src + i * 3;
        float* d = dst + n * 3 * HW + p;
        const float c0 = __fdiv_rn(static_cast<float>(s[0]), 255.0f), c1 = __fdiv_rn(static_cast<float>(s[1]), 255.0f),
                    c2 = __fdiv_rn(static_cast<float>(s[2]), 255.0f);
        d[0] = bgr2rgb ? c2 : c0;
        d[HW] = c1;
        d[2 * static_cast<long long>(HW)] = bgr2rgb ? c0 : c2;
    }
}
// Network output -> image bytes: tensor2img with out_type uint8 (basicsr/utils/img_util.py:62-97): clamp to [lo, hi],
// (x - lo) / (hi - lo), CHW -> HWC (RGB -> BGR for 3 channels), round half to even of x * 255 in fp32, uint8.  Bit-exact.
__global__ void tensor2img_u8_kernel(const float* __restrict__ src, uint8_t* __restrict__ dst, int C, int HW, long long total,
                                     int rgb2bgr, float lo, float hi) {
    const float span = __fsub_rn(hi, lo);
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long n = i / HW;
        const int p = static_cast<int>(i - n * HW);
        const float* s = src + n * C * HW + p;
        uint8_t* d = dst + i * C;
        for (int c = 0; c < C; ++c) {
            const float x = s[static_cast<long long>(c) * HW];
            const float v = fminf(fmaxf(x, lo), hi);
            const float q = rintf(__fmul_rn(__fdiv_rn(__fsub_rn(v, lo), span), 255.0f));
            d[(rgb2bgr && C == 3) ? 2 - c : c] = static_cast<uint8_t>(static_cast<int>(q));
        }
    }
}

// ------------------------------------------------------------------ bilinear x2 (align_corners=False)
// out[2k] = .25 in[k-1] + .75 in[k]; out[2k+1] = .75 in[k] + .25 in[k+1]; edges replicate (nn.Upsample(scale_factor=2,
// mode='bilinear', align_corners=False): edvr_arch.py:68,112-115,157).
// One thread = one input pixel x 8 channels -> the 2x2 output pixels it is the "near" neighbour of: nine 16-byte loads (the
// 3x3 neighbourhood, separable weights) for four 16-byte stores, 32-bit index math (image index = blockIdx.y).  The first
// version computed one output per thread with four loads and three 64-bit divisions: 0.86 ms per bench step for 1.3 GB of
// algorithmic traffic (0.2 ms at the HBM roofline).
__global__ void __launch_bounds__(256) upsample2x_kernel(const __half* __restrict__ src, int sps, int sco,
                                                         __half* __restrict__ dst, int dps, int dco, int H, int W, int C,
                                                         float mul, const __half* __restrict__ add, int aps, int aco) {
    const int groups = C >> 3, W2 = 2 * W;
    const int per_img = H * W * groups;
    const int n = blockIdx.y;
    const __half* s = src + static_cast<size_t>(n) * H * W * sps + sco;
    __half* d = dst + static_cast<size_t>(n) * 4 * H * W * dps + dco;
    const __half* a = add ? add + static_cast<size_t>(n) * 4 * H * W * aps + aco : nullptr;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < per_img; i += gridDim.x * blockDim.x) {
        const int g = i % groups, pix = i / groups;
        const int ix = pix % W, iy = pix / W;
        const int xm = max(ix - 1, 0), xp = min(ix + 1, W - 1), ym = max(iy - 1, 0), yp = min(iy + 1, H - 1);
        // horizontal pass on the three rows: l = output column 2 ix, r = output column 2 ix + 1
        H8 l[3], r[3];
        const int ys[3] = {ym, iy, yp};
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const __half* row = s + static_cast<size_t>(ys[j]) * W * sps + g * 8;
            const H8 vm = h8_load(row + static_cast<size_t>(xm) * sps), vc = h8_load(row + static_cast<size_t>(ix) * sps),
                     vp = h8_load(row + static_cast<size_t>(xp) * sps);
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                l[j].v[e] = 0.25f * vm.v[e] + 0.75f * vc.v[e];
                r[j].v[e] = 0.75f * vc.v[e] + 0.25f * vp.v[e];
            }
        }
        // vertical pass: output rows 2 iy (rows ym, iy) and 2 iy + 1 (rows iy, yp)
#pragma unroll
        for (int oy = 0; oy < 2; ++oy)
#pragma unroll
            for (int ox = 0; ox < 2; ++ox) {
                const H8& far_ = ox ? r[oy ? 2 : 0] : l[oy ? 2 : 0];
                const H8& near_ = ox ? r[1] : l[1];
                const size_t opix = static_cast<size_t>(2 * iy + oy) * W2 + 2 * ix + ox;
                H8 o;
#pragma unroll
                for (int e = 0; e < 8; ++e) o.v[e] = (0.25f * far_.v[e] + 0.75f * near_.v[e]) * mul;
                if (a != nullptr) {
                    const H8 av = h8_load(a + opix * aps + g * 8);
#pragma unroll
                    for (int e = 0; e < 8; ++e) o.v[e] += av.v[e];
                }
                h8_store(d + opix * dps + g * 8, o);
            }
    }
}

// ------------------------------------------------------------------ max + avg pool 3x3 s2 p1
__global__ void pool_max_avg_kernel(const __half* __restrict__ src, int sps, int sco,
                                    __half* __restrict__ dst, int dps, int dco, int N, int H, int W, int C) {
    const int groups = C / 8, Ho = (H + 1) / 2, Wo = (W + 1) / 2;   // floor((H+2-3)/2)+1
    const long long total = static_cast<long long>(N) * Ho * Wo * groups;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int g = i % groups;
        const long long opix = i / groups;
        const int ox = opix % Wo, oy = (opix / Wo) % Ho, n = opix / (static_cast<long long>(Wo) * Ho);
        H8 mx, sm;
#pragma unroll
        for (int e = 0; e < 8; ++e) { mx.v[e] = -INFINITY; sm.v[e] = 0.f; }
        for (int dy = 0; dy < 3; ++dy)
            for (int dx = 0; dx < 3; ++dx) {
                const int yy = 2 * oy + dy - 1, xx = 2 * ox + dx - 1;
                if (yy < 0 || yy >= H || xx < 0 || xx >= W) continue;
                const H8 v = h8_load(src + ((static_cast<size_t>(n) * H + yy) * W + xx) * sps + sco + g * 8);
#pragma unroll
                for (int e = 0; e < 8; ++e) { mx.v[e] = fmaxf(mx.v[e], v.v[e]); sm.v[e] += v.v[e]; }
            }
#pragma unroll
        for (int e = 0; e < 8; ++e) sm.v[e] *= (1.0f / 9.0f);     // count_include_pad=True
        h8_store(dst + opix * dps + dco + g * 8, mx);
        h8_store(dst + opix * dps + dco + C + g * 8, sm);
    }
}

// ------------------------------------------------------------------ TSA temporal attention
// LPP = C/8 lanes cooperate on one pixel.
__global__ void tsa_temporal_kernel(const __half* __restrict__ emb, const __half* __restrict__ emb_ref,
                                    const __half* __restrict__ aligned, __half* __restrict__ dst,
                                    int B, int T, int HW, int C) {
    const int lpp = C / 8;
    const int sub = threadIdx.x % lpp;
    const long long npix = static_cast<long long>(B) * HW;
    const long long gstride = static_cast<long long>(gridDim.x) * blockDim.x / lpp;
    // all lanes of a warp iterate the same number of times (shuffles need full participation)
    const long long first = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) / lpp;
    const long long iters = (npix + gstride - 1) / gstride;
    for (long long it = 0; it < iters; ++it) {
        const long long pix = first + it * gstride;
        const bool ok = pix < npix;
        const long long b = ok ? pix / HW : 0, hw = ok ? pix % HW : 0;
        H8 r8 = h8_load(emb_ref + (b * HW + hw) * C + sub * 8);
        for (int t = 0; t < T; ++t) {
            const size_t fp = ((b * T + t) * static_cast<size_t>(HW) + hw) * C + sub * 8;
            const H8 e8 = h8_load(emb + fp);
            float d = 0.f;
#pragma unroll
            for (int e = 0; e < 8; ++e) d = fmaf(e8.v[e], r8.v[e], d);
            for (int o = lpp >> 1; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
            const float prob = 1.0f / (1.0f + __expf(-d));
            H8 a8 = h8_load(aligned + fp);
#pragma unroll
            for (int e = 0; e < 8; ++e) a8.v[e] *= prob;
            if (ok) h8_store(dst + (b * HW + hw) * (static_cast<size_t>(T) * C) + t * C + sub * 8, a8);
        }
    }
}

// ------------------------------------------------------------------ TSA output modulation
__global__ void tsa_modulate_kernel(const __half* __restrict__ feat, int fps, int fco,
                                    const __half* __restrict__ attn, const __half* __restrict__ attn_add,
                                    __half* __restrict__ out16, float* __restrict__ out32,
                                    long long npix, int C, int H, int W, int f32_blocked) {
    const int groups = C / 8;
    const long long total = npix * groups;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int g = i % groups;
        const long long pix = i / groups;
        const H8 f = h8_load(feat + pix * fps + fco + g * 8);
        const H8 a = h8_load(attn + pix * C + g * 8);
        const H8 d = h8_load(attn_add + pix * C + g * 8);
        H8 r;
#pragma unroll
        for (int e = 0; e < 8; ++e) r.v[e] = f.v[e] * (1.0f / (1.0f + __expf(-a.v[e]))) * 2.f + d.v[e];
        if (out16) h8_store(out16 + pix * C + g * 8, r);
        if (out32) {
            if (f32_blocked) {
                const int x = pix % W, y = (pix / W) % H, img = pix / (static_cast<long long>(W) * H);
                float* o = out32 + blocked32_block(img, y, x, g >> 2, H, W, C) + ((g & 3) * 2) * 128;
                *reinterpret_cast<float4*>(o) = make_float4(r.v[0], r.v[1], r.v[2], r.v[3]);
                *reinterpret_cast<float4*>(o + 128) = make_float4(r.v[4], r.v[5], r.v[6], r.v[7]);
            } else {
                float4* o = reinterpret_cast<float4*>(out32 + pix * C + g * 8);
                o[0] = make_float4(r.v[0], r.v[1], r.v[2], r.v[3]);
                o[1] = make_float4(r.v[4], r.v[5], r.v[6], r.v[7]);
            }
        }
    }
}

__global__ void add_kernel(const __half* __restrict__ a, int aps, int aco, const __half* __restrict__ b,
                           int bps, int bco, __half* __restrict__ dst, int dps, int dco, long long npix, int C) {
    const int groups = C / 8;
    const long long total = npix * groups;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int g = i % groups;
        const long long pix = i / groups;
        H8 x = h8_load(a + pix * aps + aco + g * 8);
        const H8 y = h8_load(b + pix * bps + bco + g * 8);
#pragma unroll
        for (int e = 0; e < 8; ++e) x.v[e] += y.v[e];
        h8_store(dst + pix * dps + dco + g * 8, x);
    }
}

}  // namespace eb

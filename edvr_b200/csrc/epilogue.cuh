// epilogue.cuh — shared accumulator epilogue: TMEM row (one output pixel, 32 channels at a
// time) -> bias -> activation -> residual -> NHWC fp16 / NHWC fp32 / NCHW fp32 stores,
// optionally through the PixelShuffle(2) index map or a stride-2 subsample.
#pragma once
#include "common.cuh"

namespace eb {

enum : int { OUT_SAME = 0, OUT_PIXSHUF2 = 1, OUT_STRIDE2 = 2 };

// Epilogue kinds.  Kernels are instantiated per kind so that each role's loop stays inside the instruction cache
// (a single do-everything epilogue made the conv kernels 40-77 KB of SASS; profiles/r01_ncu_conv2_icache.txt).
enum : int { EK_PLAIN = 0,    // fp16 NHWC out (+ optional fp16 residual)
             EK_F32 = 1,      // fp32 residual stream in/out (+ optional fp16 copy): trunk blocks
             EK_PIXSHUF = 3,  // PixelShuffle(2) store
             EK_STRIDE2 = 4,  // even-pixel store
             EK_NCHW = 5,     // fp32 NCHW out (reference operator layout)
             EK_GENERIC = 6 };// any combination, resolved at run time

struct EpiParams {
    const float* bias;        // [cout_packed] or nullptr
    int act;                  // ACT_*
    int H, W;                 // spatial dims of the accumulator grid
    // residual, added AFTER the activation (ResidualBlockNoBN: act = none)
    const __half* res16;
    const float* res32;
    int res_pix_stride, res_ch_off;
    // outputs (any subset)
    __half* out16;
    int out16_pix_stride, out16_ch_off;
    float* out32;
    int out32_pix_stride, out32_ch_off;
    float* out_nchw;          // [N][nchw_C][H][W] fp32 (reference op layout)
    int nchw_C;
    int out_mode;             // OUT_*
    int f32_blocked;          // res32 / out32 in the tile-blocked layout (blocked32_offset)
    int res16_wide;           // res16 view is 32-byte aligned per 16 channels: 2 x LDG.256 instead of 4 x LDG.128
    int bf16;                 // operands and the 16-bit output are bf16 (training step); CTA-pair kernel, plain TMA store only
};

// Tile-blocked fp32 layout: float index of (pixel (img,y,x), channel c) for an [N,H,W,C] tensor, C % 32 == 0.
// Block = (16x16 tile, 16x8 half `sub`, 32-pixel quarter q, 32-channel chunk): [8 float4 slots][32 pixels][4 floats].
__host__ __device__ __forceinline__ long long blocked32_block(int img, int y, int x, int chunk, int H, int W, int C) {
    const int tiles_x = (W + 15) >> 4, tiles_y = (H + 15) >> 4;
    const long long tile = (static_cast<long long>(img) * tiles_y + (y >> 4)) * tiles_x + (x >> 4);
    const int sub = (x >> 3) & 1, m = ((y & 15) << 3) | (x & 7);
    return (((tile * 2 + sub) * 4 + (m >> 5)) * (C >> 5) + chunk) * 1024 + (m & 31) * 4;
}

// v: 32 consecutive accumulator channels [c0, c0+32) of output pixel (img, y, x); `valid` masks the memory traffic.
// EXT16: the caller stores the fp16 NHWC copy itself (TMA store in conv_pair.cuh); v[] holds the final values on return.
// Residual prefetch for the blocked fp32 stream (trunk blocks): the eight float4 slots epi_store32 would read for channels
// [c0, c0+32) of pixel (img, y, x), issued early so that their DRAM latency overlaps the wait for the accumulator and the
// previous chunk's stores (the trunk's conv2 launches were epilogue-latency bound: tensor pipe 39 % busy, DRAM 49 %).
__device__ __forceinline__ void epi_prefetch_res32_blocked(const EpiParams& p, int img, int y, int x, int c0, bool valid,
                                                           float4 (&r)[8]) {
    if (!valid) return;
    const float4* src = reinterpret_cast<const float4*>(
        p.res32 + blocked32_block(img, y, x, (p.res_ch_off + c0) >> 5, p.H, p.W, p.res_pix_stride));
#pragma unroll
    for (int q = 0; q < 8; ++q) r[q] = __ldg(src + q * 32);
}

// Same for the fp16 residual of a ResidualBlockNoBN whose stream is fp16 (feature extraction, predeblur): the 64 bytes of
// pixel (img, y, x), channels [c0, c0+32), land in r[0..3].
__device__ __forceinline__ void epi_prefetch_res16(const EpiParams& p, int img, int y, int x, int c0, bool valid, float4 (&r)[8]) {
    if (!valid) return;
    const size_t pix = (static_cast<size_t>(img) * p.H + y) * p.W + x;
    const __half* src = p.res16 + pix * p.res_pix_stride + p.res_ch_off + c0;
    uint4 u[4];
    if (p.res16_wide) {
        ldg_nc_v8(src, u[0], u[1]);
        ldg_nc_v8(src + 16, u[2], u[3]);
    } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) u[q] = ldg_nc_v4(src + q * 8);
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) r[q] = *reinterpret_cast<const float4*>(&u[q]);
}

template <int EK = EK_GENERIC, bool EXT16 = false>
__device__ __forceinline__ void epi_store32(const EpiParams& p, const float* __restrict__ bias_s,
                                            float (&v)[32], int img, int y, int x, int c0,
                                            bool valid, const float4* res_pre = nullptr) {
    if (bias_s != nullptr) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] += bias_s[c0 + j];
    }
    constexpr bool G = EK == EK_GENERIC;
    act_inplace<32>(v, p.act);
    if (!valid) return;

    const size_t pix = (static_cast<size_t>(img) * p.H + y) * p.W + x;
    if ((G || EK == EK_PLAIN) && p.res16 != nullptr) {
        const __half* r = p.res16 + pix * p.res_pix_stride + p.res_ch_off + c0;
        uint4 ru[4];
        if (EK == EK_PLAIN && res_pre != nullptr) {
#pragma unroll
            for (int q = 0; q < 4; ++q) ru[q] = *reinterpret_cast<const uint4*>(&res_pre[q]);
        } else if (p.res16_wide) {     // lanes read different pixels: a 32-byte load halves the L1 wavefronts per byte
            ldg_nc_v8(r, ru[0], ru[1]);
            ldg_nc_v8(r + 16, ru[2], ru[3]);
        } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) ru[q] = ldg_nc_v4(r + q * 8);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const uint4 u = ru[q];
            float2 f0 = unpack_h2(u.x), f1 = unpack_h2(u.y), f2 = unpack_h2(u.z), f3 = unpack_h2(u.w);
            v[q * 8 + 0] += f0.x; v[q * 8 + 1] += f0.y; v[q * 8 + 2] += f1.x; v[q * 8 + 3] += f1.y;
            v[q * 8 + 4] += f2.x; v[q * 8 + 5] += f2.y; v[q * 8 + 6] += f3.x; v[q * 8 + 7] += f3.y;
        }
    }
    // blocked fp32 stream: this thread's 32 channels are 8 float4 slots, 512 B apart, lanes 16 B apart
    const long long blk = ((G || EK == EK_F32) && p.f32_blocked)
        ? blocked32_block(img, y, x, (p.res_ch_off + c0) >> 5, p.H, p.W, p.res_pix_stride) : 0;
    if (EK == EK_F32 && res_pre != nullptr) {
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const float4 f = res_pre[q];
            v[q * 4 + 0] += f.x; v[q * 4 + 1] += f.y; v[q * 4 + 2] += f.z; v[q * 4 + 3] += f.w;
        }
    } else if ((G || EK == EK_F32) && p.res32 != nullptr) {
        const float4* r = p.f32_blocked ? reinterpret_cast<const float4*>(p.res32 + blk)
                                        : reinterpret_cast<const float4*>(p.res32 + pix * p.res_pix_stride + p.res_ch_off + c0);
        const int rs = p.f32_blocked ? 32 : 1;          // float4 stride between consecutive 4-channel slots
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            float4 f = __ldg(r + q * rs);
            v[q * 4 + 0] += f.x; v[q * 4 + 1] += f.y; v[q * 4 + 2] += f.z; v[q * 4 + 3] += f.w;
        }
    }

    if ((G && p.out_mode == OUT_SAME) || EK == EK_PLAIN || EK == EK_F32 || EK == EK_NCHW) {
        if (!EXT16 && EK != EK_NCHW && p.out16 != nullptr) {
            uint4* o = reinterpret_cast<uint4*>(p.out16 + pix * p.out16_pix_stride + p.out16_ch_off + c0);
#pragma unroll
            for (int q = 0; q < 4; ++q)
                o[q] = make_uint4(pack_h2(v[q * 8 + 0], v[q * 8 + 1]), pack_h2(v[q * 8 + 2], v[q * 8 + 3]),
                                  pack_h2(v[q * 8 + 4], v[q * 8 + 5]), pack_h2(v[q * 8 + 6], v[q * 8 + 7]));
        }
        if ((G || EK == EK_F32) && p.out32 != nullptr) {
            const long long blko = p.f32_blocked ? blocked32_block(img, y, x, (p.out32_ch_off + c0) >> 5, p.H, p.W, p.out32_pix_stride) : 0;
            float4* o = p.f32_blocked ? reinterpret_cast<float4*>(p.out32 + blko)
                                      : reinterpret_cast<float4*>(p.out32 + pix * p.out32_pix_stride + p.out32_ch_off + c0);
            const int os = p.f32_blocked ? 32 : 1;
#pragma unroll
            for (int q = 0; q < 8; ++q)
                o[q * os] = make_float4(v[q * 4 + 0], v[q * 4 + 1], v[q * 4 + 2], v[q * 4 + 3]);
        }
        if ((G || EK == EK_NCHW) && p.out_nchw != nullptr) {
            const size_t plane = static_cast<size_t>(p.H) * p.W;
            float* o = p.out_nchw + (static_cast<size_t>(img) * p.nchw_C + c0) * plane +
                       static_cast<size_t>(y) * p.W + x;
#pragma unroll
            for (int j = 0; j < 32; ++j)
                if (c0 + j < p.nchw_C) o[j * plane] = v[j];
        }
    } else if ((G && p.out_mode == OUT_PIXSHUF2) || EK == EK_PIXSHUF) {
        // nn.PixelShuffle(2): out[b, c, 2y+i, 2x+j] = in[b, 4c + 2i + j, y, x]
        // (/root/reference/basicsr/models/archs/edvr_arch.py:351,410-411)
        if (EXT16) return;      // conv_pair.cuh stages the four output pixels and stores them with one TMA box
        const int H2 = 2 * p.H, W2 = 2 * p.W;
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const size_t opix = (static_cast<size_t>(img) * H2 + 2 * y + i) * W2 + 2 * x + j;
                uint4* o = reinterpret_cast<uint4*>(p.out16 + opix * p.out16_pix_stride +
                                                    p.out16_ch_off + (c0 >> 2));
                const int s = 2 * i + j;
                *o = make_uint4(pack_h2(v[s], v[4 + s]), pack_h2(v[8 + s], v[12 + s]),
                                pack_h2(v[16 + s], v[20 + s]), pack_h2(v[24 + s], v[28 + s]));
            }
    } else {  // OUT_STRIDE2: stride-2 / pad-1 / k=3 conv == stride-1 result sampled at even pixels
        if ((y | x) & 1) return;
        const int Ho = (p.H + 1) >> 1, Wo = (p.W + 1) >> 1;
        const size_t opix = (static_cast<size_t>(img) * Ho + (y >> 1)) * Wo + (x >> 1);
        uint4* o = reinterpret_cast<uint4*>(p.out16 + opix * p.out16_pix_stride + p.out16_ch_off + c0);
#pragma unroll
        for (int q = 0; q < 4; ++q)
            o[q] = make_uint4(pack_h2(v[q * 8 + 0], v[q * 8 + 1]), pack_h2(v[q * 8 + 2], v[q * 8 + 3]),
                              pack_h2(v[q * 8 + 4], v[q * 8 + 5]), pack_h2(v[q * 8 + 6], v[q * 8 + 7]));
    }
}

}  // namespace eb

// conv_igemm2.cuh — second-generation dense conv (3x3 pad 1 / 1x1) for Cout tiles of exactly 128:
// the GEMM is transposed with respect to conv_igemm.cuh:  D[Cout=128][pixels=256] = W · X^T.
//
//   * M = 128 output channels (TMEM lanes), N = 256 pixels per MMA (a 32-row x 8-pixel image tile), K = 16.
//     One tcgen05.mma now reads 4 KB of weights + 8 KB of pixels per 128 cycles (96 B/cycle of shared-memory
//     bandwidth instead of the 128 B/cycle an M128 x N128 pair of MMAs needs), and half as many instructions.
//   * The pixel operand is the same halo-tile trick: one (32+2)x(8+2) halo of a 64-channel chunk is loaded once,
//     every 3x3 tap is a start-address offset into it (rows of the canonical no-swizzle layout = pixels).
//   * The accumulator is channel-major: an epilogue thread owns ONE output channel (its TMEM lane) for 32 pixels
//     at a time, so a warp touches 32 consecutive channels of one pixel per instruction (one L1 wavefront) and
//     bias / activation / residual / NHWC stores go straight from registers to global memory.  PixelShuffle /
//     stride-2 / DCN-record variants included.
// Same warp roles, mbarrier rings, bulk-copied pre-packed weights and persistent scheduling as conv_igemm.cuh.
#pragma once
#include "common.cuh"
#include "epilogue.cuh"
#include "conv_igemm.cuh"

namespace eb {

constexpr int C2_TH = 32, C2_TW = 8;                   // pixel tile: 32 rows x 8 columns = 256 = MMA N
constexpr int C2_A_BUFS = 2;
constexpr int C2_W_STAGES = 6;
constexpr int C2_PLANE_BYTES = 341 * 16;               // >= 34*10*16, odd number of 16-byte units
constexpr int C2_A_BUF_BYTES = 8 * C2_PLANE_BYTES;     // 43648
constexpr int C2_W_STAGE_BYTES = 128 * 128;            // 128 channels x 64 k x 2 B
constexpr int C2_THREADS = 320;
constexpr int C2_SMEM_BYTES = C2_A_BUFS * C2_A_BUF_BYTES + C2_W_STAGES * C2_W_STAGE_BYTES + 256;

template <int HALO>
__device__ __forceinline__ void conv2_load_halo(const ConvParams& P, int chunk, int img, int ty, int tx,
                                                uint32_t abuf_saddr, int tid) {
    constexpr int RPX = C2_TW + 2 * HALO;               // row pitch in pixels
    constexpr int NPIX = (C2_TH + 2 * HALO) * RPX;
    constexpr int NITEM = NPIX * 8;
    constexpr int U = 8;
    int s = 0, ch = chunk * 64;
    if (P.nsrc > 1 && ch >= P.src[0].C) { s = 1; ch -= P.src[0].C; }
    const ConvSrc& S = P.src[s];
    const bool img_ok = img < P.N;                      // ghost tiles (odd tail) read nothing
    const int simg = img_ok ? (img / S.div) * S.mul + (img % S.div) * S.keep + S.add : 0;
    const __half* base = S.ptr + S.ch_off + ch;
    const int y0 = ty * C2_TH - HALO, x0 = tx * C2_TW - HALO;
    for (int b = 0; b < NITEM; b += 128 * U) {
        uint4 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int idx = b + u * 128 + tid;
            v[u] = make_uint4(0, 0, 0, 0);
            if (idx < NITEM) {
                const int p = idx >> 3, kc = idx & 7;
                const int y = p / RPX, x = p - y * RPX;
                const int gy = y0 + y, gx = x0 + x;
                if (img_ok && gy >= 0 && gy < P.H && gx >= 0 && gx < P.W)
                    v[u] = ldg_nc_v4(base + ((static_cast<size_t>(simg) * P.H + gy) * P.W + gx) * S.pix_stride + kc * 8);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int idx = b + u * 128 + tid;
            if (idx < NITEM) sts_v4(abuf_saddr + (idx & 7) * C2_PLANE_BYTES + (idx >> 3) * 16, v[u]);
        }
    }
}

// v[i] with a runtime index, as a select tree (edge tiles only; avoids spilling the register tile to local memory)
__device__ __forceinline__ float sel32(const float (&v)[32], int i) {
    float r = v[0];
#pragma unroll
    for (int k = 1; k < 32; ++k) r = (i == k) ? v[k] : r;
    return r;
}

// cycle-counter slots of ConvParams.stats (per CTA): who waited on what
enum : int { ST_MMA_TOTAL = 0, ST_MMA_WAIT_ACC = 1, ST_MMA_WAIT_A = 2, ST_MMA_WAIT_W = 3, ST_A_TOTAL = 4,
             ST_A_WAIT_EMPTY = 5, ST_W_TOTAL = 6, ST_W_WAIT_EMPTY = 7, ST_E_TOTAL = 8, ST_E_WAIT_ACC = 9, ST_TILES = 10, ST_E_TMEM = 11, ST_E_P1 = 12, ST_E_BAR = 13, ST_E_P2 = 14 };

#define C2_TIMED_WAIT_(WAITFN, bar, parity, slot)                                  \
    do {                                                                   \
        if (STATS) {                                                       \
            const long long t_ = clock64();                                \
            WAITFN(bar, parity);                                           \
            st_acc[slot] += static_cast<unsigned long long>(clock64() - t_); \
        } else {                                                           \
            WAITFN(bar, parity);                                           \
        }                                                                  \
    } while (0)
#define C2_TIMED_WAIT(bar, parity, slot) C2_TIMED_WAIT_(mbar_wait_t<0>, bar, parity, slot)
#define C2_TIMED_WAIT_WARP(bar, parity, slot) C2_TIMED_WAIT_(mbar_wait_warp, bar, parity, slot)

// PS: pixel stride (elements) of the output / residual tensors when it is a compile-time constant (0 = runtime).
// With a constant stride the 8 pixels of a tile row are addressed as [row pointer + immediate]; with a runtime
// stride the compiler recomputes one address register pair per access and consecutive stores serialise on it.
template <int HALO, int EK, bool STATS, int PS>
__global__ void __launch_bounds__(C2_THREADS, 1) conv_igemm2_kernel(const ConvParams P) {
    unsigned long long st_acc[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    const long long st_t0 = STATS ? clock64() : 0;
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* a_smem = smem;                                         // pixel halo chunks
    uint8_t* w_smem = smem + C2_A_BUFS * C2_A_BUF_BYTES;            // weight stages
    uint64_t* bars = reinterpret_cast<uint64_t*>(w_smem + C2_W_STAGES * C2_W_STAGE_BYTES);
    uint64_t* a_full = bars;                          // [2]
    uint64_t* a_empty = bars + 2;                     // [2]
    uint64_t* w_full = bars + 4;                      // [6]
    uint64_t* w_empty = bars + 4 + C2_W_STAGES;       // [6]
    uint64_t* acc_full = bars + 4 + 2 * C2_W_STAGES;  // [2]
    uint64_t* acc_empty = acc_full + 2;               // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int RPX = C2_TW + 2 * HALO;
    const int tiles_x = (P.W + C2_TW - 1) / C2_TW;
    const int tiles_y = (P.H + C2_TH - 1) / C2_TH;
    const int total_tiles = P.N * tiles_y * tiles_x * P.n_tiles_n;
    const int cin = P.src[0].C + (P.nsrc > 1 ? P.src[1].C : 0);
    const int nchunks = cin / 64;
    const bool has_bias = P.epi.bias != nullptr;

    if (threadIdx.x == 0) {
        for (int i = 0; i < C2_A_BUFS; ++i) { mbar_init(&a_full[i], 4); mbar_init(&a_empty[i], 1); }
        for (int i = 0; i < C2_W_STAGES; ++i) { mbar_init(&w_full[i], 1); mbar_init(&w_empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 4); }
        fence_barrier_init();
    }
    if (warp == 0) tmem_alloc(tmem_slot, 512);
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ================= weight producer
        if (lane == 0) {
            uint32_t it = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const int nt = tile % P.n_tiles_n;
                const uint8_t* w = reinterpret_cast<const uint8_t*>(P.wpack) +
                                   static_cast<size_t>(nt) * nchunks * P.taps * C2_W_STAGE_BYTES;
                for (int st = 0; st < nchunks * P.taps; ++st, ++it) {
                    const uint32_t s = it % C2_W_STAGES, ph = (it / C2_W_STAGES) & 1u;
                    C2_TIMED_WAIT(&w_empty[s], ph ^ 1u, ST_W_WAIT_EMPTY);
                    mbar_arrive_expect_tx(&w_full[s], C2_W_STAGE_BYTES);
                    bulk_g2s(w_smem + s * C2_W_STAGE_BYTES, w + static_cast<size_t>(st) * C2_W_STAGE_BYTES,
                             C2_W_STAGE_BYTES, &w_full[s]);
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer: D[128 ch][256 px] += W[128 x 16] . X[256 x 16]^T
        if (lane == 0) {
            const uint32_t idesc = umma_idesc_f16(128, 256);
            uint32_t a_it = 0, w_it = 0, acc_it = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++acc_it) {
                const uint32_t ab = acc_it & 1u;
                C2_TIMED_WAIT(&acc_empty[ab], ((acc_it >> 1) & 1u) ^ 1u, ST_MMA_WAIT_ACC);
                tc_fence_after_sync();
                const uint32_t d = tmem_base + ab * 256u;
                for (int c = 0; c < nchunks; ++c, ++a_it) {
                    const uint32_t as = a_it % C2_A_BUFS, aph = (a_it / C2_A_BUFS) & 1u;
                    C2_TIMED_WAIT(&a_full[as], aph, ST_MMA_WAIT_A);
                    tc_fence_after_sync();
                    const uint32_t x_base = smem_u32(a_smem + as * C2_A_BUF_BYTES);
                    for (int t = 0; t < P.taps; ++t, ++w_it) {
                        const uint32_t ws = w_it % C2_W_STAGES, wph = (w_it / C2_W_STAGES) & 1u;
                        C2_TIMED_WAIT(&w_full[ws], wph, ST_MMA_WAIT_W);
                        tc_fence_after_sync();
                        const uint32_t w_base = smem_u32(w_smem + ws * C2_W_STAGE_BYTES);
                        const int ki = HALO ? t / 3 : 0, kj = HALO ? t % 3 : 0;
                        const uint32_t x_tap = x_base + (ki * RPX + kj) * 16;
#pragma unroll
                        for (int k16 = 0; k16 < 4; ++k16) {
                            const uint64_t wd = umma_desc_nosw(w_base + k16 * 2 * 2048, 2048, 128);
                            const uint64_t xd = umma_desc_nosw(x_tap + k16 * 2 * C2_PLANE_BYTES, C2_PLANE_BYTES, RPX * 16);
                            umma_f16(d, wd, xd, idesc, (c | t | k16) != 0 ? 1u : 0u);
                        }
                        umma_commit(&w_empty[ws]);
                    }
                    umma_commit(&a_empty[as]);
                }
                umma_commit(&acc_full[ab]);
            }
        }
    } else if (warp < 6) {
        // ================= pixel (halo) producers
        const int tid = threadIdx.x - 64;
        uint32_t a_it = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            const int pt = tile / P.n_tiles_n;
            const int tx = pt % tiles_x, ty = (pt / tiles_x) % tiles_y, img = pt / (tiles_x * tiles_y);
            for (int c = 0; c < nchunks; ++c, ++a_it) {
                const uint32_t as = a_it % C2_A_BUFS, aph = (a_it / C2_A_BUFS) & 1u;
                C2_TIMED_WAIT_WARP(&a_empty[as], aph ^ 1u, ST_A_WAIT_EMPTY);
                conv2_load_halo<HALO>(P, c, img, ty, tx, smem_u32(a_smem + as * C2_A_BUF_BYTES), tid);
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&a_full[as]);
            }
        }
    } else {
        // ================= epilogue: 4 warps, warp q owns TMEM lanes (= channels) 32q..32q+31.
        // A thread keeps ONE channel `co` for 32 pixels at a time; a warp therefore touches 32 consecutive channels
        // of one pixel per instruction = 64 (fp16) / 128 (fp32) contiguous bytes = ONE L1 wavefront, and nothing goes
        // through shared memory (its port is already saturated by the MMA operands).  Every parameter is hoisted
        // into registers and the code is specialised per epilogue kind (EK): with one epilogue warp per scheduler,
        // constant-bank loads, 64-bit multiplies and instruction-cache misses inside the loop are exposed latency.
        const int q = warp & 3;
        const EpiParams E = P.epi;
        const int H = P.H, W = P.W, NIMG = P.N, dbg = STATS ? P.dbg : 0;
        const long long ps16 = PS ? PS : E.out16_pix_stride, ps32 = PS ? PS : E.out32_pix_stride,
                        psr = PS ? PS : E.res_pix_stride;
        uint32_t acc_it = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++acc_it) {
            const int nt = tile % P.n_tiles_n, pt = tile / P.n_tiles_n;
            const int tx = pt % tiles_x, ty = (pt / tiles_x) % tiles_y, img = pt / (tiles_x * tiles_y);
            const uint32_t ab = acc_it & 1u;
            const int co = nt * 128 + 32 * q + lane;
            const float bias_c = has_bias ? __ldg(E.bias + co) : 0.f;
            const int x0 = tx * C2_TW, y0 = ty * C2_TH;
            const int xn = min(C2_TW, W - x0);                               // valid columns (warp-uniform)
            const bool img_ok = (img < NIMG) && !(dbg & 1);
            const bool interior = (xn == C2_TW) && (y0 + C2_TH <= H);
            const long long pix0 = (static_cast<long long>(img) * H + y0) * W + x0;
            __half* o16 = nullptr;
            float* o32 = nullptr;
            const __half* r16 = nullptr;
            const float* r32 = nullptr;
            long long ops16 = ps16, orow16 = static_cast<long long>(W) * ps16;   // element strides of the fp16 output
            if (EK == EK_PLAIN || EK == EK_F32) {
                if (E.out16 != nullptr) o16 = E.out16 + E.out16_ch_off + co + pix0 * ps16;
                if (EK == EK_F32 && E.out32 != nullptr) o32 = E.out32 + E.out32_ch_off + co + pix0 * ps32;
                if (EK == EK_PLAIN && E.res16 != nullptr) r16 = E.res16 + E.res_ch_off + co + pix0 * psr;
                if (EK == EK_F32 && E.res32 != nullptr) r32 = E.res32 + E.res_ch_off + co + pix0 * psr;
            } else if (EK == EK_PIXSHUF) {
                // out[b, c, 2y+i, 2x+j] = in[b, 4c + 2i + j, y, x]  (edvr_arch.py:351,410-411)
                const int i = (co >> 1) & 1, j = co & 1;
                o16 = E.out16 + E.out16_ch_off + (co >> 2) +
                      ((static_cast<long long>(img) * 2 * H + 2 * y0 + i) * (2 * W) + 2 * x0 + j) * ps16;
                ops16 = 2 * ps16;
                orow16 = 2 * static_cast<long long>(2 * W) * ps16;
            } else {   // EK_STRIDE2: even pixels only; tile origins are even
                const int Wo = (W + 1) >> 1, Hos = (H + 1) >> 1;
                o16 = E.out16 + E.out16_ch_off + co +
                      ((static_cast<long long>(img) * Hos + (y0 >> 1)) * Wo + (x0 >> 1)) * ps16;
                orow16 = static_cast<long long>(Wo) * ps16;      // per TWO input rows
            }
            C2_TIMED_WAIT_WARP(&acc_full[ab], (acc_it >> 1) & 1u, ST_E_WAIT_ACC);
            tc_fence_after_sync();
            const uint32_t t0 = tmem_base + (static_cast<uint32_t>(32 * q) << 16) + ab * 256u;
#pragma unroll 1
            for (int col = 0; col < 256; col += 32) {
                long long tq = STATS ? clock64() : 0;
                float v[32];
                tmem_ld32(t0 + col, v);
                if (STATS) { const long long t = clock64(); st_acc[ST_E_TMEM] += t - tq; tq = t; }
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] += bias_c;
                act_inplace<32>(v, E.act);
                const int yb = col >> 3;                                   // first tile row of these 32 pixels
                if (STATS) { const long long t = clock64(); st_acc[ST_E_P1] += t - tq; tq = t; }
                if (img_ok && !(dbg & 2)) {
                    if (EK == EK_PLAIN) {
                        if (interior) {
                            // full tile: straight-line code, no predicates (keeps the loop inside the L0 I-cache)
#pragma unroll
                            for (int r = 0; r < 4; ++r) {
                                const long long rofs = static_cast<long long>(yb + r) * W;
                                if (EK == EK_PLAIN && r16 != nullptr) {
                                    const __half* rp = r16 + rofs * psr;
                                    __half t[8];
#pragma unroll
                                    for (int c = 0; c < 8; ++c) t[c] = rp[c * psr];
#pragma unroll
                                    for (int c = 0; c < 8; ++c) v[r * 8 + c] += __half2float(t[c]);
                                }
                                __half* op = o16 + rofs * ps16;
#pragma unroll
                                for (int c = 0; c < 8; ++c) op[c * ps16] = __float2half_rn(v[r * 8 + c]);
                            }
                        } else {
#pragma unroll 1
                            for (int r = 0; r < 4; ++r) {
                                if (y0 + yb + r >= H) break;
                                const long long rofs = static_cast<long long>(yb + r) * W;
                                for (int c = 0; c < xn; ++c) {
                                    float val = sel32(v, r * 8 + c);
                                    if (EK == EK_PLAIN && r16 != nullptr) val += __half2float(r16[(rofs + c) * psr]);
                                    o16[(rofs + c) * ps16] = __float2half_rn(val);
                                }
                            }
                        }
                    } else if (EK == EK_F32) {
                        if (interior) {
#pragma unroll
                            for (int r = 0; r < 4; ++r) {
                                const long long rofs = static_cast<long long>(yb + r) * W;
                                if (r32 != nullptr) {
                                    const float* rp = r32 + rofs * psr;
                                    float t[8];
#pragma unroll
                                    for (int c = 0; c < 8; ++c) t[c] = __ldg(rp + c * psr);
#pragma unroll
                                    for (int c = 0; c < 8; ++c) v[r * 8 + c] += t[c];
                                }
                                if (o16 != nullptr) {
                                    __half* op = o16 + rofs * ps16;
#pragma unroll
                                    for (int c = 0; c < 8; ++c) op[c * ps16] = __float2half_rn(v[r * 8 + c]);
                                }
                                if (o32 != nullptr) {
                                    float* op = o32 + rofs * ps32;
#pragma unroll
                                    for (int c = 0; c < 8; ++c) op[c * ps32] = v[r * 8 + c];
                                }
                            }
                        } else {
#pragma unroll 1
                            for (int r = 0; r < 4; ++r) {
                                if (y0 + yb + r >= H) break;
                                const long long rofs = static_cast<long long>(yb + r) * W;
                                for (int c = 0; c < xn; ++c) {
                                    float val = sel32(v, r * 8 + c);
                                    if (r32 != nullptr) val += __ldg(r32 + (rofs + c) * psr);
                                    if (o16 != nullptr) o16[(rofs + c) * ps16] = __float2half_rn(val);
                                    if (o32 != nullptr) o32[(rofs + c) * ps32] = val;
                                }
                            }
                        }
                    } else if (EK == EK_PIXSHUF) {
#pragma unroll
                        for (int r = 0; r < 4; ++r) {
                            if (y0 + yb + r >= H) break;
                            __half* op = o16 + static_cast<long long>(yb + r) * orow16;
#pragma unroll
                            for (int c = 0; c < 8; ++c)
                                if (c < xn) op[c * ops16] = __float2half_rn(v[r * 8 + c]);
                        }
                    } else {
#pragma unroll
                        for (int r = 0; r < 4; r += 2) {
                            if (y0 + yb + r >= H) break;
                            __half* op = o16 + static_cast<long long>((yb + r) >> 1) * orow16;
#pragma unroll
                            for (int c = 0; c < 8; c += 2)
                                if (c < xn) op[(c >> 1) * ops16] = __float2half_rn(v[r * 8 + c]);
                        }
                    }
                }
                if (STATS) st_acc[ST_E_P2] += clock64() - tq;
            }
            tc_fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[ab]);
        }
    }

    if (STATS && P.stats != nullptr && lane == 0 && (warp == 0 || warp == 1 || warp == 2 || warp == 6)) {
        unsigned long long* o = P.stats + static_cast<size_t>(blockIdx.x) * 16;
        const unsigned long long tot = static_cast<unsigned long long>(clock64() - st_t0);
        if (warp == 1) { o[ST_MMA_TOTAL] = tot; o[ST_MMA_WAIT_ACC] = st_acc[ST_MMA_WAIT_ACC]; o[ST_MMA_WAIT_A] = st_acc[ST_MMA_WAIT_A]; o[ST_MMA_WAIT_W] = st_acc[ST_MMA_WAIT_W]; }
        if (warp == 2) { o[ST_A_TOTAL] = tot; o[ST_A_WAIT_EMPTY] = st_acc[ST_A_WAIT_EMPTY]; }
        if (warp == 0) { o[ST_W_TOTAL] = tot; o[ST_W_WAIT_EMPTY] = st_acc[ST_W_WAIT_EMPTY]; }
        if (warp == 6) { o[ST_E_TMEM] = st_acc[ST_E_TMEM]; o[ST_E_P1] = st_acc[ST_E_P1]; o[ST_E_BAR] = st_acc[ST_E_BAR]; o[ST_E_P2] = st_acc[ST_E_P2]; o[ST_E_TOTAL] = tot; o[ST_E_WAIT_ACC] = st_acc[ST_E_WAIT_ACC]; o[ST_TILES] = (total_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x; }
    }
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, 512);
}

}  // namespace eb
